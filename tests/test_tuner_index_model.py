"""The tuner bank's table-index fast paths, emulated on the CPU (tests/tuner_phase.py) over the inputs
tests/test_gpu_tuner_index.py sends through the GPU: the emulations equal the reference index on every
sample, the inputs put samples into every distance band around the table boundaries at every seam of
the kernels, and wrong variants of the guards give wrong indices on them.  No GPU needed."""
import numpy as np
import pytest

import tuner_phase as T

STREAM_SHAPES = [(96000, 27), (192000, 27), (192000, 64)]          # (rate, taps): D = 10, 20, 20
TILE_SHAPES = [(48000, 27), (96000, 40), (192000, 27)]                # D = 5, 10, 20
STREAM_MUTANTS = [m for m in T.MUTANTS if m.startswith("stream")] + ["table_index without its guard"]
TILE_MUTANTS = ["tile guard one-sided (== 0)", "table_index without its guard"]
# variants the model shows to be harmless, and why
HARMLESS = {
    "stream window one short at the top [-1, D]":
        "sample j of a period borrows at most j <= D-1 units from the low words, so the window's top "
        "end D+1 has two units of slack",
}

_cache = {}


def run(kind, rate, ntaps):
    key = (kind, rate, ntaps)
    if key not in _cache:
        plan = T.bank_plan(rate)
        mode = 2 if kind == "stream" else 1
        muts = STREAM_MUTANTS if kind == "stream" else TILE_MUTANTS
        _cache[key] = (plan, T.simulate(plan, mode, ntaps=ntaps, mutants=[None] + muts))
    return _cache[key]


def test_constants_are_read_from_the_source():
    assert T.K.two_pi == 2.0 * np.pi
    assert T.K.scale_hi + T.K.scale_lo == 256.0 / T.K.two_pi
    assert T.K.stream_shapes == [(27, 10), (27, 20), (64, 20)]
    assert T.K.reanchor == 12 and T.K.near_plus == 2 and T.K.tile_bound == 1 and T.K.ti_guard == 64
    assert T.dx56(np.pi / 2) != 0 and T.dx56(3.1) == 0 and T.dx48(3.1) != 0


def test_reference_recurrence_is_the_oracles():
    """After every block of a plan with retunes, O.Bpsk's tuPhase equals the numpy replay bit for bit."""
    import oracle as O
    plan = T.bank_plan(96000, lens=(2500, 9000, 333, 1, 4097))
    chans = np.arange(0, plan.nchan, 7)
    orcs = [O.Bpsk(plan.rate, float(plan.tunings[0][c]), stages=1) for c in chans]
    p = np.zeros(chans.size)
    rng = np.random.default_rng(1)
    for k, S in enumerate(plan.lens):
        tun = plan.tunings[k][chans]
        x = rng.uniform(-1, 1, 2 * S).astype(np.float32)
        for i, o in enumerate(orcs):
            o.set_tuning(float(tun[i]))
            o.receive(x)
        _, p = T.replay(p, T.tuner_inc(tun, plan.rate), S)
        got = np.array([o.s.tuPhase for o in orcs])
        assert np.array_equal(got.view(np.int64), p.view(np.int64)), k


def test_boundary_distance_is_exact():
    """boundary_offset against exact rationals on phases near and far from the boundaries."""
    from fractions import Fraction
    rng = np.random.default_rng(2)
    k = rng.integers(0, 257, 300)
    near = np.array([float(Fraction(int(j)) * Fraction(T.K.two_pi) / 256) for j in k])
    ph = np.concatenate([near, np.nextafter(near, 10.0), rng.uniform(0, T.K.two_pi, 300)])
    ph = ph[ph > 0]
    got = T.boundary_offset(ph)
    for p, g in zip(ph, got):
        x = Fraction(p) * 256 / Fraction(T.K.two_pi)
        d = x - round(x)
        assert abs(float(d) - g) <= abs(float(d)) * 2.0 ** -51 + 2.0 ** -120, (p, float(d), g)


def test_table_index_emulation_equals_the_division():
    rng = np.random.default_rng(3)
    ph = np.concatenate([rng.uniform(0, 2 * T.K.two_pi, 200000),
                         np.arange(1, 513) * T.K.two_pi / 256])
    ph = np.concatenate([ph, np.nextafter(ph, 0), np.nextafter(ph, 20)])
    ph = ph[ph > 0]
    k, ex = T.table_index(ph)
    assert np.array_equal(k, T.ref_index(ph))
    assert ex.sum() > 1000


@pytest.mark.parametrize("rate,ntaps", STREAM_SHAPES)
def test_stream_emulation_equals_the_reference(rate, ntaps):
    plan, res = run("stream", rate, ntaps)
    t = res[None]
    assert t["stream"].wrong == 0 and t["table_index"].wrong == 0, (t["stream"].wrong_where, t["table_index"].wrong_where)
    assert t["tile"].counts == {}


@pytest.mark.parametrize("rate,ntaps", TILE_SHAPES)
def test_tile_emulation_equals_the_reference(rate, ntaps):
    plan, res = run("tile", rate, ntaps)
    t = res[None]
    assert t["tile"].wrong == 0 and t["table_index"].wrong == 0, (t["tile"].wrong_where, t["table_index"].wrong_where)
    assert t["stream"].counts == {}


@pytest.mark.parametrize("rate", [96000, 192000])
def test_climbs_through_zero_land_where_planned_and_take_the_bypass(rate):
    """The plan's climbs from negative phase reach phase > 0 first at their target samples, the exact
    returns hit 0.0 at theirs (and are positive right after), and the streaming kernel's emulation takes
    the mixer bypass on every sample up to and including them."""
    plan = T.bank_plan(rate)
    D, S1 = rate // 9600, plan.lens[1]
    ph0, p0 = T.replay(np.zeros(plan.nchan), T.tuner_inc(plan.tunings[0], rate), plan.lens[0])
    ph1, _ = T.replay(p0, T.tuner_inc(plan.tunings[1], rate), S1)
    assert len(plan.zeros) == 12 and len(plan.crossings) > 40
    for c, blk, s in plan.zeros:
        assert blk == 1 and ph1[s, c] == 0.0 and ph1[s + 1, c] > 0.0 and np.all(ph1[:s, c] < 0.0), (c, s)
    for c, blk, s in plan.crossings:
        assert blk == 1 and ph1[s, c] > 0.0 and np.all(ph1[:s, c] <= 0.0), (c, s)
    chans = np.array([c for c, _, _ in plan.zeros + plan.crossings])
    ds_cnt = plan.lens[0] % D
    n0, NO = D - 1 - ds_cnt, (ds_cnt + S1) // D
    ph = ph1[:, chans]
    ckpt = np.vstack([p0[None, chans], ph[31:S1 - 1:32]])[:(S1 + 31) // 32]
    dxs = np.array([T.dx56(v) for v in T.tuner_inc(plan.tunings[1][chans], rate)], np.uint64)
    r = T.stream_block(ckpt, T.tuner_index(ph), dxs, D, 27, S1, n0, NO, T.K.r_min)
    nz = len(plan.zeros)
    for i, (c, _, s) in enumerate(plan.zeros + plan.crossings):
        last = s if i < nz else s - 1                      # the last sample that must bypass
        sel = r["used"] & (r["s"] <= last)
        assert np.all(r["path"][sel, i] == 3) and np.all(r["idx"][sel, i] == 256), (c, s)
        after = r["used"] & (r["s"] > last)
        assert np.all(r["path"][after, i] != 3), (c, s)


def _table(counts, D, seams):
    _, names = T.bands(D)
    rows = [f"{'band':>22} " + " ".join(f"{s:>16}" for s in seams)]
    for pth in ("fast", "replay", "exact", "bypass"):
        for nm in names:
            vals = [counts.get((pth, nm, s), 0) for s in seams]
            if any(vals):
                rows.append(f"{pth + ' ' + nm:>22} " + " ".join(f"{v:>16}" for v in vals))
    return "\n".join(rows)


STREAM_SEAMS = ["any", "chunk", "period", "anchor", "segment", "block"]


@pytest.mark.parametrize("rate,ntaps", STREAM_SHAPES)
def test_stream_inputs_cover_every_band_at_every_seam(rate, ntaps):
    """Every band holds samples the kernel evaluates, at every seam: in the bands below the guard they
    must be replayed (the estimate cannot decide them), in the band just above it the fast estimate
    must be right."""
    D = rate // 9600
    plan, res = run("stream", rate, ntaps)
    c = res[None]["stream"].counts
    print(f"\nk_mixdecim_stream {ntaps} taps, D = {D}: used samples per path, band and seam\n" + _table(c, D, STREAM_SEAMS))
    _, names = T.bands(D)
    for seam in STREAM_SEAMS:
        for nm in names[:4]:                                   # below the guard: replayed
            assert c.get(("replay", nm, seam), 0) >= 20, (seam, nm)
        for nm in names[3 + (seam == "block"):]:               # from the guard up: fast
            assert c.get(("fast", nm, seam), 0) >= 20, (seam, nm)


@pytest.mark.parametrize("rate,ntaps", TILE_SHAPES)
def test_tile_inputs_cover_every_band(rate, ntaps):
    D = rate // 9600
    plan, res = run("tile", rate, ntaps)
    c = res[None]["tile"].counts
    print(f"\nk_mixdecim {ntaps} taps, D = {D}: used samples per path, band and seam\n" + _table(c, D, ["any", "chunk", "block"]))
    _, names = T.bands(D)
    for seam in ("any", "chunk"):
        for nm in names[:5]:                                   # within 2^-16: the chunk is replayed
            assert c.get(("replay", nm, seam), 0) >= 20, (seam, nm)
        for nm in names[5:]:
            assert c.get(("fast", nm, seam), 0) >= 20, (seam, nm)
    assert sum(v for (p, nm, s), v in c.items() if s == "block") >= 20


def test_table_index_inputs_reach_its_guard():
    """The replays (and the history tail) evaluate table_index on samples in every band: below its 6e-5
    guard the division decides, above it the multiply must be right."""
    plan, res = run("stream", 96000, 27)
    c = res[None]["table_index"].counts
    print("\ntable_index: replayed samples per path and band\n" + _table(c, 10, ["any"]))
    _, names = T.bands(10)
    for nm in names[:6]:
        assert c.get(("exact", nm, "any"), 0) >= 100, nm
    assert c.get(("fast", names[5], "any"), 0) >= 100 and c.get(("fast", names[6], "any"), 0) >= 1000


def fuzz_plans(nseeds=24):
    """The bank scenarios test_gpu_fuzz draws, and the channels it watches."""
    from test_gpu_fuzz import scenario
    for seed in range(nseeds):
        rng, rate, nchan, shared, s16, lens, max_block, tuning, kernel, retunes = scenario(seed)
        watch = sorted(set([0, nchan - 1, int(rng.integers(0, nchan))] + [c for v in retunes.values() for c, _ in v]))
        tun, tunings = np.array(tuning, np.float64), []
        for k in range(len(lens)):
            for c, hz in retunes.get(k, []):
                tun[c] = hz
            tunings.append(tun.copy())
        yield T.Plan(rate, lens, tunings), kernel, s16, watch


def test_every_wrong_guard_is_seen():
    """Each variant of a guard gives wrong indices on the generated inputs, unless the model shows it
    harmless.  For each, whether the bank scenarios of test_gpu_fuzz (24 seeds, the watched channels)
    would have seen it too."""
    fuzz = {m: 0 for m in T.MUTANTS}
    for plan, kernel, s16, watch in fuzz_plans():
        res = T.simulate(plan, kernel, s16=s16, channels=watch, mutants=list(T.MUTANTS))
        for m, t in res.items():
            fuzz[m] += sum(x.wrong for x in t.values())
    lines = []
    for m in T.MUTANTS:
        ours = 0
        for rate, ntaps in STREAM_SHAPES:
            if m in STREAM_MUTANTS:
                ours += sum(x.wrong for x in run("stream", rate, ntaps)[1][m].values())
        for rate, ntaps in TILE_SHAPES:
            if m in TILE_MUTANTS:
                ours += sum(x.wrong for x in run("tile", rate, ntaps)[1][m].values())
        lines.append(f"{m:>48}: {ours:>8} wrong indices on the generated inputs, {fuzz[m]:>6} on test_gpu_fuzz's draws"
                     + (f"  (harmless: {HARMLESS[m]})" if m in HARMLESS else ""))
        if m in HARMLESS:
            assert ours == 0, m
        else:
            assert ours > 0, m
    print("\n" + "\n".join(lines))
    # what only the new inputs see
    assert fuzz["stream window [0, 1] (no borrow margin)"] == 0
    assert fuzz["stream window one short at the bottom [0, D+1]"] == 0
    assert fuzz["stream anchor not refreshed within a segment"] == 0
