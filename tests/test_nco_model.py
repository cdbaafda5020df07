"""The model of demod.java's NCO that tests/test_gpu_nco.py holds the GPU to (tests/nco_phase.py),
checked without a GPU: the emulation of nco_sincos against exact arithmetic, the float it rounds to
against the correctly rounded sine and cosine, the input plan against what it claims to reach, and
the checker's power against deliberately wrong kernels.

Result of the exhaustive scan over every float in [-8, 8] (tools/nco_scan.py, recorded in DESIGN
section 4.5): 2 181 038 082 floats; nco_sincos's float equals the correctly rounded float of sin
and cos for every one of them.  16 were doubtful (binary64 result within BAND ulps of a float
midpoint), all in (-0.5, 0.5): +-0.000244140625, 0.000545915042, 0.000809722871, 0.00881955586,
0.0327920094, 0.101237468, 0.218410701, 0.475609273; resolved exactly, all agree.  Here: every float
in [0.5, 2 pi] (none doubtful), a seeded stride elsewhere and every phase the GPU inputs reach."""
import numpy as np
import pytest

import nco_phase as N
import oracle as O

RATE = 96000


def _resolve(car):
    """(kernel float, correctly rounded float) of sin and cos for an array of phases, |car| <= 8."""
    ks, kc = N.kernel_sincos(car)
    cs_, cc_, _, _ = N.cr_sincos(car)
    return ks, kc, cs_, cc_


def _near_quadrants():
    """Every float within 2^-10 of k*pi/2, k = -5..5, k != 0 (for k = 0 the reduction is exact:
    r = car), and a stride of 2^12 floats through (0, 2^-10]."""
    out = []
    for k in range(-5, 6):
        if k == 0:
            continue
        c = k * np.pi / 2
        lo, hi = np.float32(c - 2.0 ** -10), np.float32(c + 2.0 ** -10)
        a, b = sorted((lo.view(np.int32), hi.view(np.int32)))
        out.append(np.arange(a, b + 1, dtype=np.int32).view(np.float32))
    tiny = np.arange(1, np.float32(2.0 ** -10).view(np.int32), 1 << 12, dtype=np.int32).view(np.float32)
    out += [tiny, -tiny]
    return np.concatenate(out)


def test_vectorised_exact_fma_equals_fractions():
    """fma_exact_vec (rounding to odd) is checked against Fractions on the chain's own operands,
    so that it may stand in for them on the million phases below."""
    rng = np.random.default_rng(1)
    car = np.concatenate([rng.uniform(-8, 8, 1500).astype(np.float32), _near_quadrants()[::97]])
    kv, sv, cv = N.chain_exact_vec(car)
    for i, x in enumerate(car):
        k, s, c = N.chain_exact_scalar(float(x))
        assert (k, s, c) == (kv[i], sv[i], cv[i]), x


def test_band_is_four_times_the_measured_distance():
    """The multiply-and-add chain against the exact one on >= 10^6 phases: the largest distance
    (binary64 ulps) times four must fit BAND, and no quadrant may differ."""
    rng = np.random.default_rng(2)
    car = np.concatenate([rng.uniform(-8, 8, 1_000_000).astype(np.float32), _near_quadrants()])
    assert car.size >= 1_000_000
    km, sm, cm = N.chain_muladd(car)
    ke, se, ce = N.chain_exact_vec(car)
    assert np.array_equal(km, ke)
    worst = max(np.max(np.abs(sm - se) / np.spacing(np.abs(se))), np.max(np.abs(cm - ce) / np.spacing(np.abs(ce))))
    print(f"mul+add vs FMA chain: {worst} binary64 ulps at most over {car.size} phases; BAND {N.BAND}")
    assert 4 * worst <= N.BAND


def test_libm_band_is_four_times_numpys_measured_error():
    """numpy's binary64 sin / cos against mpmath at 200 bits, on the recurrence's range, the fast
    path's and the library path's (up to the stall near 2^25): LIBM_BAND covers four times it."""
    import mpmath
    rng = np.random.default_rng(3)
    car = np.concatenate([rng.uniform(0, 2 * np.pi, 1000), rng.uniform(-8, 8, 1000),
                          rng.uniform(8, 2.0 ** 25, 1000)]).astype(np.float32)
    worst = 0.0
    with mpmath.workprec(200):
        for x in car:
            for f, g in ((np.sin, mpmath.sin), (np.cos, mpmath.cos)):
                t = g(mpmath.mpf(float(x)))
                worst = max(worst, float(abs(mpmath.mpf(float(f(np.float64(x)))) - t)) / float(np.spacing(abs(float(t)))))
    print(f"numpy sin/cos: {worst} binary64 ulps at most; LIBM_BAND {N.LIBM_BAND}")
    assert 4 * worst <= N.LIBM_BAND


def test_emulation_equals_exact_on_the_doubt_set_and_libm_elsewhere():
    rng = np.random.default_rng(4)
    car = np.concatenate([rng.uniform(-8, 8, 2_000_000).astype(np.float32), _near_quadrants()])
    stats = {}
    ks, kc = N.kernel_sincos(car, stats)
    x = car.astype(np.float64)
    assert np.array_equal(ks, np.sin(x).astype(np.float32))
    assert np.array_equal(kc, np.cos(x).astype(np.float32))
    _, fs, fc = N.chain_muladd(car)
    doubt = np.flatnonzero(N.near_half(car) | (N.midpoint_ulps(fs) <= N.BAND) | (N.midpoint_ulps(fc) <= N.BAND))
    ke, se, ce = N.chain_exact_vec(car[doubt])
    es, ec = N._quadrant(ke, se, ce)
    assert np.array_equal(ks[doubt], es) and np.array_equal(kc[doubt], ec)
    assert stats["doubt"] == doubt.size


def test_every_float_from_half_to_two_pi_is_correctly_rounded():
    """All 29.95 M floats of [0.5, 2 pi]: the kernel's float == the correctly rounded float."""
    a, b = np.float32(0.5).view(np.int32), N.TWOPI.view(np.int32)
    bad, doubt = [], 0
    for lo in range(int(a), int(b) + 1, 1 << 22):
        car = np.arange(lo, min(lo + (1 << 22), int(b) + 1), dtype=np.int32).view(np.float32)
        stats = {}
        ks, kc = N.kernel_sincos(car, stats)
        cs_, cc_, _, _ = N.cr_sincos(car)
        doubt += stats.get("doubt", 0)
        bad += list(car[(ks != cs_) | (kc != cc_)])
    print(f"[0.5, 2 pi]: {int(b) - int(a) + 1} floats, {doubt} resolved exactly, {len(bad)} differ")
    assert bad == []


def _reachable():
    """Every phase the planned GPU inputs reach on the fast path."""
    out = []
    for rate in N.RATES:
        for flo, m in N.zero_returns(rate):
            out.append(N.phases(N.phi_of(flo, rate), 0, m)[:-1])
        for flo in N.planned_tunings(rate):
            out.append(N.phases(N.phi_of(flo, rate), 0, 4200)[:-1])
    c = np.unique(np.concatenate(out))
    return c[np.abs(c) <= 8]


def test_stride_below_half_and_negative_and_the_reachable_phases():
    rng = np.random.default_rng(5)
    a = np.float32(0.5).view(np.int32)
    pos = np.arange(1, a, 499, dtype=np.int32).view(np.float32)                       # (0, 0.5)
    neg = -np.arange(1, np.float32(8).view(np.int32) + 1, 997, dtype=np.int32).view(np.float32)   # [-8, 0)
    car = np.concatenate([pos, neg, _reachable(), rng.uniform(-8, 0.5, 200_000).astype(np.float32),
                          np.float32([0.0, -0.0, 8.0, -8.0, 2.4414062e-4, 0.47560927])])
    ks, kc, cs_, cc_ = _resolve(car)
    assert np.array_equal(ks, cs_) and np.array_equal(kc, cc_)


# ------------------------------------------------------------------ the plan
@pytest.mark.parametrize("rate", N.RATES)
def test_zero_returns_land_on_every_planned_seam(rate):
    z = N.zero_returns(rate)
    assert len([f for f, _ in z if f < rate]) >= 20
    for flo, m in z:
        tr = N.phases(N.phi_of(flo, rate), 0.0, m + 1)
        assert tr[m] == 0.0 and np.all(tr[1:m] != 0.0), flo
        for q in N.SEAMS:
            p = N.placement(m, q)
            seen = N.phases(N.phi_of(flo, rate), 0.0, p + q + 1)
            assert p >= 0 and seen[p + q] == 0.0 and (p + q) % m == 0, (flo, q)


@pytest.mark.parametrize("rate", N.RATES)
def test_out_of_range_tunings_reach_the_library_path(rate):
    for flo in N.planned_tunings(rate):
        tr = N.phases(N.phi_of(flo, rate), 0.0, 4100)
        if flo < 0:
            assert np.max(tr) > 8, flo                                  # within one 4100-sample call
        elif flo == rate:
            assert np.all(tr == 0), flo                                 # phi == (float)(2 pi): car stays 0
        elif flo > rate:
            assert np.min(tr) < 0, flo                                  # phi > 2 pi: car runs negative
        else:
            assert 0 <= np.min(tr) and np.max(tr) <= N.TWOPI, flo


def test_the_long_run_reaches_the_stall():
    assert N.stall_flo(RATE) == N.LONG_FLO
    phi = N.phi_of(N.LONG_FLO, RATE)
    total = sum(N.LONG_CALLS)
    k = N.stall_point(phi, total)
    assert 0 < k < total - 256, k
    tr = N.phases(phi, 0.0, total)
    assert np.all(tr[k:] == tr[k]) and abs(float(tr[k])) == 2.0 ** 24


# ------------------------------------------------------------------ power
def _plan_inputs():
    """(phi, car trace, FIR output) for the power tests: every zero-return tuning at 96 kS/s at
    the seams, a prefix call of ragged length in front, and the out-of-range tunings."""
    rng = np.random.default_rng(6)
    cases = []
    for flo, m in N.zero_returns(RATE)[:8] + tuple((f, 0) for f in N.planned_tunings(RATE)):
        p = N.placement(m, N.TILE - 1) if m else 45
        n = p + 1100
        o = O.Demod(RATE, True, False)
        o.weights(flo, flo + 5000)
        y = o.receive(rng.uniform(-1, 1, 2 * n).astype(np.float32))
        cases.append((N.phi_of(flo, RATE), p, y))
    return cases


def _run(cases, trace_fn=None, sincos_fn=None, carry_fn=None):
    """Per case the mixed floats of a two-call run (prefix p, then the rest) with one piece of
    the model replaced; returns the list of (wrong, reference) pairs."""
    out = []
    for phi, p, y in cases:
        n = y.size // 2
        ref_tr = N.phases(phi, 0.0, n)
        ref, _ = N.mix_reference(y, ref_tr)
        tr = trace_fn(phi, n) if trace_fn else ref_tr.copy()
        if carry_fn:
            tr = np.concatenate([tr[:p], N.phases(phi, carry_fn(tr, p), n - p)])
        if sincos_fn:
            sn, cs = sincos_fn(tr[:n])
            wrong = N._mix(y, cs, sn)
        else:
            wrong, _ = N.mix_reference(y, tr)
        out.append((wrong, ref))
    return out


def _old_bars_accept(pairs):
    """The bars the suite held the NCO to before: 1e-6 on the mixed floats (and so well inside one
    s16 LSB of the audio)."""
    return all(np.max(np.abs(w - r)) <= 1e-6 * max(1.0, np.max(np.abs(r))) for w, r in pairs)


VARIANTS = {
    "wrap on car <= 0": dict(trace_fn=lambda phi, n: N.phases_variant(phi, 0.0, n, wrap_le=True)),
    "binary32 sin / cos": dict(sincos_fn=lambda car: (np.sin(car.astype(np.float32)), np.cos(car.astype(np.float32)))),
    "car in binary64, rounded at checkpoints": dict(trace_fn=lambda phi, n: N.phases_variant(phi, 0.0, n, f64=True)),
    "the updated car used for the current sample": dict(trace_fn=lambda phi, n: N.phases(phi, 0.0, n + 1)[1:]),
    "last partial chunk not carried": dict(carry_fn=lambda tr, p: tr[(p // N.CHUNK) * N.CHUNK]),
}
# Which of these the 1e-6 / one-LSB bars let through (asserted below, so that it stays true).
OLD_BARS_ACCEPT = {"wrap on car <= 0", "binary32 sin / cos"}


@pytest.mark.parametrize("name", list(VARIANTS))
def test_wrong_kernels_fail_the_reference(name):
    pairs = _run(_plan_inputs(), **VARIANTS[name])
    assert any(not np.array_equal(w.view(np.uint32), r.view(np.uint32)) for w, r in pairs), name
    assert _old_bars_accept(pairs) == (name in OLD_BARS_ACCEPT), name


def test_cody_waite_tail_term():
    """The reduction's second step (c_trig[14], the low part of pi/2) is not a variant the GPU
    tests can reject: dropping it changes no float on a stride through [0.5, 8] or at any phase the
    plan reaches (tools/nco_scan.py counts the whole of [-8, 8]).  Asserted, so that a change of the
    coefficients or the reduction that makes it matter is noticed here."""
    c = N.coefficients()
    b = np.float32(8).view(np.int32)
    stride = np.arange(np.float32(0.5).view(np.int32), b, 13, dtype=np.int32).view(np.float32)
    car = np.concatenate([_reachable(), stride, -stride[::7]])
    x = car.astype(np.float64)
    kd = (x * c[12] + N.MAGIC) - N.MAGIC
    r = x - kd * c[13]                                          # no "- kd * c[14]"
    z = r * r
    ps = np.full_like(z, c[5])
    for i in (4, 3, 2, 1, 0):
        ps = ps * z + c[i]
    pc = np.full_like(z, c[11])
    for i in (10, 9, 8, 7, 6):
        pc = pc * z + c[i]
    ws, wc = N._quadrant(kd, r + (z * r) * ps, (1.0 - 0.5 * z) + (z * z) * pc)
    ks, kc = N.kernel_sincos(car)
    assert np.array_equal(ws, ks) and np.array_equal(wc, kc)
