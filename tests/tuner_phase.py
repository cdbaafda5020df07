"""The tuner bank's table index (FUNcubeBPSKDemod.java:384-390) and the three fast paths that compute it.

RxMixTuner takes the cos/sin table index of every input sample as (int)(tuPhase*256/(2pi)) % 256, with
tuPhase a binary64 accumulator (`p += inc; if (p > 2pi) p -= 2pi`); a phase <= 0 bypasses the mixer.
Three places in java-sdr_b200/csrc estimate that index without the division and fall back to the
reference's own arithmetic when the estimate is too close to a table boundary:

  table_index        (bpsk.cu)             multiply by 1/2pi, guard on the quotient's 20 fraction bits
  k_mixdecim         (bpsk.cu, phase 1)    8.48 fixed point stepped from the 32-sample checkpoint
  k_mixdecim_stream  (bpsk_stream.cuh)     8.56 fixed point anchored every kReanchor periods, and
                                           hi32(x_top) - j*hi32(dx) per sample with a borrow margin

This module restates the reference recurrence in numpy binary64, measures every sample's exact distance
to the nearest table boundary, emulates each fast path bit for bit (the constants are read out of the
CUDA source, so the model follows the code), and generates tunings whose phases sweep through every
boundary band at the kernels' seams.  tests/test_tuner_index_model.py shows that the emulations agree
with the reference and that the inputs see wrong variants of the guards; tests/test_gpu_tuner_index.py
runs the same inputs through the bank on the GPU against the oracle.
"""
from __future__ import annotations

import math
import os
import re
from dataclasses import dataclass, field

import numpy as np

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "java-sdr_b200", "csrc")
U64 = np.uint64
M64 = (1 << 64) - 1


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _grab(txt, pat, conv=float):
    m = re.search(pat, txt, re.S)
    assert m, f"pattern not found in the CUDA source: {pat}"
    return [conv(g) for g in m.groups()] if len(m.groups()) > 1 else conv(m.group(1))


class Constants:
    """Every number the index paths depend on, read out of bpsk.cu and bpsk_stream.cuh."""

    def __init__(self):
        b, s = _src("bpsk.cu"), _src("bpsk_stream.cuh")
        self.two_pi = 2.0 * _grab(b, r"constexpr double kTwoPi = 2\.0 \* ([0-9.]+);")
        self.inv_two_pi = 1.0 / self.two_pi
        self.scale_hi = _grab(b, r"constexpr double kIdxScaleHi = ([-0-9.e]+);")
        self.scale_lo = _grab(b, r"constexpr double kIdxScaleLo = ([-0-9.e]+);")
        # table_index: y = fma(t, kInvTwoPi * 2^20, 1.5 * 2^52), guard on the low 20 bits
        assert "__fma_rn(t, kInvTwoPi * 1048576.0, 6755399441055744.0)" in b
        assert "const int frac = yi & 0xfffff;" in b and "int k = yi >> 20;" in b
        g1, g2 = _grab(b, r"if \(frac < (\d+) \|\| frac > 1048576 - (\d+)\)", int)
        assert g1 == g2
        self.ti_guard = g1
        # k_mixdecim phase 1: near |= ((xh + 1) & 0xffff) <= B
        self.tile_mask = 0xffff
        assert "near |= ((xh + 1u) & 0xffffu) <=" in b
        self.tile_bound = _grab(b, r"near \|= \(\(xh \+ 1u\) & 0xffffu\) <= (\d+)u;", int)
        # the fixed-point steps (host, long double)
        self.dx48_limit = _grab(b, r"if \(!\(inc > 0\.0\) \|\| !\(inc < ([0-9.e]+)\)\) return 0ull;\s*const long double c = 256\.0L / \(long double\)\(2\.0 \* M_PI\);\s*long double d = fmodl\(\(long double\)inc \* c, 256\.0L\);\s*unsigned long long v = \(unsigned long long\)\(d \* 281474976710656\.0L")
        self.dx56_limit = _grab(b, r"if \(!\(inc > 0\.0\) \|\| !\(inc < ([0-9.e]+)\)\) return 0ull;\s*const long double c = 256\.0L / \(long double\)\(2\.0 \* M_PI\);\s*long double d = fmodl\(\(long double\)inc \* c, 256\.0L\);\s*unsigned long long v = \(unsigned long long\)\(d \* 72057594037927936\.0L")
        # segment length of the streaming kernel (launch_stream)
        self.r_min = _grab(b, r"if \(R < (\d+)\) R = \1;", int)
        self.segs_per_warp = _grab(b, r'env_int\("JSDR_STREAM_SEGS", 1, 64, (\d+)\)', int)
        self.scout_big, self.scout_wide, self.scout_narrow = _grab(b, r"return \(pump && b->nchan >= (\d+)\) \? (\d+) : (\d+);", int)
        # the streaming kernel
        self.reanchor = _grab(s, r"constexpr int kReanchor = (\d+);", int)
        self.warps_s16 = _grab(s, r"constexpr int kWarps = (\d+);", int)
        self.warps_f32 = _grab(s, r"constexpr int kWarpsF32 = (\d+);", int)
        self.near_plus = _grab(s, r"near \|= \(nt \+ \(unsigned\)j \* ndx8\) <= 256u \* \(unsigned\)\(DD \+ (\d+)\);", int)
        assert "const unsigned nt = (xt << 8) + 256u, ndx8 = ndx << 8;" in s
        assert "taddr[j] = lane_tab + ((xj >> 17) & 0x7f80u);" in s
        # the streaming kernel's compiled (taps, D) shapes, and the choice between the kernels
        self.stream_shapes = sorted({(int(t), int(d)) for t, d in re.findall(r"b->ntaps == (\d+) && D == (\d+)", b)})


K = Constants()
assert np.finfo(np.longdouble).nmant == 63, "the fixed-point steps are computed in x87 extended precision"


# ------------------------------------------------------------------ the reference
def tuner_inc(tuning, rate):
    """tuPhaseInc = 2.0*Math.PI*tuning/rate (:196), in the reference's operation order."""
    return (2.0 * math.pi * np.asarray(tuning, np.float64)) / float(rate)


def replay(p0, inc, S):
    """The reference recurrence for S samples from phase p0 (vectors over channels): the phase of every
    sample, [S, nchan], and the phase after the last."""
    p = np.array(p0, np.float64, copy=True)
    inc = np.asarray(inc, np.float64)
    out = np.empty((S, p.size))
    if p.size <= 8:                                 # few channels: Python floats are binary64 too, and faster
        for c in range(p.size):
            q, d, col = float(p[c]), float(inc[c]), out[:, c]
            two_pi = K.two_pi
            vals = []
            for _ in range(S):
                q += d
                if q > two_pi:
                    q -= two_pi
                vals.append(q)
            col[:] = vals
            p[c] = q
        return out, p
    for s in range(S):
        p = p + inc
        p = np.where(p > K.two_pi, p - K.two_pi, p)
        out[s] = p
    return out, p


def ref_index(p):
    """(int)(p*256/(2pi)) % 256 for p > 0, 256 (mixer bypass) otherwise (:388-390)."""
    p = np.asarray(p, np.float64)
    q = np.where(p > 0.0, (p * 256.0) / K.two_pi, 0.0)
    return np.where(p > 0.0, np.floor(q).astype(np.int64) & 255, 256)


# ------------------------------------------------------------------ exact arithmetic helpers
def _split(a):
    c = 134217729.0 * a
    hi = c - (c - a)
    return hi, a - hi


def two_prod(a, b):
    """a*b = p + e exactly (Dekker; no FMA needed)."""
    p = a * b
    ah, al = _split(a)
    bh, bl = _split(b)
    e = ((ah * bh - p) + ah * bl + al * bh) + al * bl
    return p, e


def boundary_offset(p):
    """Signed distance of the real quotient p*256/kTwoPi to its nearest integer, in table entries.

    t = 256p is exact, k = the nearest integer, k*kTwoPi = P + e exactly (two_prod), and t - P is exact
    (Sterbenz: t lies within kTwoPi/2 of k*kTwoPi).  The only roundings are (t - P) - e and the final
    division, so the result is within a relative 2^-52 of the true offset: far finer than any band
    edge used here (the coarsest distinction needed is 2^-44 absolute)."""
    t = np.asarray(p, np.float64) * 256.0
    k = np.rint(t / K.two_pi)
    P, e = two_prod(k, np.full_like(k, K.two_pi))
    return ((t - P) - e) / K.two_pi


def _rint_dd(h, l):
    """Round-half-even of the exact sum h + l (|l| <= ulp(h)/2) to an integer."""
    r = np.rint(h)
    d = (h - r) + l
    odd = np.mod(r, 2.0) != 0.0
    r = np.where((d > 0.5) | ((d == 0.5) & odd), r + 1.0, r)
    r = np.where((d < -0.5) | ((d == -0.5) & odd), r - 1.0, r)
    return r


def phase_to_x48(ph):
    """hi = ph*kIdxScaleHi, lo = fma(ph, kIdxScaleLo, fma(ph, kIdxScaleHi, -hi)), x = rn(hi*2^48) + rn(lo*2^48)
    as uint64.  The inner fma is exactly the product's rounding error e.  The outer one is first taken as
    (a + e) + b from the exact product a + b = ph*kIdxScaleLo, within an ulp of lo (2^-97) of the fused
    result; that can move rn(lo*2^48) only where lo*2^48 lies next to a half, and there lo is recomputed
    as the correctly rounded value of the exact ph*kIdxScaleLo + e (Python's Fraction -> float rounds
    correctly), so the result is the kernel's bit for bit."""
    ph = np.asarray(ph, np.float64)
    hi, e = two_prod(ph, np.full_like(ph, K.scale_hi))
    a, b = two_prod(ph, np.full_like(ph, K.scale_lo))
    lo = (a + e) + b
    v = lo * 281474976710656.0
    doubt = np.abs(np.abs(v - np.trunc(v)) - 0.5) < 2.0 ** -30
    if doubt.any():
        from fractions import Fraction
        lo = lo.copy()
        for i in zip(*np.nonzero(doubt)):
            lo[i] = float(Fraction(float(ph[i])) * Fraction(K.scale_lo) + Fraction(float(e[i])))

    def d2ll(v):                                    # __double2ll_rn: out of range -> 0x8000000000000000
        ok = np.abs(v) < 2.0 ** 63
        return np.where(ok, np.rint(np.where(ok, v, 0.0)), 0.0).astype(np.int64) | np.where(ok, 0, np.int64(-2 ** 63))
    xh = d2ll(hi * 281474976710656.0)
    xl = d2ll(lo * 281474976710656.0)
    with np.errstate(over="ignore"):
        return (xh + xl).view(U64)


def _fixed_step(inc, limit, scale):
    inc = float(inc)
    if not (inc > 0.0) or not (inc < limit):
        return 0
    c = np.longdouble(256) / np.longdouble(K.two_pi)
    d = np.fmod(np.longdouble(inc) * c, np.longdouble(256))
    v = int(d * np.longdouble(scale) + np.longdouble(0.5))
    return v if v else 1


def dx48(inc):
    """index_step_fixed: the per-sample index step in 2^-48 units (0: exact path)."""
    return _fixed_step(inc, K.dx48_limit, 2.0 ** 48)


def dx56(inc):
    """index_step_fixed56: the same in 2^-56 units (0: exact replay)."""
    return _fixed_step(inc, K.dx56_limit, 2.0 ** 56)


# ------------------------------------------------------------------ the three index paths
def table_index(p, guard=True):
    """table_index (bpsk.cu) for phases 0 < p < 16: (index, exact) where exact marks the samples whose
    quotient came within the guard of an integer and were decided by the IEEE division."""
    p = np.asarray(p, np.float64)
    assert np.all(p < 16.0)
    t = p * 256.0
    h, l = two_prod(t, np.full_like(t, K.inv_two_pi * 1048576.0))
    yi = _rint_dd(h, l).astype(np.int64)            # the low word of fma(t, c, 1.5*2^52)
    frac = yi & 0xfffff
    k = yi >> 20
    exact = (frac < K.ti_guard) | (frac > 1048576 - K.ti_guard) if guard else np.zeros(p.shape, bool)
    k = np.where(exact, np.floor(t / K.two_pi).astype(np.int64), k)
    return k & 255, exact


def tuner_index(p, guard=True):
    """tuner_index: table_index for p > 0, 256 otherwise; (index, exact, bypass)."""
    p = np.asarray(p, np.float64)
    pos = p > 0.0
    k, ex = table_index(np.where(pos, p, 1.0), guard)
    return np.where(pos, k, 256), ex & pos, ~pos


def tile_chunks(ckpt, dx, bound=None):
    """k_mixdecim phase 1 on chunks with checkpoints ckpt[nchunks, nchan] and steps dx[nchan] (8.48): the
    fast index of the 32 samples of every chunk [nchunks, 32, nchan] and whether the chunk takes the
    fast path [nchunks, nchan]."""
    bound = K.tile_bound if bound is None else bound
    ckpt = np.asarray(ckpt, np.float64)
    dx = np.asarray(dx, np.uint64)
    fast = (dx != 0)[None, :] & (ckpt >= 0.0)
    x = phase_to_x48(np.where(fast, ckpt, 0.0))
    idx = np.empty((ckpt.shape[0], 32, ckpt.shape[1]), np.int64)
    near = np.zeros(ckpt.shape, bool)
    with np.errstate(over="ignore"):
        for j in range(32):
            x = x + dx[None, :]
            xh = (x >> U64(32)).astype(np.int64)
            near |= ((xh + 1) & K.tile_mask) <= bound
            idx[:, j] = (xh >> 16) & 255
    return idx, fast & ~near


@dataclass
class StreamMutant:
    """Variants of k_mixdecim_stream's index path.  A sample is `near` when the 24 fraction bits of X_j
    lie in [lo, hi] units of 2^-24; the code has lo = -1, hi = D + near_plus - 1.  hi_abs fixes hi,
    hi_rel sets hi = D + hi_rel.  reanchor = periods between anchors (None: anchored only at the top of
    a segment)."""
    lo: int = -1
    hi_rel: int | None = None
    hi_abs: int | None = None
    reanchor: int | None = -1

    def window(self, D):
        if self.hi_abs is not None:
            return self.lo, self.hi_abs
        return self.lo, D + (K.near_plus - 1 if self.hi_rel is None else self.hi_rel)


def stream_layout(nchan, NO, s16=True, pump=False, sm_count=148):
    """launch_stream's segment length R (outputs per warp item) for a bank of nchan channels."""
    ncw = (nchan + 31) // 32
    st = K.scout_wide if (pump and nchan >= K.scout_big) else K.scout_narrow
    scout_ctas = (nchan + st - 1) // st
    grid = sm_count if pump else max(sm_count - scout_ctas, sm_count // 2)
    resident = grid * (K.warps_s16 if s16 else K.warps_f32)
    nseg = max(1, K.segs_per_warp * resident // ncw)
    R = max((NO + nseg - 1) // nseg, K.r_min)
    return R


def stream_block(ckpt, replayed, dx, D, ntaps, S, n0, NO, R, mut=StreamMutant()):
    """k_mixdecim_stream's table indices for one block, vectorised over channels.

    ckpt [nchunks, nchan]: the phase before every 32-sample chunk; replayed: tuner_index() of the
    reference's phases [S, nchan] (the exact replay is the reference's own arithmetic).  Returns one record
    per (segment, period, sample) the kernel evaluates: dict of arrays s, seam flags, used (the sample
    feeds a stored output), and per channel idx, path (0 fast, 1 replayed through table_index's fast
    path, 2 replayed and divided, 3 bypass)."""
    nchunks, nchan = ckpt.shape
    dx = np.asarray(dx, np.uint64)
    NQ = (ntaps + D - 1) // D
    nseg = (NO + R - 1) // R
    nper = R + NQ - 1
    reanchor = K.reanchor if mut.reanchor == -1 else mut.reanchor
    lo, hi = mut.window(D)
    ndx = ((U64(0) - (dx >> U64(32))) & U64(0xffffffff)).astype(np.int64)
    dxh_mask = np.int64(0xffffffff)
    exact_lane = dx == 0
    x56 = (phase_to_x48(ckpt.ravel()) << U64(8)).reshape(ckpt.shape)
    dxD = dx * U64(D)
    jj = np.arange(D)
    recs = []
    with np.errstate(over="ignore"):
        for seg in range(nseg):
            m_top = (seg + 1) * R - 1
            n_top = n0 + m_top * D
            x_top = np.zeros(nchan, U64)
            bad = np.zeros(nchan, bool)
            for tt in range(nper):
                s_hi = n_top - tt * D
                if (tt % reanchor == 0) if reanchor else tt == 0:
                    c = min(max(s_hi >> 5, 0), nchunks - 1)
                    ck = ckpt[c]
                    steps = np.uint64((s_hi - (c << 5) + 1) & M64)
                    x_top = x56[c] + steps * dx
                    c_lo = min(max((s_hi - K.reanchor * D + 1) >> 5, 0), nchunks - 1)
                    bad = ~(ck >= 0.0) | ~(ckpt[c_lo] >= 0.0)
                xt = (x_top >> U64(32)).astype(np.int64)
                x_top = x_top - dxD
                xj = (xt[:, None] + jj[None, :] * ndx[:, None]) & dxh_mask          # [nchan, D]
                idx = (xj >> 24) & 255
                frac = xj & 0xffffff
                near = ((frac - lo) & 0xffffff) <= (hi - lo)
                lane_near = exact_lane | bad | near.any(axis=1)
                s = s_hi - jj
                path = np.zeros((nchan, D), np.int64)
                if lane_near.any():
                    sv = np.clip(s, 0, S - 1)
                    ti, ex, byp = (a[sv][:, lane_near].T for a in replayed)          # [nlanes, D]
                    idx[lane_near] = ti
                    path[lane_near] = np.where(byp, 3, np.where(ex, 2, 1))
                # which samples feed a stored output: role q of this period is output tt - q
                used = np.zeros(D, bool)
                for q in range(NQ):
                    r = tt - q
                    if 0 <= r < R and m_top - r < NO:
                        used |= jj + q * D < ntaps
                used &= (s >= 0) & (s < S)
                recs.append(dict(s=s, used=used, idx=idx.T, path=path.T,
                                 seam_period=(jj == 0) | (jj == D - 1),
                                 seam_anchor=np.full(D, (tt % K.reanchor) in (0, K.reanchor - 1)),
                                 seam_segment=np.full(D, tt in (0, nper - 1))))
    if not recs:
        return None
    out = {k: np.concatenate([r[k] for r in recs]) for k in ("s", "used", "idx", "path", "seam_period", "seam_anchor", "seam_segment")}
    return out


# ------------------------------------------------------------------ a whole bank, block by block
def bands(D):
    """Upper edges of the distance bands (table entries) and their names."""
    e = [2.0 ** -44, 2.0 ** -36, 2.0 ** -24, (D + 2) * 2.0 ** -24, 2.0 ** -16, K.ti_guard * 2.0 ** -20, np.inf]
    names = ["<2^-44", "2^-44..2^-36", "2^-36..2^-24", f"2^-24..{D + 2}*2^-24", f"{D + 2}*2^-24..2^-16",
             "2^-16..6e-5", ">6e-5"]
    return np.array(e), names


@dataclass
class Plan:
    """A bank's input: its rate, the block lengths, and every channel's tuning for each block (a change
    between blocks is a retune)."""
    rate: int
    lens: list
    tunings: list                    # [nblocks] arrays of Hz
    what: str = ""
    zeros: list = field(default_factory=list)        # (channel, block, sample) where the phase is exactly 0.0
    crossings: list = field(default_factory=list)    # (channel, block, sample): first phase > 0 after a climb

    @property
    def nchan(self):
        return len(self.tunings[0])


@dataclass
class Tally:
    """What the emulation of one kernel saw: wrong indices on used samples, and per path and distance
    band how many used samples there were, overall and at each seam."""
    wrong: int = 0
    wrong_where: list = field(default_factory=list)
    counts: dict = field(default_factory=dict)

    def add(self, key, n):
        self.counts[key] = self.counts.get(key, 0) + int(n)


def kernel_for(mode, nchan, NO, ntaps, D, prec_f32=False):
    """mix_decimate's choice: 'stream' or 'tile' (mode 0 auto, 1 tile, 2 stream)."""
    if NO <= 0:
        return None
    if mode != 1:
        shape_ok = (ntaps, D) in K.stream_shapes
        want = mode == 2 or (nchan >= 32 and NO >= 64) or (prec_f32 and nchan >= 8)
        if shape_ok and want:
            return "stream"
    return "tile"


def simulate(plan, mode, ntaps=27, s16=True, pump=False, channels=None, mutants=(None,), sm_count=148):
    """Emulate the bank's table indices over every block of `plan` and compare each used sample's index
    with the reference's.  mode: 0 auto, 1 tile, 2 stream; mutants: names from MUTANTS (None: the code as
    it is).  Returns {mutant: {kernel: Tally}} with kernels 'stream', 'tile' and 'table_index'."""
    rate = plan.rate
    D = rate // 9600
    H = ntaps - 1
    chans = np.arange(plan.nchan) if channels is None else np.asarray(channels)
    nch = chans.size
    out = {m: {k: Tally() for k in ("stream", "tile", "table_index")} for m in mutants}
    p = np.zeros(nch)
    ds_cnt = 0
    for blk, S in enumerate(plan.lens):
        inc = tuner_inc(np.asarray(plan.tunings[blk])[chans], rate)
        NO = (ds_cnt + S) // D
        n0 = D - 1 - ds_cnt
        if S == 0:
            continue
        ph, p_end = replay(p, inc, S)
        nchunks = (S + 31) // 32
        ckpt = np.vstack([p[None, :], ph[31:S - 1:32]])[:nchunks]
        ref = ref_index(ph)                                             # [S, nch]
        dist = np.abs(boundary_offset(ph))
        blk_edge = lambda s: (s == 0) | (s == S - 1)
        kern = kernel_for(mode, plan.nchan, NO, ntaps, D)
        # samples of this block that feed an output of this block
        s_all = np.arange(S)
        m_min = np.maximum(-((n0 - s_all) // D), 0)                     # first output at or after sample s
        used_s = (m_min < NO) & (n0 + m_min * D - s_all < ntaps)
        count = True
        replayed = {}
        for mutant, tallies in out.items():
            mut = MUTANTS[mutant] if mutant else {}
            ti_guard = mut.get("ti_guard", True)
            if ti_guard not in replayed:
                replayed[ti_guard] = tuner_index(ph, ti_guard)
            ti, ex, byp = replayed[ti_guard]
            if kern == "stream":
                R = stream_layout(plan.nchan, NO, s16, pump, sm_count)
                dxs = np.array([dx56(v) for v in inc], np.uint64)
                r = stream_block(ckpt, replayed[ti_guard], dxs, D, ntaps, S, n0, NO, R, mut.get("stream", StreamMutant()))
                sv = np.clip(r["s"], 0, S - 1)
                used = r["used"][:, None] & np.ones((1, nch), bool)
                seams = {"any": np.ones(sv.size, bool), "chunk": (sv % 32 == 0) | (sv % 32 == 31),
                         "period": r["seam_period"], "anchor": r["seam_anchor"], "segment": r["seam_segment"],
                         "block": blk_edge(r["s"])}
                _tally_kernel(tallies, "stream", r["idx"], r["path"], ref[sv], dist[sv], used, seams, D, blk, r["s"], count)
            elif kern == "tile":
                fidx, fast = tile_chunks(ckpt, [dx48(v) for v in inc], mut.get("tile_bound"))
                ff = np.repeat(fast, 32, axis=0)[:S]
                idx = np.where(ff, fidx.reshape(-1, nch)[:S], ti)
                path = np.where(ff, 0, np.where(byp, 3, np.where(ex, 2, 1)))
                used = used_s[:, None] & np.ones((1, nch), bool)
                seams = {"any": np.ones(S, bool), "chunk": (s_all % 32 == 0) | (s_all % 32 == 31), "block": blk_edge(s_all)}
                _tally_kernel(tallies, "tile", idx, path, ref, dist, used, seams, D, blk, s_all, count)
            # k_tuner_tail: the last H mixed samples become the next block's history
            if H > 0:
                st = np.arange(max(S - H, 0), S)
                tpath = np.where(byp[st], 3, np.where(ex[st], 2, 1))
                seams = {"any": np.ones(st.size, bool), "block": blk_edge(st)}
                _tally_kernel(tallies, "tail", ti[st], tpath, ref[st], dist[st], np.ones(tpath.shape, bool), seams, D, blk, st, count)
            count = False                           # (the bands are tallied for the first variant only)
        p = p_end
        ds_cnt = (ds_cnt + S) % D
    return out


def _tally_kernel(tallies, kern, idx, path, ref, dist, used, seams, D, blk, s, count=True):
    """Count wrong indices among the used samples, and the used samples per path, band and seam.  The
    kernel's own fast path counts under the kernel; every replayed sample also counts under
    table_index, as its fast path (path 1) or its exact division (path 2)."""
    bad = used & np.where(path == 3, ref != 256, idx != ref)
    t = tallies["table_index" if kern == "tail" else kern]
    if bad.any():
        t.wrong += int(bad.sum())
        t.wrong_where += [(blk, int(s[i]), int(c)) for i, c in np.argwhere(bad)[:3]]
    if not count:
        return
    edges, names = bands(D)
    band = np.searchsorted(edges, dist, side="right")
    groups = [] if kern == "tail" else [(t, "fast", path == 0), (t, "replay", (path == 1) | (path == 2)),
                                        (t, "bypass", path == 3)]
    ti = tallies["table_index"]
    groups += [(ti, "fast", path == 1), (ti, "exact", path == 2)]
    for tal, pname, sel in groups:
        sel = sel & used
        if not sel.any():
            continue
        for seam, flag in seams.items():
            if tal is ti and seam != "any":
                continue
            m = sel & flag[:, None]
            if m.any():
                cnt = np.bincount(band[m], minlength=len(names))
                for i in np.nonzero(cnt)[0]:
                    tal.add((pname, names[i], seam), cnt[i])


MUTANTS = {
    "stream window [0, 1] (no borrow margin)": {"stream": StreamMutant(lo=0, hi_abs=1)},
    "stream window one short at the bottom [0, D+1]": {"stream": StreamMutant(lo=0)},
    "stream window one short at the top [-1, D]": {"stream": StreamMutant(hi_rel=K.near_plus - 2)},
    "tile guard one-sided (== 0)": {"tile_bound": 0},
    "table_index without its guard": {"ti_guard": False},
    "stream anchor not refreshed within a segment": {"stream": StreamMutant(reanchor=None)},
}


# ------------------------------------------------------------------ the inputs
G = 0.7548776662466927        # 1/(the plastic ratio): far from any short binary fraction
NEAR_K = (1, 7, 32, 63, 101, 126, 127)
NEAR_M = (14, 16, 18, 20, 22, 24, 26, 28, 30, 33, 36, 40, 44, 50)
ON_K = (1, 7, 16, 32, 64, 101, 126, 127)


def near_grid(rate, ks=NEAR_K, ms=NEAR_M, g=G):
    """rate*(k + s*g*2^-m)/256: the index advances by k + s*g*2^-m table entries per sample, so from a
    phase on the grid the fraction creeps away from (s = +1) or towards (s = -1) a boundary by g*2^-m
    per sample, and the samples of a block spread over every band from 2^-m up.  k = 126 and 127 sit
    on either side of the streaming kernel's inc < 3.1 cut-off (above it: exact replay only)."""
    return [rate * (k + s * g * 2.0 ** -m) / 256 for k in ks for s in (1, -1) for m in ms]


def on_grid(rate, ks=ON_K):
    """rate*k/256: every sample a whole number of table entries from the start, up to the rounding
    of the accumulation (the band below 2^-44, where the quotient's own rounding decides)."""
    return [rate * k / 256 for k in ks]


def tuning_for_inc(a, rate):
    """A tuning whose increment 2.0*Math.PI*tuning/rate is exactly the double a, or None (about one
    double in two is reachable from some tuning)."""
    lo = hi = a * rate / (2.0 * math.pi)
    for _ in range(64):
        for c in (lo, hi):
            if (2.0 * math.pi * c) / float(rate) == a:
                return c
        lo, hi = math.nextafter(lo, -math.inf), math.nextafter(hi, math.inf)
    return None


def dyadic_return(rate, L0, s):
    """Tunings (down, up) with increments -a1 and +a2, short binary fractions with L0*a1 = (s+1)*a2, so
    that after L0 samples down and s+1 samples up the phase is exactly 0.0 (every partial sum exact)."""
    for e in range(10, 24):
        for q in range(1, 64, 2):
            a1, a2 = (s + 1) * q * 2.0 ** -e, L0 * q * 2.0 ** -e
            if a2 >= K.dx56_limit:
                continue
            down, up = tuning_for_inc(-a1, rate), tuning_for_inc(a2, rate)
            if down is not None and up is not None:
                return down, up
    raise ValueError(f"no short binary increments return to 0.0 at sample {s}")


def crossing_targets(rate, S1, R, n0):
    """Samples of a block at which a climb through phase 0 is placed: the tops of the first segments of
    the streaming kernel (R outputs each, the first at sample n0), its anchors and the low ends of their
    windows, and 32-sample chunk edges, each with its neighbour."""
    D = rate // 9600
    t = set()
    for seg in range(3):
        n_top = n0 + ((seg + 1) * R - 1) * D
        for tt in range(0, R, K.reanchor):
            s_hi = n_top - tt * D
            lo = s_hi - K.reanchor * D + 1
            t |= {s_hi, s_hi + 1, lo, lo - 1, (lo >> 5) << 5, ((lo >> 5) << 5) - 1}
    t |= {1, 31, 32, 33}
    return sorted(s for s in t if 1 <= s < S1)


def crossing_tunings(rate, L0, targets, dyadic_targets):
    """Channels that run backwards (negative tuning) through a first block of L0 samples and are then
    retuned positive so that the first sample with phase > 0 is targets[i] of the second block.
    dyadic_targets: channels whose increments are short binary fractions (dyadic_return), so that the
    phase returns to exactly 0.0 at sample s (which must take the mixer bypass) and is positive from
    s+1.  Returns (tunings of block 0, tunings of the later blocks)."""
    t0, t1 = [], []
    for i, s in enumerate(targets):
        a = 2.0 * math.pi * (1 + (37 * i) % 125 + G) / 256.0          # the climb's increment, below 3.1
        down = -(s + 0.5) * a / L0 * rate / (2.0 * math.pi)
        (p,) = replay([0.0], tuner_inc([down], rate), L0)[1]
        up = (-p / (s + 0.5)) * rate / (2.0 * math.pi)
        t0.append(down)
        t1.append(up)
    for s in dyadic_targets:
        down, up = dyadic_return(rate, L0, s)
        t0.append(down)
        t1.append(up)
    return t0, t1


def bank_plan(rate, lens=(2500, 9000, 333, 20000, 1, 4097), s16=True, pump=False, sm_count=148):
    """The inputs of the GPU tests: every near-grid and on-grid tuning, from phase 0 in the first block,
    carried through ragged blocks; half of the near-grid channels retuned to each other's frequencies
    before the fourth block (so that they start mid-phase); and channels whose phase climbs through 0
    at the seams of the second block, including exact returns to 0.0.  The seams are those of the
    streaming kernel's segments on a device of sm_count SMs; the plan checks that every block of the
    bank it describes has that segment length."""
    D = rate // 9600
    lens = list(lens)
    base = near_grid(rate) + on_grid(rate)
    L0 = lens[0]
    n0_1 = D - 1 - L0 % D
    R = K.r_min
    targets = crossing_targets(rate, lens[1], R, n0_1)
    dy = [s for s in targets if s < 3000][:12]
    c0, c1 = crossing_tunings(rate, L0, targets, dy)
    first = np.array(base + c0)
    later = np.array(base + c1)
    swapped = later.copy()
    half = np.arange(0, len(NEAR_K) * 2 * len(NEAR_M), 2)
    swapped[half] = later[half[::-1]]
    tunings = [first] + [later] * 2 + [swapped] * (len(lens) - 3)
    ds_cnt = 0
    for S in lens:
        NO = (ds_cnt + S) // D
        assert stream_layout(len(first), NO, s16, pump, sm_count) == R, "the crossings would miss the segment seams"
        ds_cnt = (ds_cnt + S) % D
    first_dyadic = len(base) + len(targets)
    zeros = [(first_dyadic + i, 1, s) for i, s in enumerate(dy)]
    crossings = [(len(base) + i, 1, s) for i, s in enumerate(targets)]
    return Plan(rate, lens, tunings, what=f"{rate} S/s, {len(first)} channels, blocks {lens}",
                zeros=zeros, crossings=crossings)
