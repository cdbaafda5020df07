"""demod.java's NCO (:423-433) as k_demod / k_demod_s16 compute it, restated on the CPU bit for bit,
and the inputs that drive the GPU through the phase recurrence's edges.

The phase.  car is a float accumulator, `car -= phi; if (car < 0) car += (float)(2 pi)` (:427-429),
data independent; oracle.demod_phases replays it in C (orc_demod_phases, next to orc_demod_receive).
For 0 <= phi < 2 pi it stays in [0, 2 pi] and returns exactly to 0.0 for many tunings (the sequence
is then periodic from there); for phi < 0 (flo < 0, a lower-sideband passband) it grows without
bound until car - phi rounds back to car, and for phi >= 2 pi (flo >= rate) it runs negative.

The sine and cosine.  For |car| <= 8 the kernel evaluates `nco_sincos` (csrc/demod_fir.cu): one
Cody-Waite step and two minimax polynomials in binary64, every step a fused multiply-add, then
rounded to float.  `kernel_sincos` restates it vectorised with each FMA as a multiply and an add,
and recomputes with every FMA exact (Fractions) the samples whose binary64 result lies within
BAND binary64 ulps of a float rounding midpoint: everywhere else the two chains round to the same
float.  BAND is four times the largest distance between the two chains measured by
tests/test_nco_model.py, not assumed.  Beyond |car| > 8 (and NaN) the kernel calls the CUDA
library's binary64 sincos (documented to 2 ulps) and rounds that; the reference there is the
correctly rounded float, and samples whose true value lies within SLOW_DOUBT binary64 ulps of a
float midpoint accept either neighbour.

`mix_reference` is then the whole down-shift (:432-433) with one float rounding per operation.
"""
from __future__ import annotations

import functools
from fractions import Fraction

import mpmath
import numpy as np

import oracle as O
from test_nco_sincos import coefficients

TWOPI = np.float32(2 * np.pi)           # (float)(2 * Math.PI)
MAGIC = 6755399441055744.0              # 1.5 * 2^52
BAND = 8                                # binary64 ulps; >= 4x the measured mul+add vs FMA distance
LIBM_BAND = 16                          # binary64 ulps; >= 4x numpy's measured sin / cos error
SLOW_DOUBT = 3                          # CUDA's binary64 sin / cos: 2 ulps, plus one
CHUNK, TILE = 32, 1024                  # k_car_scout checkpoints, k_demod tile
RATES = (44100, 96000, 192000)
LONG_FLO = -15278                       # 96 kS/s: phi = -0.99994, just inside a power of two (stall_flo)
LONG_CALLS = (4194560,) * 4             # 2^24 + 1024 samples: past the stall at sample 2^24 + 1


# ------------------------------------------------------------------ the phase
def phi_of(flo: int, rate: int) -> np.float32:
    """demod.java:350-368: phi = (float)(2 pi * ((float)flo / (float)rate))."""
    nlo = np.float32(np.float32(flo) / np.float32(rate))
    return np.float32(2 * np.pi * np.float64(nlo))


def phases(phi, car0, n: int) -> np.ndarray:
    """float32[n + 1]: car of each of n samples from car0, then the value carried on."""
    return O.demod_phases(np.float32(phi), np.float32(car0), n)


def phases_variant(phi, car0, n: int, wrap_le=False, f64=False) -> np.ndarray:
    """The recurrence with one deliberate change, for tests of the checker's power: the wrap on
    `car <= 0`, or the chain carried in binary64 and rounded to float at every 32-sample
    checkpoint (each sample sees the binary64 value rounded)."""
    out = np.empty(n + 1, np.float32)
    phi32 = np.float32(phi)
    if f64:
        car = float(np.float32(car0))
        for k in range(n):
            if k % CHUNK == 0:
                car = float(np.float32(car))
            out[k] = np.float32(car)
            car -= float(phi32)
            if car < 0:
                car += float(TWOPI)
        out[n] = np.float32(car)
        return out
    car = np.float32(car0)
    for k in range(n):
        out[k] = car
        car = np.float32(car - phi32)
        if (car <= 0) if wrap_le else (car < 0):
            car = np.float32(car + TWOPI)
    out[n] = car
    return out


# ------------------------------------------------------------------ nco_sincos
def _chain(x, fma, mul, sub):
    """nco_sincos's binary64 steps on x = (double)car with the given fma / mul / sub: returns
    (k, sine kernel before its float rounding, cosine kernel before its float rounding)."""
    c = coefficients()
    t = fma(x, c[12], MAGIC)
    kd = sub(t, MAGIC)
    r = fma(-kd, c[13], x)
    r = fma(-kd, c[14], r)
    z = mul(r, r)
    ps = fma(z, c[5], c[4])
    for i in (3, 2, 1, 0):
        ps = fma(z, ps, c[i])
    fs = fma(mul(z, r), ps, r)
    pc = fma(z, c[11], c[10])
    for i in (9, 8, 7, 6):
        pc = fma(z, pc, c[i])
    fc = fma(mul(z, z), pc, fma(z, -0.5, 1.0))
    return kd, fs, fc


def _quadrant(kd, fs, fc):
    k = np.asarray(kd).astype(np.int64)
    fs = np.asarray(fs, np.float64).astype(np.float32)
    fc = np.asarray(fc, np.float64).astype(np.float32)
    a = np.where(k & 1, fc, fs)
    b = np.where(k & 1, fs, fc)
    return np.where(k & 2, -a, a).astype(np.float32), np.where((k + 1) & 2, -b, b).astype(np.float32)


def chain_muladd(car):
    """The chain vectorised, each FMA a binary64 multiply and add."""
    x = np.asarray(car, np.float32).astype(np.float64)
    return _chain(x, lambda a, b, c: a * b + c, lambda a, b: a * b, lambda a, b: a - b)


def _fma_frac(a, b, c):
    return float(Fraction(a) * Fraction(b) + Fraction(c))      # correctly rounded (Fraction.__float__)


def chain_exact_scalar(car: float):
    """The chain for one phase with every __fma_rn exact: the kernel's own binary64 values."""
    return _chain(float(np.float32(car)), _fma_frac, lambda a, b: a * b, lambda a, b: a - b)


def _two_prod(a, b):
    p = a * b
    sa = 134217729.0 * a
    ah = sa - (sa - a)
    al = a - ah
    sb = 134217729.0 * b
    bh = sb - (sb - b)
    bl = b - bh
    return p, ((ah * bh - p) + ah * bl + al * bh) + al * bl


def _two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


def fma_exact_vec(a, b, c):
    """RN(a*b + c) for binary64 arrays without an FMA instruction: Boldo and Melquiond's emulation
    (exact product and sum, then the low parts added with rounding to odd).  Checked against
    Fractions by tests/test_nco_model.py on the chain's own operands."""
    a, b, c = np.broadcast_arrays(*(np.asarray(v, np.float64) for v in (a, b, c)))
    uh, ul = _two_prod(a, b)
    th, tl = _two_sum(c, uh)
    s, e = _two_sum(tl, ul)
    odd = (s.view(np.int64) & 1) == 1
    v = np.where((e != 0) & ~odd, np.nextafter(s, np.where(e > 0, np.inf, -np.inf)), s)
    return th + v


def chain_exact_vec(car):
    x = np.asarray(car, np.float32).astype(np.float64)
    return _chain(x, fma_exact_vec, lambda a, b: a * b, lambda a, b: a - b)


def midpoint_ulps(d) -> np.ndarray:
    """Distance of each binary64 value from the nearest rounding midpoint between two floats, in
    binary64 ulps of the value (inf for values that do not round: NaN, inf)."""
    d = np.asarray(d, np.float64)
    with np.errstate(all="ignore"):
        f = d.astype(np.float32)
        lo = (f.astype(np.float64) + np.nextafter(f, np.float32(-np.inf)).astype(np.float64)) / 2
        hi = (f.astype(np.float64) + np.nextafter(f, np.float32(np.inf)).astype(np.float64)) / 2
        dist = np.minimum(np.abs(d - lo), np.abs(d - hi)) / np.spacing(np.abs(d))
    return np.where(np.isfinite(d) & np.isfinite(dist), dist, np.inf)


def near_half(car) -> np.ndarray:
    """Phases whose quadrant k = nearest(car * 2/pi) the multiply-and-add form might pick
    differently from the FMA (car * 2/pi within 2^-40 of a half-integer)."""
    y = np.asarray(car, np.float32).astype(np.float64) * coefficients()[12]
    return np.abs(np.abs(y - np.round(y)) - 0.5) < 2.0 ** -40


def kernel_sincos(car, stats: dict | None = None):
    """(sin, cos) as nco_sincos returns them for |car| <= 8 (float32 arrays); other entries NaN."""
    car = np.asarray(car, np.float32)
    kd, fs, fc = chain_muladd(car)
    sn, cs = _quadrant(kd, fs, fc)
    fast = np.abs(car) <= 8
    doubt = np.flatnonzero(fast & (near_half(car) | (midpoint_ulps(fs) <= BAND) | (midpoint_ulps(fc) <= BAND)))
    for i in doubt:
        e = _quadrant(*[np.array([v]) for v in chain_exact_scalar(float(car.flat[i]))])
        sn.flat[i], cs.flat[i] = e[0][0], e[1][0]
    if stats is not None:
        stats["doubt"] = stats.get("doubt", 0) + doubt.size
    sn = np.where(fast, sn, np.float32(np.nan))
    cs = np.where(fast, cs, np.float32(np.nan))
    return sn.astype(np.float32), cs.astype(np.float32)


# ------------------------------------------------------------------ correctly rounded float
def _mp_f32(v) -> tuple[np.float32, float]:
    """The float nearest to the mpf v (rounded straight to 24 bits, no binary64 step) and v's
    distance from the nearest float midpoint in binary64 ulps of v."""
    with mpmath.workprec(24):
        f = np.float32(float(+v))
    fd = float(f)
    up = float(np.nextafter(f, np.float32(np.inf)))
    dn = float(np.nextafter(f, np.float32(-np.inf)))
    m = min(abs(v - (fd + up) / 2), abs(v - (fd + dn) / 2))
    return f, float(m) / float(np.spacing(abs(float(v))))


@functools.lru_cache(maxsize=None)
def _mp_sincos(c: float):
    with mpmath.workprec(200):
        x = mpmath.mpf(c)
        return _mp_f32(mpmath.sin(x)), _mp_f32(mpmath.cos(x))


def cr_sincos(car):
    """Correctly rounded float sin and cos of every float in car, and the distance of each true
    value from a float midpoint (binary64 ulps; inf where numpy's value is far from any):
    numpy's binary64 value rounded, and mpmath at 200 bits wherever that lies within LIBM_BAND."""
    car = np.asarray(car, np.float32)
    x = car.astype(np.float64)
    ds, dc = np.sin(x), np.cos(x)
    sn, cs = ds.astype(np.float32), dc.astype(np.float32)
    dist_s, dist_c = np.full(car.shape, np.inf), np.full(car.shape, np.inf)
    for i in np.flatnonzero((midpoint_ulps(ds) <= LIBM_BAND) | (midpoint_ulps(dc) <= LIBM_BAND)):
        (s, s_d), (c, c_d) = _mp_sincos(float(car.flat[i]))
        sn.flat[i], cs.flat[i], dist_s.flat[i], dist_c.flat[i] = s, c, s_d, c_d
    return sn, cs, dist_s, dist_c


def _other(f, v64):
    """The float on the other side of the midpoint nearest to f's exact value."""
    up, dn = np.nextafter(f, np.float32(np.inf)), np.nextafter(f, np.float32(-np.inf))
    return np.where(v64 > f.astype(np.float64), up, dn).astype(np.float32)


# ------------------------------------------------------------------ the down-shift
def _mix(fir_out, ci, cq):
    a, b = fir_out[0::2], fir_out[1::2]
    out = np.empty_like(fir_out)
    out[0::2] = a * ci - b * cq                 # :432, float32 products and difference, each rounded
    out[1::2] = a * cq + b * ci                 # :433
    return out


def sincos_reference(car, stats: dict | None = None):
    """(sin, cos, alt_sin, alt_cos): the kernel's floats (the fast path emulated, the correctly
    rounded float beyond |car| > 8 and for NaN) and, where a library-path value lies within
    SLOW_DOUBT ulps of a float midpoint, the other neighbour (elsewhere equal to the first)."""
    car = np.asarray(car, np.float32)
    slow = ~(np.abs(car) <= 8)
    sn = np.full(car.shape, np.nan, np.float32)
    cs = sn.copy()
    fast = np.flatnonzero(~slow)
    sn[fast], cs[fast] = kernel_sincos(car[fast], stats)
    alt_s, alt_c = sn.copy(), cs.copy()
    if slow.any():
        idx = np.flatnonzero(slow)
        s, c, ds_, dc_ = cr_sincos(car[idx])
        sn[idx], cs[idx] = s, c
        alt_s[idx], alt_c[idx] = s, c
        x = car[idx].astype(np.float64)
        ms, mc = ds_ <= SLOW_DOUBT, dc_ <= SLOW_DOUBT
        alt_s[idx[ms]] = _other(s[ms], np.sin(x[ms]))
        alt_c[idx[mc]] = _other(c[mc], np.cos(x[mc]))
        if stats is not None:
            stats["slow"] = stats.get("slow", 0) + idx.size
            stats["slow_doubt"] = stats.get("slow_doubt", 0) + int((ms | mc).sum())
    return sn, cs, alt_s, alt_c


def mix_reference(fir_out, car_trace, stats: dict | None = None):
    """The FIR-only output of the oracle (O.Demod(rate, dofir, False), interleaved float32) down-
    shifted by the phases car_trace[:n] as k_demod does: returns (out, allowed) where `allowed` is
    a list of further outputs that differ from `out` only at library-path samples within
    SLOW_DOUBT ulps of a float midpoint (empty when there are none)."""
    fir_out = np.asarray(fir_out, np.float32)
    n = fir_out.size // 2
    sn, cs, alt_s, alt_c = sincos_reference(np.asarray(car_trace, np.float32)[:n], stats)
    out = _mix(fir_out, cs, sn)
    allowed = []
    if not (np.array_equal(sn, alt_s) and np.array_equal(cs, alt_c)):
        allowed = [_mix(fir_out, c, s) for c, s in ((alt_c, sn), (cs, alt_s), (alt_c, alt_s))]
    return out, allowed


def matches(got, ref, allowed=()) -> bool:
    """Every float of got equal (bit for bit) to ref's, or at a doubtful sample to an allowed one."""
    g = np.ascontiguousarray(got, np.float32).view(np.uint32)
    ok = g == np.ascontiguousarray(ref, np.float32).view(np.uint32)
    for a in allowed:
        ok |= g == np.ascontiguousarray(a, np.float32).view(np.uint32)
    return bool(ok.all())


class RefDemod:
    """demod.java's receive up to the down-shift, from the oracle's FIR and this module's mix: the
    oracle carries the delay line (with the NCO off) and this class the phase, as the Java does
    (weights() with flo == INT_MIN keeps phi and car, any other resets car; set_flags with dodwn
    off leaves car where it is)."""

    def __init__(self, rate: int, dofir: bool = True, dodwn: bool = True):
        self.rate, self.dodwn = rate, dodwn
        self.fir = O.Demod(rate, dofir, False)
        self.phi, self.car = np.float32(0), np.float32(0)
        self.stats: dict = {}

    def weights(self, flo: int, fhi: int):
        self.fir.weights(flo, fhi)
        if flo != O.INT_MIN:
            self.phi, self.car = phi_of(flo, self.rate), np.float32(0)

    def set_flags(self, dofir: bool, dodwn: bool):
        self.fir.s.dofir = int(dofir)
        self.dodwn = dodwn

    def receive(self, buf):
        """(out, allowed) for one block, as mix_reference returns them."""
        y = self.fir.receive(buf)
        if not self.dodwn:
            return y, []
        tr = phases(self.phi, self.car, y.size // 2)
        self.car = tr[-1]
        return mix_reference(y, tr, self.stats)


# ------------------------------------------------------------------ the input plan
@functools.lru_cache(maxsize=None)
def zero_returns(rate: int, nmax: int = 4096) -> tuple:
    """((flo, m), ...) for every flo in (-rate, 2 rate) whose phase from car = 0 returns exactly
    to 0.0 at some sample m <= nmax, the first such m (the sequence has period m from there).
    flo <= 0 never returns: car only grows."""
    flo = np.arange(1, 2 * rate, dtype=np.int64)
    nlo = (flo.astype(np.float32) / np.float32(rate)).astype(np.float32)
    phi = (2 * np.pi * nlo.astype(np.float64)).astype(np.float32)
    car = np.zeros_like(phi)
    first = np.zeros(flo.size, np.int64)
    for m in range(1, nmax + 1):
        car -= phi
        np.add(car, TWOPI, out=car, where=car < 0)
        first[(car == 0) & (first == 0)] = m
    sel = np.flatnonzero(first)
    return tuple((int(flo[i]), int(first[i])) for i in sel)


SEAMS = (0, 31, 32, 33, TILE - 1, TILE)     # positions within a call: chunk and tile seams


def placement(m: int, q: int) -> int:
    """Length of the prefix call that puts a return to 0.0 (period m from car = 0) at position q
    of the next call: the smallest P >= 0 with P + q a multiple of m."""
    return (-q) % m


def planned_tunings(rate: int) -> list:
    """Tunings whose phase leaves the fast path's comfortable range or sits on its edges: 0,
    rate/2, just below rate, rate and above (phi >= 2 pi: car runs negative), and negative flo
    (car grows past 8 to the library path)."""
    return [0, rate // 2, rate - 1, rate, rate + 1, rate + rate // 3, -100, -rate // 7, -rate // 2, -rate + 1]


def stall_flo(rate: int) -> int:
    """A negative flo whose |phi| lies just below a power of two (1.0): car then climbs to 2^24,
    where car - phi rounds back to car, in about 2^24 samples."""
    f = -int(rate / (2 * np.pi))
    while abs(float(phi_of(f, rate))) >= 1.0:
        f += 1
    return f


def stall_point(phi, n: int) -> int:
    """The first sample of n from car = 0 whose car no longer moves (car - phi == car), or -1."""
    tr = phases(phi, 0.0, n)
    still = np.flatnonzero(np.float32(tr[:-1] - np.float32(phi)) == tr[:-1])
    return int(still[0]) if still.size else -1
