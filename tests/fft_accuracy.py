"""Binary64 reference and error bounds for the FFT / PSD kernels (fft_kernels.cuh,
fft_fourstep.cuh, fft_generic.cu).

The parity bar of tests/test_gpu_parity.py (1e-4 of full scale) is the contract with the Java
reference; it is not a test of the transform.  One wrong input sample moves every bin by at most
2|d|/N of full scale, which that bar cannot see at N >= 16384.  The checks here hold every block
to the normwise error bound of a correct binary32 FFT instead:

    ||X^ - X||_2 / ||X||_2 <= B(N),

X the binary64 spectrum of exactly the input the kernel saw.  A correct binary32 FFT sits about
100x below B(N); one wrong sample in full-range noise sits 200x or more above it.
tests/test_fft_accuracy_model.py shows both on the CPU, tests/test_gpu_fft_accuracy.py applies
the checks to every path the dispatcher can pick.
"""
import functools
import math
import os
import re

import numpy as np

# One length per path the dispatcher can pick (fft.cu: find_plan, split_plan, the four-step
# pair, then the staged path), from fft_plans.h and Plan in fft_kernels.cuh.
MULTI_BLOCK = [128, 256, 512, 1024]                 # G = 8, 8, 4, 4 blocks per CTA
ORDINARY = [2048, 4096, 4800, 4410, 8192, 9600]     # 2-4 passes; 4410 EARLY (s16); 8192, 9600 TW_SMEM_NP
PERSISTENT = [16384, 19200]                         # s16: persistent CTAs (PREFETCH / L2_NEXT + EARLY, TWP)
SPLIT = [32768]                                     # two 16384-point CTAs per block
FOUR_STEP = [65536]                                 # 256 x 256, chunks of 64 blocks on two streams
STAGED = [2, 3, 7, 100, 1000, 2401, 3125, 6000, 6561, 49152]   # fft_generic.cu
LENGTHS = MULTI_BLOCK + ORDINARY + PERSISTENT + SPLIT + FOUR_STEP + STAGED

U = 2.0 ** -24                     # unit round-off of binary32
MU = 16 * U                        # twiddle error assumed where none is measured (see plan_mu)
FLT_MAX = float(np.finfo(np.float32).max)
PLANS_H = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "java-sdr_b200", "csrc", "fft_plans.h")


@functools.lru_cache(maxsize=None)
def plans():
    """fft_plans.h: N -> (threads per CTA, blocks per CTA, radices in pass order)."""
    with open(PLANS_H) as fh:
        rows = re.findall(r"X\(\s*(\d+)\s*,\s*(\d+)\s*,\s*(\d+)\s*,\s*(\d+)\s*,\s*(\d+)\s*,\s*(\d+)\s*,\s*(\d+)\s*\)", fh.read())
    out = {}
    for r in rows:
        n, t, g, *rad = (int(v) for v in r)
        out[n] = (t, g, tuple(x for x in rad if x > 1))
    return out


# ------------------------------------------------------------------ twiddle error, emulated
# mu in the bound is the error of the twiddle factors the butterflies actually use.  It is
# measured here by running the kernels' twiddle arithmetic in binary32 on the CPU: the table
# exp(-2 pi i t/N) rounded once, then twiddle_powers (fft_kernels.cuh) -- powers w1^r by a product
# tree, or for radix >= 64 as (w1^8)^a * w1^b -- with cmul's two packed operations (a.y*b rounded,
# then one FMA per half), and the four-step's 16-step recurrence w <- w * step (fft_fourstep.cuh).
# Each power inherits r times the table's rounding, so the tree's depth alone does not bound it:
# radix-32 passes reach about 23u and the radix-64 passes of N = 4096 about 48u.
def _fma32(a, b, c):
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def _cmul32(a, b):
    py = (a[1] * b[1]).astype(np.float32)
    px = (a[1] * b[0]).astype(np.float32)
    return _fma32(a[0], b[0], -py), _fma32(a[0], b[1], px)


def _table32(m):
    ang = 2.0 * np.pi * np.arange(m) / m
    return np.cos(ang).astype(np.float32), (-np.sin(ang)).astype(np.float32)


def _powers32(R, w1):
    w = {1: w1}
    if R >= 64 and R % 8 == 0:
        wb = {1: w1}
        for b in range(2, 8):
            wb[b] = _cmul32(wb[b // 2], wb[b - b // 2])
        wa = {1: _cmul32(wb[4], wb[4])}
        for q in range(2, R // 8):
            wa[q] = _cmul32(wa[q // 2], wa[q - q // 2])
        for r in range(2, R):
            x = wb[r % 8] if r % 8 else None
            if r // 8:
                x = wa[r // 8] if x is None else _cmul32(x, wa[r // 8])
            w[r] = x
        return w
    for r in range(2, R):
        w[r] = _cmul32(w[r // 2], w[r - r // 2])
    return w


def _err(w, exact):
    return float(np.max(np.abs(w[0].astype(np.float64) + 1j * w[1].astype(np.float64) - exact)))


def _pass_mu(n, tw, R, M):
    """Twiddles of a pass of radix R after passes whose radices multiply to M (L = M*R)."""
    L = M * R
    j = np.arange(M)
    w = _powers32(R, (tw[0][j * (n // L)], tw[1][j * (n // L)]))
    return max(_err(w[r], np.exp(-2j * np.pi * ((j * r) % L) / L)) for r in w)


@functools.lru_cache(maxsize=None)
def emulated_mu(n: int) -> float:
    """Largest twiddle error of the plan that runs length n (0 where none is emulated: the staged
    path rounds the angle in turns once and calls sincospif, a few u)."""
    if n == 65536:                                       # four-step 256 x 256: radix-16 powers + recurrence
        tw = _table32(n)
        mu = _pass_mu(n, tw, 16, 16)
        n2, j = np.arange(256)[:, None], np.arange(16)[None, :]
        w = (tw[0][(n2 * j) % n], tw[1][(n2 * j) % n])
        step = tuple(np.broadcast_to(t[16 * n2], w[0].shape) for t in tw)
        for q in range(16):
            mu = max(mu, _err(w, np.exp(-2j * np.pi * ((n2 * (j + 16 * q)) % n) / n)))
            w = _cmul32(w, step)
        return mu
    m = n // 2 if n in SPLIT else n                      # a split plan runs the n/2-point plan per CTA
    if m not in plans():
        return 0.0
    rad = plans()[m][2]
    tw = _table32(m)
    mu, M = 0.0, rad[0]
    for R in rad[1:]:                                    # pass 0 has no twiddles
        mu = max(mu, _pass_mu(m, tw, R, M))
        M *= R
    return mu


def plan_mu(n: int) -> float:
    """mu for length n: the emulated twiddle error plus 2u (the FMA emulation rounds twice), never
    below 16u.  The floor is chosen, not derived.  It is what the staged path gets (its twiddles,
    sincospif of an angle rounded once in turns, are within a few u) and it leaves room for the
    split plan's radix-2 rotation on the way in (one table value and one constant, not emulated)."""
    return max(MU, emulated_mu(n) + 2 * U)


def bound(n: int, mu: float = None) -> float:
    """Higham, Accuracy and Stability of Numerical Algorithms (2nd ed.), Thm 24.2: a radix-2
    FFT computed with twiddles of error <= mu satisfies ||X^-X|| / ||X|| <= L*eta / (1 - L*eta),
    L = log2 N, eta = mu + gamma_4 * (sqrt2 + mu), gamma_4 = 4u / (1 - 4u).  mu defaults to
    plan_mu(n).  The theorem covers radix 2 only; that the mixed-radix and odd-radix stages here
    (radix 4, 8, ..., 64 in registers, 3, 5, 7, 15, 21 as direct sums) stay below it with
    L = ceil(log2 N) is an assumption, not a derivation.  The measured errors of every plan sit
    far below B(N), which is consistent with it but does not prove it."""
    if mu is None:
        mu = plan_mu(n)
    L = max(1, math.ceil(math.log2(n)))
    g4 = 4 * U / (1 - 4 * U)
    eta = mu + g4 * (math.sqrt(2.0) + mu)
    return L * eta / (1 - L * eta)


# ------------------------------------------------------------------ exact inputs
def wrap16(v):
    """Two's-complement 16-bit wrap of integers (numpy int64 arithmetic)."""
    v = np.asarray(v, dtype=np.int64)
    return ((v + 0x8000) & 0xFFFF) - 0x8000


def s16_ints(raw, n: int, ic: int = 0, qc: int = 0):
    """JavaAudio.java:281-288: s += (short)ic with 16-bit wrap, for int16 IQ [..., 2n].
    Returns (I, Q) as int64 [batch, n]; ic / qc are C ints and may lie outside 16 bits."""
    r = np.asarray(raw, dtype=np.int64).reshape(-1, n, 2)
    return wrap16(r[..., 0] + wrap16(ic)), wrap16(r[..., 1] + wrap16(qc))


def s16_input(raw, n: int, ic: int = 0, qc: int = 0) -> np.ndarray:
    """The s16 kernels' input as complex128 [batch, n]: wrapped ints divided by 32767 in binary64
    (the kernels fold the 1/32767 into the PSD scale, so this is what they transform)."""
    i, q = s16_ints(raw, n, ic, qc)
    return (i + 1j * q) / 32767.0


def f32_input(x, n: int) -> np.ndarray:
    """Interleaved float32 IQ [..., 2n] as complex128 [batch, n], exactly."""
    return np.asarray(x, dtype=np.float32).reshape(-1, n, 2).astype(np.float64).view(np.complex128)[..., 0]


def reference(z: np.ndarray) -> np.ndarray:
    """The unnormalised forward DFT (JTransforms complexForward) in binary64."""
    return np.fft.fft(np.asarray(z, dtype=np.complex128), axis=-1)


# ------------------------------------------------------------------ PSD -> amplitude
def kernel_db_off(n: int, s16: bool) -> np.float32:
    """fft.cu's db_off, computed the way fft.cu computes it: cf = (2f/N)^2 in float, / 32767^2
    in double for s16 input, then 10*log10 in double rounded to float."""
    cf = np.float32(2.0) / np.float32(n)
    cf = np.float32(cf * cf)
    if s16:
        cf = np.float32(np.float64(cf) / (32767.0 * 32767.0))
    return np.float32(10.0 * math.log10(float(cf)))


def amplitude(psd: np.ndarray, n: int) -> np.ndarray:
    """|X| (of the float input, i.e. after the 1/32767 for s16) from published dB: the PSD is
    10*log10(|X|^2 (2/N)^2), so |X| = 10^(dB/20) * N/2.  -inf dB reads as 0."""
    return np.power(10.0, np.asarray(psd, dtype=np.float64)[..., :n] / 20.0) * (n / 2.0)


# The kernels publish dB = fma(c, lg2.approx(pw), db_off): pw = re^2 + im^2 of the kernel's own
# values (integers for s16 input), c = 10*log10(2) rounded to float.  Against 10*log10(|X|^2 cf)
# in exact arithmetic the published value differs by at most
#   e_off                       db_off's offset from 10*log10 of the exact cf: cf rounded in float
#                               (and, for s16, rounded again after / 32767^2), the log rounded to
#                               float -- computed here exactly as fft.cu does it;
#   ulp(dB)                     the FMA's final rounding (half an ulp; a whole one is taken so a
#                               published value at a binade edge is covered);
#   c_lg2 * (2^-21 + ulp(lg2))  MUFU.LG2: the PTX ISA gives lg2.approx.f32 a maximum absolute error
#                               of 2^-22 (taken twice) in the logarithm of the mantissa, plus the
#                               rounding of a result as large as |lg2 pw| (62 for s16 at N = 65536);
#   |c - 10 log10 2| * |lg2|    the rounded constant, scaled by the logarithm it multiplies;
#   (10/ln10) * 2.5u            pw = fma(x, x, y*y): two roundings, relative 2u in power.
# A dB error e scales the recovered amplitude by 10^(+-e/20), so a bin's relative amplitude error
# from the formatting is r = 10^(e/20) - 1 (about 0.115 e).  The transform's own error then adds
# to it: | |X^|(1+rho) - |X| | <= | |X^| - |X| | + r |X^|, so the normwise PSD bound is
# B + ||r |X| ||_2 / ||X||_2 * (1 + B).  Bins below 2^-126 in power flush to zero (-inf dB), which
# adds at most sqrt(N) * 2^-63 in the kernel's units; that is included too.
C_LG2 = float(np.float32(3.0102999566398120))
C_ERR = abs(C_LG2 - 10.0 * math.log10(2.0))


def psd_roundoff(absx: np.ndarray, n: int, s16: bool) -> np.ndarray:
    """Per-bin bound r on the relative amplitude error that the dB formatting adds (see above).
    absx: binary64 |X| [batch, n] of the float input."""
    absx = np.asarray(absx, dtype=np.float64)
    scale = 32767.0 if s16 else 1.0
    db_off = kernel_db_off(n, s16)
    cf_exact = (2.0 / n) ** 2 / (scale * scale)
    e_off = abs(float(db_off) - 10.0 * math.log10(cf_exact)) + 1e-12
    with np.errstate(divide="ignore"):
        pw = (absx * scale) ** 2
        lg2 = np.where(pw > 0, np.log2(np.where(pw > 0, pw, 1.0)), 0.0)
        db = lg2 * (10.0 * math.log10(2.0)) + float(db_off)
    ulp_db = np.spacing(np.abs(db).astype(np.float32)).astype(np.float64)
    ulp_lg2 = np.spacing(np.abs(lg2).astype(np.float32)).astype(np.float64)
    e_db = e_off + ulp_db + C_LG2 * (2.0 ** -21 + ulp_lg2) + C_ERR * np.abs(lg2) + (10.0 / math.log(10.0)) * 2.5 * U
    return np.power(10.0, e_db / 20.0) - 1.0


# ------------------------------------------------------------------ normwise checks
def _norms(X):
    return np.sqrt(np.sum(np.abs(X) ** 2, axis=-1))


def spectrum_errors(Xhat: np.ndarray, X: np.ndarray) -> np.ndarray:
    """||X^ - X||_2 / ||X||_2 per block (0 where both are zero)."""
    Xhat = np.asarray(Xhat).reshape(X.shape).astype(np.complex128)
    num = _norms(Xhat - X)
    den = _norms(X)
    return np.where(den > 0, num / np.where(den > 0, den, 1.0), np.where(num > 0, np.inf, 0.0))


class PsdRef:
    """A binary64 spectrum prepared for PSD checks: |X|, ||X|| and the formatting part of the
    bound per block.  Slicing selects blocks, so a prefix of a batch costs nothing to prepare."""

    def __init__(self, X, s16: bool, mu: float = None, _parts=None):
        self.X, self.s16, self.mu = X, s16, mu
        if _parts is None:
            n = X.shape[-1]
            absx = np.abs(X)
            den = _norms(X)
            safe = np.where(den > 0, den, 1.0)
            B = bound(n, mu)
            fmt = _norms(psd_roundoff(absx, n, s16) * absx) / safe * (1.0 + B)
            ftz = math.sqrt(n) * 2.0 ** -63 / (32767.0 if s16 else 1.0) / safe
            _parts = (absx, den, B + fmt + ftz)
        self.absx, self.den, self.bnd = _parts

    def __getitem__(self, sl):
        return PsdRef(self.X[sl], self.s16, self.mu, tuple(p[sl] for p in (self.absx, self.den, self.bnd)))


def psd_errors(psd: np.ndarray, X, s16: bool, mu: float = None):
    """(|| |X^| - |X| ||_2 / ||X||_2, its bound) per block for published PSD rows [batch, n+2].
    X: the binary64 spectrum, or a PsdRef of it."""
    ref = X if isinstance(X, PsdRef) else PsdRef(X, s16, mu)
    n = ref.X.shape[-1]
    amp = amplitude(np.asarray(psd).reshape(ref.X.shape[0], n + 2), n)
    num = _norms(amp - ref.absx)
    err = np.where(ref.den > 0, num / np.where(ref.den > 0, ref.den, 1.0), np.where(num > 0, np.inf, 0.0))
    return err, ref.bnd


def _first_bad(ok):
    bad = np.flatnonzero(~np.asarray(ok))
    return int(bad[0]) if bad.size else None


def check_spectrum(Xhat: np.ndarray, X: np.ndarray, mu: float = None, what: str = "") -> np.ndarray:
    """Every block of a spectrum output within B(N); returns the per-block errors."""
    err = spectrum_errors(Xhat, X)
    B = bound(X.shape[-1], mu)
    b = _first_bad(err <= B)
    assert b is None, f"{what}: block {b} normwise error {err[b]:.3e} > B(N) = {B:.3e} ({int(np.sum(err > B))} blocks)"
    return err


def check_psd(psd: np.ndarray, X: np.ndarray, s16: bool, mu: float = None, what: str = "") -> np.ndarray:
    """Every block of a PSD output within its bound (B(N) plus the formatting); returns the
    per-block errors.  X: the binary64 spectrum or a PsdRef of it."""
    err, bnd = psd_errors(psd, X, s16, mu)
    b = _first_bad(err <= bnd)
    assert b is None, f"{what}: block {b} normwise amplitude error {err[b]:.3e} > bound {bnd[b]:.3e} ({int(np.sum(err > bnd))} blocks)"
    return err


# ------------------------------------------------------------------ peak (fft.java:208-224)
def peak_hz(bins, n: int, rate: int) -> np.ndarray:
    """fft.java:214-221 on bin k: p = 2k, p -= dat.length if p >= dat.length/2, then p*rate in
    wrapping int32 arithmetic, divided by dat.length = 2N with truncation.  bin -1 (no maximum)
    gives p = -1 as the Java loop leaves it."""
    k = np.asarray(bins, dtype=np.int64)
    p = np.where(k < 0, -1, 2 * k)
    p = np.where(p >= n, p - 2 * n, p)
    prod = ((p * rate + 2 ** 31) % 2 ** 32) - 2 ** 31
    q = np.abs(prod) // (2 * n)
    return np.where(prod < 0, -q, q)


def check_peak(psd: np.ndarray, pk: np.ndarray, X: np.ndarray, rate: int, what: str = "", sep: float = 1e-3):
    """The published maximum of every row is its own (psd[N+1] is the row maximum, the bin is the
    first index holding it, psd[N] its frequency), and wherever the binary64 top two magnitudes
    differ by more than `sep` relative, the bin is the binary64 argmax."""
    a = X.absx if isinstance(X, PsdRef) else np.abs(X)
    n = a.shape[-1]
    psd = np.asarray(psd).reshape(a.shape[0], n + 2)
    pk = np.asarray(pk).ravel()
    body = psd[:, :n]
    m = body.max(axis=1)
    none = ~(m > -FLT_MAX)                          # all -inf: nothing beats -Float.MAX_VALUE
    first = np.where(none, -1, np.argmax(body == m[:, None], axis=1))
    b = _first_bad(pk == first)
    assert b is None, f"{what}: block {b} publishes bin {pk[b]}, its row's first maximum is bin {first[b]}"
    b = _first_bad(psd[:, n + 1] == np.where(none, np.float32(-FLT_MAX), m))
    assert b is None, f"{what}: block {b} publishes maximum {psd[b, n + 1]}, its row's maximum is {m[b]}"
    b = _first_bad(psd[:, n] == peak_hz(first, n, rate).astype(np.float32))
    assert b is None, f"{what}: block {b} publishes {psd[b, n]} Hz for bin {first[b]}"
    if n >= 2:
        top = np.partition(a, n - 2, axis=1)[:, n - 2:]
        clear = top[:, 1] > top[:, 0] * (1.0 + sep)
        ref = np.argmax(a, axis=1)
        b = _first_bad(~clear | (pk == ref))
        assert b is None, f"{what}: block {b} publishes bin {pk[b]}, the binary64 maximum is bin {ref[b]}"


# ------------------------------------------------------------------ dynamic range
def two_tones_f32(n: int, k0: int, kw: int, weak_db: float = -100.0) -> np.ndarray:
    """Full-scale on-bin complex tone at k0 plus one weak_db below it at kw, float32 IQ [2n]."""
    a = 10.0 ** (weak_db / 20.0)
    t = np.arange(n)
    z = (1.0 - a) * np.exp(2j * np.pi * ((k0 * t) % n) / n) + a * np.exp(2j * np.pi * ((kw * t) % n) / n)
    return z.astype(np.complex64).view(np.float32)


def two_tones_s16(n: int, k0: int, kw: int, weak_db: float = -80.0) -> np.ndarray:
    """The same in s16 IQ [2n]; the weak tone is -80 dBFS so that it survives quantisation."""
    a = 32767.0 * 10.0 ** (weak_db / 20.0)
    t = np.arange(n)
    z = (32767.0 - 1.0 - a) * np.exp(2j * np.pi * ((k0 * t) % n) / n) + a * np.exp(2j * np.pi * ((kw * t) % n) / n)
    out = np.empty(2 * n, np.int16)
    out[0::2] = np.rint(z.real)
    out[1::2] = np.rint(z.imag)
    return out


def check_dynamic_range(absx_hat: np.ndarray, X: np.ndarray, amp: float, kw, s16: bool, psd: bool,
                        what: str = "", db_tol: float = 0.05) -> np.ndarray:
    """Every bin within 1e-6 * N * amp of binary64 (120 dB below the carrier; a PSD output is
    allowed its formatting error r|X| on top), and the weak tone at bin kw within db_tol dB.
    Returns the worst per-bin error in dB relative to the carrier (dBc), per block."""
    n = X.shape[-1]
    absx = np.abs(X)
    tol = 1e-6 * n * amp
    if psd:
        tol = tol + psd_roundoff(absx, n, s16) * absx
    d = np.abs(absx_hat - absx)
    bad = d > tol
    b = _first_bad(~bad.any(axis=1))
    if b is not None:
        k = int(np.argmax(d[b] - tol[b] if np.ndim(tol) else d[b]))
        raise AssertionError(f"{what}: block {b} bin {k} off by {d[b, k]:.3e} (|X| {absx[b, k]:.3e}); limit 1e-6*N*A = {1e-6 * n * amp:.3e}")
    kw = np.broadcast_to(np.asarray(kw), (X.shape[0],))
    rows = np.arange(X.shape[0])
    with np.errstate(divide="ignore"):
        got = 20.0 * np.log10(absx_hat[rows, kw])
        want = 20.0 * np.log10(absx[rows, kw])
        dbc = 20.0 * np.log10(np.max(d, axis=1) / (n * amp))
    b = _first_bad(np.abs(got - want) <= db_tol)
    assert b is None, f"{what}: block {b} weak tone at bin {kw[b]}: {got[b]:.4f} dB against {want[b]:.4f} dB"
    return dbc
