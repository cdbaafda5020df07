"""The binary32 decimator (JSDR_PREC_F32, k_mixdecim_stream's PREC_F32 body) against the binary64
reference: a bound on every output, derived from the kernel's arithmetic, tight enough to see one wrong
table index at almost every tap.

What period_body<.., PREC_F32, ..> does per input sample x (the reference's float, or an s16 value s
with x = s/32767) and table entry (c, s) of index i:
  - table   t = (float)(cos / 32767.0) for s16 input (the conversion's 1/32767 folded in), (float)cos
            for float input: one binary32 rounding (the binary64 division before it adds 2^-53);
  - product m = x*t (s16: s*t) in binary32: one rounding;  history samples instead take the binary64
            mixed sample rounded to float: one rounding;
  - taps    h' = (float)h: one rounding (none for the default taps, which are float literals);
  - FIR     acc = fmaf(m, h'_k, acc) over the NTAPS taps: NTAPS roundings, each at most u times the
            running sum, which is at most sum_k |m_k h'_k| (to first order);
  - output  (double)acc * 0.9*32768 in binary64.
The reference (FUNcubeBPSKDemod.java:389-390, 479-486) converts s16 as (float)s/32767f (one binary32
rounding of x) and mixes, multiplies and sums in binary64.  So, with u = 2^-24 and S = sum_k |h_k| |x_{n-k}|
per component (|cos|, |sin| <= 1),

  |y_kernel - y_ref| <= c * u * S * 0.9*32768,   c = NTAPS + 3 (table, product, taps) + 1 (s16: the
                                                  reference's conversion) + 1,

where the last unit covers every binary64 rounding of both sides (at most NTAPS + 3 of 2^-53 relative to
S) and the second-order terms ((c u)^2 < 2^-36).  A wrong index moves a mixed sample by
|x| * 2 sin(pi/256) ~ 0.0245 |x| in (cos, sin), so by at least 0.0173 |x| in one of the two components:
for |x| >= 1/2 that is outside the bound wherever |h_k| exceeds about 3e-4 (the default filter: 25 of its
27 taps).  The former bar, 1e-4 of full scale, was blind to a wrong index wherever |h_k| |x| < 4e-3.
"""
import numpy as np

U = 2.0 ** -24
FULL_SCALE = 0.9 * 32768.0


def units(ntaps, s16):
    """c of the bound (see the module's docstring)."""
    return ntaps + 3 + (1 if s16 else 0) + 1


class Bound:
    """The bound of every output of one channel, block by block: feed each block's input as the reference
    sees it (float IQ pairs, after the s16 conversion and I/Q correction); the history of the last taps
    and the decimation phase carry across blocks, as in the bank."""

    def __init__(self, taps, D, s16):
        self.h = np.abs(np.asarray(taps, np.float64))
        self.D = D
        self.s16 = s16
        self.tail = np.zeros((self.h.size - 1, 2))
        self.cnt = 0

    def block(self, x, s16=None):
        """The bound of every output of the block x (s16: whether the kernel read it as s16 input)."""
        c = units(self.h.size, self.s16 if s16 is None else s16)
        a = np.abs(np.asarray(x, np.float64).reshape(-1, 2))
        n = a.shape[0]
        if n == 0:
            return np.zeros((0, 2))
        full = np.vstack([self.tail, a])
        S = np.stack([np.convolve(full[:, i], self.h, mode="valid") for i in (0, 1)], axis=1)   # [n, 2]
        j = np.arange(n)
        out = S[(self.cnt + j + 1) % self.D == 0]
        self.cnt = (self.cnt + n) % self.D
        if self.h.size > 1:
            self.tail = full[-(self.h.size - 1):]
        return c * U * FULL_SCALE * out


def kernel_f32(x, idx, taps, D, s16):
    """A numpy binary32 emulation of the PREC_F32 body on one channel from a zero history: x the input
    (s16 values if s16, else floats) as [n, 2], idx the table index of every sample (256: bypass).  fmaf
    is taken as the binary64 sum of the exact product, rounded to binary32 (a double rounding the kernel
    does not have: at most 2^-53 more per tap, inside the bound's last unit)."""
    cs = np.array([[np.cos(n * 2.0 * np.pi / 256), np.sin(n * 2.0 * np.pi / 256)] for n in range(256)] + [[1.0, 1.0]])
    tab = (cs / (32767.0 if s16 else 1.0)).astype(np.float32)
    xf = np.asarray(x).astype(np.float32)
    m = (xf * tab[idx]).astype(np.float32)                     # binary32 product
    hf = np.asarray(taps, np.float64).astype(np.float32)
    n = xf.shape[0]
    outs = np.arange(D - 1, n, D)
    acc = np.zeros((outs.size, 2), np.float32)
    for k in range(hf.size):
        s = outs - k
        mk = np.where((s >= 0)[:, None], m[np.maximum(s, 0)], np.float32(0))
        acc = (mk.astype(np.float64) * np.float64(hf[k]) + acc.astype(np.float64)).astype(np.float32)
    return acc.astype(np.float64) * FULL_SCALE


def reference(xref, idx, taps, D):
    """The reference's decimator outputs (binary64, its order) from the floats it sees and the indices."""
    cs = np.array([[np.cos(n * 2.0 * np.pi / 256), np.sin(n * 2.0 * np.pi / 256)] for n in range(256)] + [[1.0, 1.0]])
    m = np.asarray(xref, np.float64) * cs[idx]
    h = np.asarray(taps, np.float64)
    n = m.shape[0]
    outs = np.arange(D - 1, n, D)
    acc = np.zeros((outs.size, 2))
    for k in range(h.size):
        s = outs - k
        acc = acc + np.where((s >= 0)[:, None], m[np.maximum(s, 0)], 0.0) * h[k]
    return acc * FULL_SCALE
