"""The input a windowed FFT handle transforms (jsdr_fft_set_window), rebuilt exactly in numpy.

The kernels multiply each converted sample by win[t] once in binary32, before any butterfly:
RN(x * w[t]) for float input, RN((float)s * w[t]) for s16 input with s the wrapped value after
ic / qc (the 1/32767 stays in the PSD scale).  numpy's float32 multiply rounds the same way, so
the binary64 DFT of these arrays is the X of tests/fft_accuracy.py for a windowed handle, and the
bound B(N) applies unchanged."""
import numpy as np

import fft_accuracy as A


def hamming(n: int) -> np.ndarray:
    """fft.java's win[] (:72-73): 0.54 - 0.46 cos(2 pi t / n), float32[n]."""
    t = np.arange(n)
    return (0.54 - 0.46 * np.cos(2.0 * np.pi * t / n)).astype(np.float32)


def random_window(n: int, seed: int) -> np.ndarray:
    """Entries in [0.25, 1): no symmetry, so a window read at a shifted or mirrored index, or a
    block's second half read with the first half's entries, moves the spectrum far beyond B(N)."""
    return np.random.default_rng(seed).uniform(0.25, 1.0, n).astype(np.float32)


def s16_products(raw, n: int, win, ic: int = 0, qc: int = 0, i_only: bool = False):
    """RN((float)s * w[t]) for I and Q as float32 [batch, n] each (i_only: Q left unwindowed)."""
    i, q = A.s16_ints(raw, n, ic, qc)
    w = np.asarray(win, dtype=np.float32)
    wi = i.astype(np.float32) * w
    wq = q.astype(np.float32) if i_only else q.astype(np.float32) * w
    return wi, wq


def s16_input(raw, n: int, win, ic: int = 0, qc: int = 0, i_only: bool = False) -> np.ndarray:
    """A windowed s16 handle's input as complex128 [batch, n]: the products divided by 32767 in
    binary64, as A.s16_input does for an unwindowed one."""
    wi, wq = s16_products(raw, n, win, ic, qc, i_only)
    return (wi.astype(np.float64) + 1j * wq.astype(np.float64)) / 32767.0


def f32_pairs(x, n: int, win, i_only: bool = False) -> np.ndarray:
    """RN(x * w[t]) on interleaved float32 IQ: float32 [batch, 2n] (i_only: Q left unwindowed)."""
    z = np.asarray(x, dtype=np.float32).reshape(-1, n, 2).copy()
    w = np.asarray(win, dtype=np.float32)
    z[..., 0] *= w
    if not i_only:
        z[..., 1] *= w
    return z.reshape(-1, 2 * n)


def f32_input(x, n: int, win, i_only: bool = False) -> np.ndarray:
    """A windowed float handle's input as complex128 [batch, n], exactly."""
    return A.f32_input(f32_pairs(x, n, win, i_only), n)
