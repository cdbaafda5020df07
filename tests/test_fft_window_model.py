"""The windowed FFT's checker on the CPU (tests/fft_window.py with tests/fft_accuracy.py): at every
length the GPU tests run, a binary32 FFT (scipy, complex64) of exactly the windowed input passes
B(N), and each mistake a windowed kernel could make is rejected -- the window read one sample
late, the window applied to I only, and no window at all."""
import numpy as np
import pytest

import fft_accuracy as A
import fft_window as W
from test_fft_accuracy_model import fp32_fft, fp32_psd

RATE = 192000
BATCH = 3


def noise_s16(n, seed):
    return np.random.default_rng(seed).integers(-32768, 32768, (BATCH, 2 * n)).astype(np.int16)


def s16_psd(raw, n, win, ic=0, qc=0, i_only=False):
    """What a binary32 FFT of the windowed s16 input publishes (the 1/32767 applied in float32)."""
    wi, wq = W.s16_products(raw, n, win, ic, qc, i_only)
    z = (wi / np.float32(32767.0)) + 1j * (wq / np.float32(32767.0))
    return fp32_psd(fp32_fft(z.astype(np.complex64)), n)


def f32_spectrum(x, n, win, i_only=False):
    return fp32_fft(W.f32_pairs(x, n, win, i_only).view(np.complex64))


def test_products_are_one_binary32_rounding():
    """The emulated products equal the binary64 product rounded once to float32, for every s16
    value against a few windows (both factors are exact in binary64, the product too)."""
    s = np.arange(-32768, 32768, dtype=np.int64)
    raw = np.stack([s, s[::-1]], axis=1).astype(np.int16).ravel()
    n = s.size
    for win in (W.hamming(n), W.random_window(n, 1), np.ones(n, np.float32)):
        wi, wq = W.s16_products(raw, n, win)
        assert np.array_equal(wi[0], (s.astype(np.float64) * win.astype(np.float64)).astype(np.float32))
        assert np.array_equal(wq[0], (s[::-1].astype(np.float64) * win.astype(np.float64)).astype(np.float32))
    assert np.array_equal(W.s16_input(raw, n, np.ones(n, np.float32)), A.s16_input(raw, n))


@pytest.mark.parametrize("n", A.LENGTHS)
def test_checker_accepts_windowed_fp32_fft(n):
    for win in (W.random_window(n, n), W.hamming(n)):
        raw = noise_s16(n, n)
        for ic, qc in ((0, 0), (70000, -32768)):
            X = A.reference(W.s16_input(raw, n, win, ic, qc))
            psd, pk = s16_psd(raw, n, win, ic, qc)
            A.check_psd(psd, X, s16=True, what="scipy fp32 windowed PSD, s16")
            A.check_peak(psd, pk, X, RATE, what="scipy fp32 windowed PSD, s16")
        x = (raw.astype(np.float32) / np.float32(32767.0)).astype(np.float32)
        Xf = A.reference(W.f32_input(x, n, win))
        S = f32_spectrum(x, n, win)
        A.check_spectrum(S, Xf, what="scipy fp32 windowed spectrum")
        psd, pk = fp32_psd(S, n)
        A.check_psd(psd, Xf, s16=False, what="scipy fp32 windowed PSD, f32")
        A.check_peak(psd, pk, Xf, RATE, what="scipy fp32 windowed PSD, f32")


@pytest.mark.parametrize("n", A.LENGTHS)
def test_checker_rejects_window_shifted_by_one(n):
    win = W.random_window(n, n + 1)
    late = np.roll(win, 1)                                       # sample t times win[t - 1]
    raw = noise_s16(n, n + 1)
    X = A.reference(W.s16_input(raw, n, win))
    with pytest.raises(AssertionError):
        A.check_psd(s16_psd(raw, n, late)[0], X, s16=True)
    x = (raw.astype(np.float32) / np.float32(32767.0)).astype(np.float32)
    with pytest.raises(AssertionError):
        A.check_spectrum(f32_spectrum(x, n, late), A.reference(W.f32_input(x, n, win)))


@pytest.mark.parametrize("n", A.LENGTHS)
def test_checker_rejects_window_on_i_only(n):
    win = W.random_window(n, n + 2)
    raw = noise_s16(n, n + 2)
    X = A.reference(W.s16_input(raw, n, win))
    with pytest.raises(AssertionError):
        A.check_psd(s16_psd(raw, n, win, i_only=True)[0], X, s16=True)
    x = (raw.astype(np.float32) / np.float32(32767.0)).astype(np.float32)
    with pytest.raises(AssertionError):
        A.check_spectrum(f32_spectrum(x, n, win, i_only=True), A.reference(W.f32_input(x, n, win)))


@pytest.mark.parametrize("n", A.LENGTHS)
def test_checker_rejects_unwindowed_transform(n):
    win = W.random_window(n, n + 3)
    raw = noise_s16(n, n + 3)
    X = A.reference(W.s16_input(raw, n, win))
    ones = np.ones(n, np.float32)
    with pytest.raises(AssertionError):
        A.check_psd(s16_psd(raw, n, ones)[0], X, s16=True)
    x = (raw.astype(np.float32) / np.float32(32767.0)).astype(np.float32)
    with pytest.raises(AssertionError):
        A.check_spectrum(f32_spectrum(x, n, ones), A.reference(W.f32_input(x, n, win)))
