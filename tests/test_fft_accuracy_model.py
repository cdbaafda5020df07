"""The FFT accuracy checker (tests/fft_accuracy.py) on the CPU: it accepts an honest binary32
FFT (scipy, complex64) at every length the GPU tests run, and rejects each fault that the 1e-4
parity bar lets through at large N -- one sample read from the neighbouring block, an ic
correction added without its 16-bit wrap, a spectrum at bf16 precision -- and a wrong peak bin."""
import numpy as np
import pytest
import scipy.fft

import fft_accuracy as A
import oracle as O

RATE = 192000
BATCH = 3


def noise_s16(n, seed, batch=BATCH):
    return np.random.default_rng(seed).integers(-32768, 32768, (batch, 2 * n)).astype(np.int16)


def fp32_fft(z):
    return scipy.fft.fft(np.asarray(z, dtype=np.complex64), axis=-1)


def fp32_psd(Xf, n, rate=RATE):
    """fft.java:199-224 on a binary32 spectrum in float32 arithmetic (np.log10 for the logarithm)."""
    Xf = np.asarray(Xf, dtype=np.complex64)
    cf = np.float32(2.0) / np.float32(n)
    cf = np.float32(cf * cf)
    re, im = Xf.real, Xf.imag
    with np.errstate(divide="ignore"):
        db = np.float32(10.0) * np.log10((re * re + im * im) * cf)
    m = db.max(axis=1)
    pk = np.argmax(db == m[:, None], axis=1)
    psd = np.empty((Xf.shape[0], n + 2), np.float32)
    psd[:, :n] = db
    psd[:, n] = A.peak_hz(pk, n, rate)
    psd[:, n + 1] = m
    return psd, pk


def s16_floats(raw, n, ic=0, qc=0):
    """JavaAudio's conversion to float32 (what an fp32 FFT of the s16 path would transform)."""
    return O.s16_to_float(raw, ic, qc).view(np.complex64).reshape(-1, n)


def bf16(Xf):
    """Round real and imaginary parts to bf16 (8 significant bits), nearest even."""
    u = np.ascontiguousarray(Xf, dtype=np.complex64).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.complex64).reshape(np.shape(Xf))


def test_s16_reference_wrap_matches_oracle():
    """The binary64 reference's ic/qc wrap is JavaAudio's (oracle.s16_to_float), including
    corrections outside 16 bits: the C ABI takes an int."""
    s = np.arange(-32768, 32768, dtype=np.int64)
    raw = np.stack([s, s[::-1]], axis=1).astype(np.int16).ravel()
    n = s.size
    for ic, qc in ((0, 0), (9, -9), (-9, 9), (70000, -32768), (-70000, 32768), (32767, -32767), (65536, 131071)):
        ref = A.s16_input(raw, n, ic, qc)[0]
        got = O.s16_to_float(raw, ic, qc).astype(np.float64).view(np.complex128)
        assert np.array_equal(ref.astype(np.complex64), got.astype(np.complex64)), (ic, qc)


def test_bound_is_tight_enough_to_see_one_sample():
    """B(N) from about 1e-5 (N = 128) to about 2e-5 (N = 65536) and 4e-5 at 4096 (radix-64 twiddle
    powers, mu about 50u), always under 1e-4: one wrong full-range sample (normwise about
    |d| / (sqrt(N) rms)) stays far above it.  mu is never below the emulated twiddle error."""
    assert 0.8e-5 < A.bound(128) < 1.1e-5 and 1.9e-5 < A.bound(65536) < 2.2e-5
    for n in A.LENGTHS:
        assert A.bound(n) < 1e-4
        assert 1.0 / (np.sqrt(n) * np.sqrt(2.0 / 3.0)) > 100 * A.bound(n)
        assert A.plan_mu(n) >= max(A.MU, A.emulated_mu(n))
    assert 45 * A.U < A.emulated_mu(4096) < 50 * A.U and 20 * A.U < A.emulated_mu(16384) < 24 * A.U


@pytest.mark.parametrize("n", A.LENGTHS)
def test_checker_accepts_fp32_fft(n):
    raw = noise_s16(n, n)
    X = A.reference(A.s16_input(raw, n))
    psd, pk = fp32_psd(fp32_fft(s16_floats(raw, n)), n)
    A.check_psd(psd, X, s16=True, what="scipy fp32 PSD, s16")
    A.check_peak(psd, pk, X, RATE, what="scipy fp32 PSD, s16")
    x = O.s16_to_float(raw).reshape(BATCH, 2 * n)                # float input, complex spectrum
    Xf = A.reference(A.f32_input(x, n))
    Xhat = fp32_fft(x.view(np.complex64))
    A.check_spectrum(Xhat, Xf, what="scipy fp32 spectrum")
    psd, pk = fp32_psd(Xhat, n)
    A.check_psd(psd, Xf, s16=False, what="scipy fp32 PSD, f32")
    A.check_peak(psd, pk, Xf, RATE, what="scipy fp32 PSD, f32")
    k0, kw = n // 3, (n // 3 + max(1, n // 3)) % n             # dynamic range, both formats
    t = A.two_tones_f32(n, k0, kw).reshape(1, 2 * n)
    Xt = A.reference(A.f32_input(t, n))
    Xht = fp32_fft(t.view(np.complex64))
    A.check_dynamic_range(np.abs(Xht), Xt, 1.0, kw, s16=False, psd=False)
    psd, _ = fp32_psd(Xht, n)
    A.check_dynamic_range(A.amplitude(psd, n), Xt, 1.0, kw, s16=False, psd=True)
    r = A.two_tones_s16(n, k0, kw).reshape(1, 2 * n)
    Xr = A.reference(A.s16_input(r, n))
    psd, pk = fp32_psd(fp32_fft(s16_floats(r, n)), n)
    A.check_dynamic_range(A.amplitude(psd, n), Xr, 32766.0 / 32767.0, kw, s16=True, psd=True)
    A.check_peak(psd, pk, Xr, RATE)


@pytest.mark.parametrize("n", A.LENGTHS)
def test_checker_rejects_sample_from_neighbouring_block(n):
    raw = noise_s16(n, n + 1)
    X = A.reference(A.s16_input(raw, n))
    bad = raw.copy()
    bad[:-1, 0:2] = raw[1:, 0:2]                                 # sample 0 of block b+1 in block b
    psd, _ = fp32_psd(fp32_fft(s16_floats(bad, n)), n)
    with pytest.raises(AssertionError):
        A.check_psd(psd, X, s16=True)


@pytest.mark.parametrize("n", A.LENGTHS)
def test_checker_rejects_ic_without_wrap(n):
    ic, qc = 9, -9
    raw = noise_s16(n, n + 2)
    raw[:, 2 * (n // 2)] = 32767                                 # I + 9 wraps to -32760
    X = A.reference(A.s16_input(raw, n, ic, qc))
    z = s16_floats(raw, n, ic, qc).copy()
    z[:, n // 2] = np.complex64((32767 + ic) / 32767.0 + 1j * z[:, n // 2].imag)
    psd, _ = fp32_psd(fp32_fft(z), n)
    with pytest.raises(AssertionError):
        A.check_psd(psd, X, s16=True)


@pytest.mark.parametrize("n", A.LENGTHS)
def test_checker_rejects_bf16_spectrum(n):
    raw = noise_s16(n, n + 3)
    X = A.reference(A.s16_input(raw, n))
    psd, _ = fp32_psd(bf16(fp32_fft(s16_floats(raw, n))), n)
    with pytest.raises(AssertionError):
        A.check_psd(psd, X, s16=True)
    x = O.s16_to_float(raw).reshape(BATCH, 2 * n)
    with pytest.raises(AssertionError):
        A.check_spectrum(bf16(fp32_fft(x.view(np.complex64))), A.reference(A.f32_input(x, n)))


@pytest.mark.parametrize("n", A.LENGTHS)
def test_checker_rejects_wrong_peak_bin(n):
    k0, kw = n // 3, (n // 3 + max(1, n // 3)) % n
    r = A.two_tones_s16(n, k0, kw).reshape(1, 2 * n)
    X = A.reference(A.s16_input(r, n))
    psd, pk = fp32_psd(fp32_fft(s16_floats(r, n)), n)
    A.check_peak(psd, pk, X, RATE)
    wrong = (k0 + 1) % n
    psd2 = psd.copy()
    psd2[0, n] = A.peak_hz([wrong], n, RATE)[0]
    with pytest.raises(AssertionError):
        A.check_peak(psd2, np.array([wrong]), X, RATE)
    psd4 = psd.copy()                                            # a self-consistent row, maximum in the wrong bin:
    psd4[0, [k0, wrong]] = psd[0, [wrong, k0]]                   # only the binary64 argmax can tell
    psd4[0, n] = A.peak_hz([wrong], n, RATE)[0]
    with pytest.raises(AssertionError, match="binary64 maximum"):
        A.check_peak(psd4, np.array([wrong]), X, RATE)
    psd3 = psd.copy()                                            # the right bin with another's frequency
    psd3[0, n] = A.peak_hz([wrong], n, RATE)[0]
    if psd3[0, n] != psd[0, n]:
        with pytest.raises(AssertionError):
            A.check_peak(psd3, pk, X, RATE)
