"""GPU parity of the section-8f rows built so far: demod.java's detectors / AGC / s16
narrowing (:405-481) and waterfall.java's row (:90-107).  Integer outputs: bit-exact."""
import numpy as np
import pytest

import jsdrcuda as J
import nco_phase as N
import oracle as O

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("doagc", [False, True])
def test_demod_audio_bit_exact_without_nco(ctx, mode, doagc):
    """FIR (exact float order) + detector + AGC + (short) narrowing; the NCO is off so no
    transcendental enters and every s16 sample must equal the oracle's."""
    rate, nchan = 96000, 3
    rng = np.random.default_rng(10 + mode)
    d = J.demod(ctx, J.AudioDescriptor(rate), nchan=nchan, max_block=9600, dofir=True, dodwn=False)
    d.set_mode(mode, doagc)
    os_, lilq = [], [np.zeros(2, np.float32) for _ in range(nchan)]
    for c in range(nchan):
        d.weights(-8000 + 3000 * c, 6000 + 3000 * c, chan=c)
        o = O.Demod(rate, True, False)
        o.weights(-8000 + 3000 * c, 6000 + 3000 * c)
        os_.append(o)
    for n in (9600, 1, 777, 2048, 2049, 4100):
        x = (rng.standard_normal((nchan, 2 * n)) * 0.3).astype(np.float32)
        audio, ma = d.receive_audio(x)
        for c in range(nchan):
            ref_a, ref_ma = O.demod_detect(os_[c].receive(x[c]), mode, rate, doagc, lilq[c])
            assert np.array_equal(audio[c], ref_a), (n, c)
            assert np.array_equal(ma[c], ref_ma, equal_nan=True), (n, c)
    d.close()


@pytest.mark.parametrize("doagc", [False, True])
def test_am_running_mean_special_operands(ctx, doagc):
    """demod.java:451's running mean over the operands the kernel's reciprocal-pair quotient hands
    to the IEEE division instead (amplitudes below 2^-38, infinities, NaN), zeros, and both sides of
    that guard; no FIR, no NCO: every s16 sample, max and avg equal to the oracle's."""
    rate = 96000
    scales = [0.0, 1e-25, 3e-19, 9e-19, 1e-12, 3e-12, 1e-9, 1.0, 1e15, 1e19, 3e19]
    nchan = len(scales) + 3
    rng = np.random.default_rng(451)
    d = J.demod(ctx, J.AudioDescriptor(rate), nchan=nchan, max_block=9600, dofir=False, dodwn=False)
    d.set_mode(J.demod.MODE_AM, doagc)
    lilq = np.zeros(2, np.float32)
    for n in (9600, 5, 777, 2056, 4100):
        x = np.empty((nchan, 2 * n), np.float32)
        for c, sc in enumerate(scales):
            x[c] = (rng.standard_normal(2 * n) * sc).astype(np.float32)
        x[len(scales)] = rng.standard_normal(2 * n).astype(np.float32)
        x[len(scales), : 2 * (n // 2)] = 0.0                     # silence, then signal
        x[len(scales) + 1] = rng.standard_normal(2 * n).astype(np.float32)
        x[len(scales) + 1, 2 * (n // 3)] = np.inf                # one infinite sample: avg = inf, then NaN
        x[len(scales) + 2] = rng.standard_normal(2 * n).astype(np.float32)
        x[len(scales) + 2, 2 * (n // 2) + 1] = np.nan
        audio, ma = d.receive_audio(x)
        for c in range(nchan):
            o = O.Demod(rate, False, False)
            with np.errstate(all="ignore"):
                ref_a, ref_ma = O.demod_detect(o.receive(x[c]), 2, rate, doagc, lilq)
            assert np.array_equal(audio[c], ref_a), (n, c)
            assert np.array_equal(ma[c], ref_ma, equal_nan=True), (n, c)
    d.close()


def test_demod_audio_with_nco_bit_exact(ctx):
    """With the down-shift on: every s16 sample and max/avg pair equal to the oracle's detectors on
    the NCO model of tests/nco_phase.py (the kernel's own sine / cosine, emulated bit for bit)."""
    rate = 96000
    rng = np.random.default_rng(3)
    d = J.demod(ctx, J.AudioDescriptor(rate), max_block=9600)
    d.weights(9000, 15000)
    d.set_mode(J.demod.MODE_NFM, False)
    o = N.RefDemod(rate)
    o.weights(9000, 15000)
    lilq = np.zeros(2, np.float32)
    for _ in range(3):
        x = (rng.standard_normal(2 * 9600) * 0.2).astype(np.float32)
        audio, ma = d.receive_audio(x)
        mixed, allowed = o.receive(x)
        assert not allowed
        ref, rma = O.demod_detect(mixed, 3, rate, False, lilq)
        assert np.array_equal(audio[0], ref) and np.array_equal(ma[0], rma)
    d.close()


def test_waterfall_rows_bit_exact(ctx):
    rng = np.random.default_rng(5)
    for n, width in ((4096, 512), (9600, 1000), (19200, 1919), (4410, 640)):
        psd = rng.uniform(-130, 5, (7, n + 2)).astype(np.float32)
        psd[0, :n] = -np.inf                                  # log10(0) rows (SURVEY Q4)
        pix = J.waterfall_rows(ctx, psd, width)
        for r in range(psd.shape[0]):
            assert np.array_equal(pix[r], O.waterfall_row(psd[r], width)), (n, width, r)
    # chained behind the FFT: the published psd of a tone, straight to a pixel row
    n = 4096
    t = np.arange(n)
    x = np.empty(2 * n, np.float32)
    x[0::2], x[1::2] = np.cos(2 * np.pi * 400 * t / n), np.sin(2 * np.pi * 400 * t / n)
    f = J.fft(ctx, None, J.AudioDescriptor(44100, blen=4 * n))
    row = J.waterfall_rows(ctx, f.receive(x), 512).view(np.uint32)[0]
    assert int(np.argmax(row & 0xFF)) == (400 // 8 + 256) % 512
    f.close()
