"""GPU parity cases added in round 2 (VERDICT r1 "what's weak" 1 and ADVICE r1):
  * BASELINE config 3 at its real launch size — 10^4 blocks per launch — for N in
    {256, 4096, 19200} (fft.java:190-224; 19200 = rate/10 at 192 kS/s, fft.java:67);
  * the four-step path (N = 32768 / 65536) at a batch that spans >= 3 chunks of its
    32 MB work buffers, s16 and float input;
  * the streaming tuner + decimator across a retune from a negative to a positive
    frequency (tuPhase climbs through zero: mixer bypass at :388,395) against the tile
    kernel and the oracle;
  * JavaAudio's I/Q DC correction (JavaAudio.java:281-288) through the pump call.
"""
import numpy as np
import pytest

import jsdrcuda as J
import oracle as O
from test_gpu_parity import check_psd

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n,rate", [(256, 96000), (4096, 44100), (19200, 192000)])
def test_fft_config3_ten_thousand_blocks_per_launch(ctx, n, rate):
    """Float input, Philox-like uniform [-1,1) blocks with the three known answers in blocks
    0..2 (SURVEY §8d config 3); sampled blocks against the binary64 oracle, every block's
    published maximum against its own row (size independent)."""
    batch = 10000
    rng = np.random.default_rng(42)
    x = rng.uniform(-1, 1, (batch, 2 * n)).astype(np.float32)
    x[0] = 0
    x[0, 0] = 1.0                                            # unit impulse
    x[1] = 0
    x[1, 0::2] = 0.5                                         # DC
    t = np.arange(n)
    tone = 0.8 * np.exp(2j * np.pi * 37 * t / n)             # on-bin tone
    x[2, 0::2], x[2, 1::2] = tone.real, tone.imag
    f = J.fft(ctx, None, J.AudioDescriptor(rate), max_batch=batch, n=n)
    psd, pk = f.receive_batch(x)
    f.close()
    assert np.allclose(psd[0, :n], 10 * np.log10(4.0 / n / n), atol=1e-3)          # flat spectrum
    assert pk[1] == 0 and abs(psd[1, 0] - 20 * np.log10(2 * 0.5)) < 1e-3            # cf = (2/N)^2
    assert pk[2] == 37 and abs(psd[2, 37] - 20 * np.log10(2 * 0.8)) < 1e-3
    for b in [0, 1, 2, 3, 4999, 9998, 9999] + rng.choice(batch, 5, replace=False).tolist():
        check_psd(psd[b], x[b], rate, n)
    # every block: the published maximum is the row maximum at the first bin that holds it
    rows = psd[:, :n]
    assert np.array_equal(psd[:, n + 1], rows.max(axis=1))
    assert np.array_equal(pk, rows.argmax(axis=1))


@pytest.mark.parametrize("fmt", ["f32", "s16"])
def test_fft_fourstep_multi_chunk(ctx, fmt):
    """N = 65536 at batch 200: the host path splits the batch into 32 MB chunks of the
    intermediate (64 blocks each) and alternates two streams and two work buffers; blocks from
    every chunk, including both sides of each chunk boundary and the ragged last one."""
    n, batch = 65536, 200
    rng = np.random.default_rng(65536)
    if fmt == "f32":
        x = rng.uniform(-1, 1, (batch, 2 * n)).astype(np.float32)
        as_float = lambda b: x[b]
    else:
        x = rng.integers(-32768, 32768, (batch, 2 * n)).astype(np.int16)
        as_float = lambda b: O.s16_to_float(x[b])
    f = J.fft(ctx, None, J.AudioDescriptor(192000), max_batch=batch, n=n)
    psd, pk = f.receive_batch(x, s16=(fmt == "s16"))
    f.close()
    for b in (0, 63, 64, 65, 127, 128, 191, 192, 199):
        pw = O.fft_power_f64(as_float(b))
        amp = np.power(10.0, psd[b, :n].astype(np.float64) / 20.0)
        assert np.max(np.abs(amp - np.sqrt(pw))) <= 2e-4, f"block {b}"
    rows = psd[:, :n]
    assert np.array_equal(psd[:, n + 1], rows.max(axis=1))
    assert np.array_equal(pk, rows.argmax(axis=1))


def test_stream_kernel_across_negative_to_positive_retune(ctx):
    """ADVICE r1: after a retune from -f to +f tuPhase starts below zero and climbs; samples
    with phase <= 0 take the bypass.  64 channels so the STREAM kernel is the one that runs;
    it must equal the tile kernel and the oracle bit for bit on every block around the
    crossing (block lengths chosen so the crossing falls inside an anchor window)."""
    rate, nchan = 192000, 64
    rng = np.random.default_rng(77)
    f0 = rng.uniform(100.0, 60000.0, nchan)
    blocks = [777, 4096, 241, 2000]
    raw = [rng.integers(-20000, 20000, (nchan, 2 * s)).astype(np.int16) for s in blocks]
    banks = {k: J.FUNcubeBPSKDemod(ctx, None, J.AudioDescriptor(rate), tuning=-f0, stages=1, max_block=4096)
             for k in (J.KERNEL_STREAM, J.KERNEL_TILE)}
    for k, b in banks.items():
        b.set_kernel(k)
    orcs = [O.Bpsk(rate, -f, stages=1) for f in f0]
    for step, blk in enumerate(raw):
        if step == 1:                                  # now retune every channel to +f (one to 0: stays in bypass)
            for c in range(nchan):
                hz = 0.0 if c == 9 else f0[c]
                for b in banks.values():
                    b.set_tuning(c, hz)
                orcs[c].set_tuning(hz)
        out = {}
        for k, b in banks.items():
            b.receive_raw(blk)
            out[k] = b.read_ds()
        assert np.array_equal(out[J.KERNEL_STREAM], out[J.KERNEL_TILE]), f"block {step}"
        for c in (0, 9, 31, 32, 63):
            assert np.array_equal(out[J.KERNEL_STREAM][c], orcs[c].receive(O.s16_to_float(blk[c]))["ds"]), f"block {step} ch {c}"
    for b in banks.values():
        b.close()


def test_pump_applies_iq_correction(ctx):
    """jsdr_pump_receive_s16(ic, qc): both handlers see s += (short)ic with 16-bit wrap
    (JavaAudio.java:281-288), host and device buffers."""
    rate, nch, n, nblk, ic, qc = 96000, 40, 1024, 2, 117, -9
    rng = np.random.default_rng(5)
    raw = rng.integers(-32768, 32768, (nch, 2 * n * nblk)).astype(np.int16)
    raw[0, :4] = [32767, 32767, -32768, -32768]          # wraps
    tun = rng.uniform(2000, 40000, nch)
    adsc = J.AudioDescriptor(rate)
    f = J.fft(ctx, None, adsc, max_batch=nch * nblk, n=n)
    bank = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tun, max_block=n * nblk, stages=1)
    psd = np.empty((nch * nblk, n + 2), np.float32)
    before = raw.copy()
    J.pump_receive_s16(f, bank, raw, nblk, psd, ic=ic, qc=qc)
    assert np.array_equal(raw, before)                   # raw handlers (recorder.java:66) see uncorrected bytes
    ds = bank.read_ds()
    for c in (0, 17, 39):
        o = O.Bpsk(rate, tun[c], stages=1)
        assert np.array_equal(ds[c], o.receive(O.s16_to_float(raw[c], ic=ic, qc=qc))["ds"])
        check_psd(psd[c * nblk + 1], O.s16_to_float(raw[c, 2 * n:4 * n], ic=ic, qc=qc), rate, n)
    f.close()
    bank.close()


@pytest.mark.parametrize("mem", ["host", "device"])
def test_pump_waterfall_pixels_equal_paintline_of_the_psd(ctx, mem):
    """jsdr_pump_waterfall_s16: the pixel rows are waterfall.paintLine (waterfall.java:90-107) of
    exactly the PSD rows jsdr_pump_receive_s16 returns, the two trailing floats are psd[N] and
    psd[N+1] (fft.java:223-224), and the tuner bank behind it is unchanged."""
    rate, nch, n, nblk, width = 96000, 40, 1024, 3, 400
    rng = np.random.default_rng(8)
    raw = rng.integers(-20000, 20000, (nch, 2 * n * nblk)).astype(np.int16)
    tun = rng.uniform(2000, 40000, nch)
    adsc = J.AudioDescriptor(rate)
    f = J.fft(ctx, None, adsc, max_batch=nch * nblk, n=n)
    b1 = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tun, max_block=n * nblk, stages=1)
    b2 = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tun, max_block=n * nblk, stages=1)
    psd = np.empty((nch * nblk, n + 2), np.float32)
    J.pump_receive_s16(f, b1, raw, nblk, psd)
    pix = np.zeros((nch * nblk, width), np.int32)
    peak = np.zeros((nch * nblk, 2), np.float32)
    pk = np.zeros(nch * nblk, np.int32)
    if mem == "host":
        J.pump_waterfall_s16(f, b2, raw, nblk, width, pix, peak, pk)
    else:
        d_raw, d_pix, d_peak, d_pk = (ctx.dev_alloc(x.nbytes) for x in (raw, pix, peak, pk))
        d_raw.upload(raw)
        J.pump_waterfall_s16(f, b2, d_raw, nblk, width, d_pix, d_peak, d_pk, mem=J.MEM_DEVICE)
        ctx.sync()
        pix = d_pix.download(np.int32, pix.size).reshape(pix.shape)
        peak = d_peak.download(np.float32, peak.size).reshape(peak.shape)
        pk = d_pk.download(np.int32, pk.size)
        for d in (d_raw, d_pix, d_peak, d_pk):
            d.free()
    assert np.array_equal(peak, psd[:, n:])
    for r in (0, 1, 57, nch * nblk - 1):
        assert np.array_equal(pix[r], O.waterfall_row(psd[r], width)), r
    assert np.array_equal(pix, J.waterfall_rows(ctx, psd, width))
    assert np.array_equal(pk, psd[:, :n].argmax(axis=1))
    assert np.array_equal(b1.read_ds(), b2.read_ds())
    for h in (f, b1, b2):
        h.close()


def test_waterfall_rows_more_than_65535(ctx):
    """A pump batch has nchan*nblocks rows: far beyond the 65535 limit of a grid's y dimension."""
    n, rows, width = 128, 70000, 64
    rng = np.random.default_rng(1)
    psd = rng.uniform(-100, 0, (rows, n + 2)).astype(np.float32)
    pix = J.waterfall_rows(ctx, psd, width)
    for r in (0, 65535, 65536, rows - 1):
        assert np.array_equal(pix[r], O.waterfall_row(psd[r], width)), r


def test_pump_waterfall_argument_errors(ctx):
    """Bad arguments are refused with a status code (nothing throws across the ABI)."""
    adsc = J.AudioDescriptor(96000)
    f = J.fft(ctx, None, adsc, max_batch=8, n=256)
    b = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=[12000.0] * 4, max_block=512, stages=1)
    raw = np.zeros((4, 2 * 512), np.int16)
    pix = np.zeros((8, 300), np.int32)
    peak = np.zeros((8, 2), np.float32)
    with pytest.raises(J.JsdrError):
        J.pump_waterfall_s16(f, b, raw, 2, 300, pix, peak)          # width > n
    with pytest.raises(J.JsdrError):
        J.pump_waterfall_s16(f, b, raw, 3, 64, pix, peak)           # nblocks*n beyond the bank's block / the fft's batch
    pix = np.zeros((8, 64), np.int32)
    J.pump_waterfall_s16(f, b, raw, 2, 64, pix, peak)               # and the good call still works afterwards
    assert np.all(np.isneginf(peak[:, 1]) | (peak[:, 1] < -300))    # silence: no bin ever compared greater
    f.close()
    b.close()
