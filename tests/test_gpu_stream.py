"""GPU parity of the streaming tuner + decimator kernel (csrc/bpsk_stream.cuh): one
lane per channel.  binary64 mode must be bit-identical to the oracle's restatement
of FUNcubeBPSKDemod.java:382-397,467-492 and to the tile kernel; binary32 mode must
stay within a per-output bound derived from its arithmetic (tests/f32_bound.py), far inside 1e-4 of full
scale (BASELINE.json north_star) of the binary64 path."""
import numpy as np
import pytest

import jsdrcuda as J
import oracle as O
from oracle import siggen

pytestmark = pytest.mark.gpu

FULL_SCALE = 0.9 * 32768.0        # decimator output for a full-scale input (:469, taps sum to ~1)


def make_bank(ctx, rate, tun, taps, kernel, prec=J.PREC_F64, max_block=None):
    bank = J.FUNcubeBPSKDemod(ctx, None, J.AudioDescriptor(rate), tuning=tun, stages=1, max_block=max_block)
    if taps is not None:
        bank.set_ds_filter(taps)
    bank.set_kernel(kernel)
    bank.set_precision(prec)
    return bank


@pytest.mark.parametrize("fmt", ["s16", "f32"])
@pytest.mark.parametrize("rate,ntaps", [(96000, 27), (192000, 27), (192000, 64)])
def test_stream_bit_exact_vs_oracle_ragged_blocks(ctx, rate, ntaps, fmt):
    """Every compiled (taps, D) shape, 37 channels (one full warp + a partial one),
    ragged block lengths so that the decimation phase, the history and the tuner
    checkpoints all carry across calls."""
    nchan = 37
    rng = np.random.default_rng(100 + ntaps + rate // 1000)
    tun = rng.uniform(2000, rate * 0.47, nchan)
    tun[3] = 0.0                      # mixer bypass (tuPhase stays 0, :388,395)
    tun[5] = rate * 0.4999            # increment just under pi: exact-replay lane
    tun[7] = 12000.0
    taps = siggen.lowpass_taps(64, 4800.0, rate) if ntaps == 64 else None
    bank = make_bank(ctx, rate, tun, taps, J.KERNEL_STREAM, max_block=8192)
    orcs = [O.Bpsk(rate, t, ds_taps=taps, stages=1) for t in tun]
    for S in (4000, 1, 19, 8192, 777, 2561, 64, 3000):
        if fmt == "s16":                                   # IRawHandler bytes, converted on the device
            raw = rng.integers(-32768, 32768, (nchan, 2 * S)).astype(np.int16)
            bank.receive_raw(raw)
            fin = [O.s16_to_float(raw[c]) for c in range(nchan)]
        else:                                              # IAudioHandler floats
            fin = rng.uniform(-1, 1, (nchan, 2 * S)).astype(np.float32)
            bank.receive(fin)
        ds = bank.read_ds()
        for c, o in enumerate(orcs):
            ref = o.receive(fin[c])["ds"]
            assert ds[c].shape == ref.shape, (S, c)
            assert np.array_equal(ds[c], ref), (S, c)
    bank.close()


def test_stream_equals_tile_kernel_many_segments(ctx):
    """Config-4 shape (64 taps, D=20) with enough outputs for several segments per
    channel; the two kernels must agree bit for bit, with I/Q correction on."""
    rate, nchan, S = 192000, 96, 40000
    rng = np.random.default_rng(5)
    tun = rng.uniform(2000, 90000, nchan)
    taps = siggen.lowpass_taps(64, 4800.0, rate)
    a = make_bank(ctx, rate, tun, taps, J.KERNEL_STREAM, max_block=S)
    b = make_bank(ctx, rate, tun, taps, J.KERNEL_TILE, max_block=S)
    for k in range(3):
        raw = rng.integers(-32768, 32768, (nchan, 2 * S)).astype(np.int16)
        a.receive_raw(raw, ic=37, qc=-1234)
        b.receive_raw(raw, ic=37, qc=-1234)
        assert np.array_equal(a.read_ds(), b.read_ds()), k
    o = O.Bpsk(rate, tun[40], ds_taps=taps, stages=1)          # anchor one channel on the oracle too
    a2 = make_bank(ctx, rate, tun, taps, J.KERNEL_STREAM, max_block=S)
    raw = rng.integers(-32768, 32768, (nchan, 2 * S)).astype(np.int16)
    a2.receive_raw(raw)
    assert np.array_equal(a2.read_ds()[40], o.receive(O.s16_to_float(raw[40]))["ds"])
    for h in (a, b, a2):
        h.close()


def test_stream_shared_stream_fans_out(ctx):
    """chan_stride == 0: one stream to every tuner (jsdr.java:479-483)."""
    rate, nchan, S = 96000, 40, 9600
    rng = np.random.default_rng(6)
    tun = rng.uniform(2000, 40000, nchan)
    raw = rng.integers(-20000, 20000, 2 * S).astype(np.int16)
    a = make_bank(ctx, rate, tun, None, J.KERNEL_STREAM)
    a.receive_raw(raw, shared=True)
    ds = a.read_ds()
    for c in (0, 17, 39):
        o = O.Bpsk(rate, tun[c], stages=1)
        assert np.array_equal(ds[c], o.receive(O.s16_to_float(raw))["ds"])
    a.close()


@pytest.mark.parametrize("rate,ntaps", [(96000, 27), (192000, 64)])
def test_stream_f32_within_tolerance(ctx, rate, ntaps):
    """binary32 mix + FIR against the binary64 oracle, every channel: every output within the bound derived
    from the kernel's arithmetic (tests/f32_bound.py), and so within 1e-4 of full scale (s16 and float
    input)."""
    import f32_bound as F
    nchan, S = 64, 19200
    rng = np.random.default_rng(8)
    tun = rng.uniform(2000, rate * 0.45, nchan)
    taps = siggen.lowpass_taps(64, 4800.0, rate) if ntaps == 64 else None
    a = make_bank(ctx, rate, tun, taps, J.KERNEL_STREAM, prec=J.PREC_F32, max_block=S)
    orcs = [O.Bpsk(rate, t, ds_taps=taps, stages=1) for t in tun]
    bounds = [F.Bound(O.default_taps()[0] if taps is None else taps, rate // 9600, True) for _ in tun]
    worst = 0.0
    for k in range(4):
        raw = rng.integers(-32768, 32768, (nchan, 2 * S)).astype(np.int16)
        fin = O.s16_to_float(raw.ravel()).reshape(nchan, 2 * S)
        if k < 2:
            a.receive_raw(raw)
        else:
            a.receive(fin)
        ds = a.read_ds()
        for c, o in enumerate(orcs):
            ref = o.receive(fin[c])["ds"]
            assert np.all(np.abs(ds[c] - ref) <= bounds[c].block(fin[c], s16=k < 2)), (k, c)
            worst = max(worst, float(np.max(np.abs(ds[c] - ref))) / FULL_SCALE)
    assert worst <= 1e-4, worst
    assert worst <= 2e-6, worst       # what binary32 actually achieves here
    a.close()


def test_pump_host_path_chunked_equals_separate_handlers(ctx):
    """jsdr_pump_receive_s16 with host buffers pipelines the batch over channel chunks
    (upload / FFT / download overlapped); results must equal the two handlers run apart."""
    rate, nchan, n, nblk = 192000, 44, 4096, 2
    rng = np.random.default_rng(21)
    tun = rng.uniform(2000, 90000, nchan)
    raw = rng.integers(-30000, 30000, (nchan, nblk * n * 2)).astype(np.int16)
    adsc = J.AudioDescriptor(rate)
    f = J.fft(ctx, None, adsc, max_batch=nchan * nblk, n=n)
    b1 = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tun, max_block=nblk * n, stages=1)
    b2 = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tun, max_block=nblk * n, stages=1)
    psd = np.empty((nchan * nblk, n + 2), np.float32)
    pk = np.empty(nchan * nblk, np.int32)
    for k in range(2):
        J.pump_receive_s16(f, b1, raw, nblk, psd, pk)
        psd2, pk2 = f.receive_batch(raw.reshape(nchan * nblk, 2 * n), s16=True)
        assert np.array_equal(psd, psd2) and np.array_equal(pk, pk2)
        b2.receive_raw(raw)
        assert np.array_equal(b1.read_ds(), b2.read_ds())
    for h in (f, b1, b2):
        h.close()


def test_async_ds_read_equals_blocking_read_and_orders_the_next_block(ctx):
    """jsdr_bpsk_read_ds_async copies on the download stream without waiting; the rows must
    equal the blocking read's, also when the next block is submitted straight behind it
    (that block's decimator has to wait for the copy before it overwrites the device rows)."""
    rate, nchan, S = 192000, 96, 8192
    rng = np.random.default_rng(5)
    tun = rng.uniform(2000, 90000, nchan)
    adsc = J.AudioDescriptor(rate)
    a = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tun, max_block=S, stages=1)
    b = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tun, max_block=S, stages=1)
    outs = [ctx.host_alloc((nchan * (S // 20 + 1) * 2,), np.float64) for _ in range(3)]
    raws = [rng.integers(-30000, 30000, (nchan, 2 * S)).astype(np.int16) for _ in range(3)]
    want, counts = [], []
    for k in range(3):
        a.receive_raw(raws[k])
        want.append(a.read_ds())
        b.receive_raw(raws[k])
        counts.append(b.read_ds_async(outs[k]))     # no wait: the next receive follows at once
    ctx.sync()
    for k in range(3):
        n = counts[k]
        assert n == want[k].shape[1]
        assert np.array_equal(outs[k][: nchan * n * 2].reshape(nchan, n, 2), want[k]), k
    a.close()
    b.close()


def test_full_size_bank_stream_equals_tile_and_is_linear(ctx):
    """BASELINE config 4's full bank (4096 channels, 192 kS/s, 64 taps, D=20) on 32768-sample
    blocks: the streaming kernel (every SM, several segments per channel, phase checkpoints
    from the look-ahead scout) must equal the tile kernel bit for bit on every channel, and a
    sample of channels must equal the oracle."""
    rate, nchan, S = 192000, 4096, 32768
    rng = np.random.default_rng(77)
    from jsdrcuda import sharding
    tun = sharding.channel_tuning(0, nchan)
    taps = siggen.lowpass_taps(64, 4800.0, rate)
    a = make_bank(ctx, rate, tun, taps, J.KERNEL_STREAM, max_block=S)
    b = make_bank(ctx, rate, tun, taps, J.KERNEL_TILE, max_block=S)
    base = rng.integers(-32768, 32768, (64, 2 * S)).astype(np.int16)
    raw = np.ascontiguousarray(np.tile(base, (nchan // 64, 1)))
    orcs = {c: O.Bpsk(rate, tun[c], ds_taps=taps, stages=1) for c in (0, 1777, 4095)}
    for k in range(2):
        raw = np.roll(raw, 12345 * (k + 1), axis=1)
        a.receive_raw(raw)
        b.receive_raw(raw)
        da, db = a.read_ds(), b.read_ds()
        assert da.shape == db.shape and da.shape[0] == nchan and abs(da.shape[1] - S / 20) < 1
        assert np.array_equal(da, db), k
        for c, o in orcs.items():
            assert np.array_equal(da[c], o.receive(O.s16_to_float(raw[c]))["ds"]), (k, c)
    a.close()
    b.close()
