"""demod.java on raw s16 IQ (jsdr_demod_receive_s16 / _audio_s16) and as the third handler of the
pump (jsdr_pump_demod_s16).  The s16 forms convert each sample as JavaAudio.java:276-293 does and
then run the float path, so every output must equal the float entry points on
oracle.s16_to_float(raw, ic, qc) bit for bit."""
import ctypes as C

import numpy as np
import pytest

import jsdrcuda as J
import oracle as O

pytestmark = pytest.mark.gpu

RATE = 96000
LENGTHS = (1, 19, 777, 1024, 1025, 4100)


def raw_block(rng, rows, n):
    """s16 IQ with the values that wrap under ic = +9 / qc = -9 at the start of every row."""
    raw = rng.integers(-32768, 32768, (rows, 2 * n)).astype(np.int16)
    edge = np.array([32767, -32767, -32768, 32760, 32760, -32760, 0, 0], np.int16)
    k = min(edge.size, 2 * n)
    raw[:, :k] = edge[:k]
    return raw


def to_float(raw, ic, qc):
    return np.stack([O.s16_to_float(r, ic, qc) for r in raw])


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint32), np.ascontiguousarray(b).view(np.uint32))


def twin_demods(ctx, nchan, max_block, dofir, dodwn, mode=0, doagc=False):
    out = []
    for _ in range(2):
        d = J.demod(ctx, J.AudioDescriptor(RATE), nchan=nchan, max_block=max_block, dofir=dofir, dodwn=dodwn)
        for c in range(nchan):
            d.weights(-8000 + 3000 * c, 6000 + 3000 * c, chan=c)
        d.set_mode(mode, doagc)
        out.append(d)
    return out


@pytest.mark.parametrize("dofir,dodwn", [(True, True), (True, False), (False, True), (False, False)])
def test_receive_raw_equals_receive_on_converted_floats(ctx, dofir, dodwn):
    """FIR + NCO output, several consecutive calls of ragged lengths, per-channel rows and one
    shared stream, ic/qc that wrap."""
    nchan = 3
    rng = np.random.default_rng(16)
    ds, df = twin_demods(ctx, nchan, 4100, dofir, dodwn)
    for shared in (False, True):
        for n in LENGTHS:
            raw = raw_block(rng, 1 if shared else nchan, n)
            got = ds.receive_raw(raw[0] if shared else raw, ic=9, qc=-9)
            x = to_float(raw, 9, -9)
            ref = df.receive(x[0] if shared else x)
            assert same_bits(got, ref), (shared, n)
    ds.close()
    df.close()


def test_receive_raw_channel_stride_wider_than_block(ctx):
    """chan_stride > nsamples through the C ABI: the gap between rows is never read."""
    L = J.lib()
    nchan, n, stride = 3, 1025, 1100
    rng = np.random.default_rng(17)
    ds, df = twin_demods(ctx, nchan, 4100, True, True)
    for _ in range(3):
        raw = raw_block(rng, nchan, stride)
        out = np.empty((nchan, 2 * n), np.float32)
        J._ck(L.jsdr_demod_receive_s16(ds.h, J._ptr(raw), n, stride, -9, 9, J._ptr(out), J.MEM_HOST))
        ref = df.receive(to_float(raw[:, : 2 * n], -9, 9))
        assert same_bits(out, ref)
    ds.close()
    df.close()


@pytest.mark.parametrize("dofir,dodwn", [(True, True), (True, False), (False, True), (False, False)])
@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("doagc", [False, True])
def test_receive_audio_raw_equals_receive_audio(ctx, dofir, dodwn, mode, doagc):
    nchan = 2
    rng = np.random.default_rng(100 + mode)
    ds, df = twin_demods(ctx, nchan, 4100, dofir, dodwn, mode, doagc)
    for n in LENGTHS:
        raw = raw_block(rng, nchan, n)
        a, ma = ds.receive_audio_raw(raw, ic=9, qc=-9)
        ra, rma = df.receive_audio(to_float(raw, 9, -9))
        assert np.array_equal(a, ra), n
        assert same_bits(ma, rma), n
    ds.close()
    df.close()


def test_s16_and_f32_blocks_alternate_on_one_handle(ctx):
    """The delay line holds converted floats: s16 and f32 blocks on one handle give what an
    all-f32 run on the converted stream gives."""
    nchan = 2
    rng = np.random.default_rng(18)
    dm, df = twin_demods(ctx, nchan, 4100, True, True, J.demod.MODE_NFM, True)
    for i, n in enumerate(LENGTHS * 2):
        raw = raw_block(rng, nchan, n)
        x = to_float(raw, 9, -9)
        a, ma = dm.receive_audio_raw(raw, ic=9, qc=-9) if i % 2 == 0 else dm.receive_audio(x)
        ra, rma = df.receive_audio(x)
        assert np.array_equal(a, ra) and same_bits(ma, rma), (i, n)
        if i % 3 == 2:                                         # the FIR + NCO entry points share the state
            o = dm.receive_raw(raw, ic=9, qc=-9) if i % 2 == 0 else dm.receive(x)
            assert same_bits(o, df.receive(x)), (i, n)
    dm.close()
    df.close()


@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
def test_audio_raw_against_the_oracle(ctx, mode):
    """Without the NCO every s16 sample equals the oracle's; with it (cos/sin from another libm)
    within one LSB."""
    nchan = 2
    rng = np.random.default_rng(200 + mode)
    for dodwn in (False, True):
        d = J.demod(ctx, J.AudioDescriptor(RATE), nchan=nchan, max_block=4100, dofir=True, dodwn=dodwn)
        d.set_mode(mode, True)
        orc, lilq = [], [np.zeros(2, np.float32) for _ in range(nchan)]
        for c in range(nchan):
            d.weights(9000 + 1000 * c, 15000, chan=c)
            o = O.Demod(RATE, True, dodwn)
            o.weights(9000 + 1000 * c, 15000)
            orc.append(o)
        for n in LENGTHS:
            raw = (rng.standard_normal((nchan, 2 * n)) * 6000).astype(np.int16)
            audio, ma = d.receive_audio_raw(raw, ic=9, qc=-9)
            for c in range(nchan):
                ref, rma = O.demod_detect(orc[c].receive(O.s16_to_float(raw[c], 9, -9)), mode, RATE, True, lilq[c])
                if dodwn:
                    assert np.max(np.abs(audio[c].astype(np.int32) - ref.astype(np.int32))) <= 1, (n, c)
                else:
                    assert np.array_equal(audio[c], ref), (n, c)
                    assert np.array_equal(ma[c], rma, equal_nan=True), (n, c)
        d.close()


# ---------------------------------------------------------------------------- the pump
def _pump_handles(ctx, n, nblk, nchan, mode):
    adsc = J.AudioDescriptor(RATE)
    tun = [12000.0, -7000.0, 30000.0][:nchan]
    f = [J.fft(ctx, None, adsc, max_batch=nchan * nblk, n=n) for _ in range(2)]
    b = [J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tun, max_block=nblk * n, stages=3) for _ in range(2)]
    d, dref = twin_demods(ctx, nchan, nblk * n, True, True, mode, True)
    return f, b, d, dref


@pytest.mark.parametrize("mem", [J.MEM_HOST, J.MEM_DEVICE])
@pytest.mark.parametrize("nblk", [1, 3])
@pytest.mark.parametrize("mode", [2, 3, 4])
def test_pump_demod_equals_the_handlers_one_by_one(ctx, mem, nblk, mode):
    """PSD, peak bins, decimated rows, bits and counters equal jsdr_pump_receive_s16's on twin
    handles; audio and max_avg equal nblocks successive receive_audio calls of n samples per
    channel on the converted input.  Two pump calls in a row."""
    n, nchan, ic, qc = 1024, 3, 9, -9
    S = nblk * n
    rng = np.random.default_rng(300 + 10 * mode + nblk)
    f, b, d, dref = _pump_handles(ctx, n, nblk, nchan, mode)
    for call in range(2):
        raw = raw_block(rng, nchan, S)
        psd = [np.zeros((nchan * nblk, n + 2), np.float32) for _ in range(2)]
        pk = [np.zeros(nchan * nblk, np.int32) for _ in range(2)]
        audio = np.zeros((nchan, S), np.int16)
        ma = np.zeros((nchan, nblk, 2), np.float32)
        J.pump_receive_s16(f[0], b[0], raw, nblk, psd[0], pk[0], ic=ic, qc=qc)
        if mem == J.MEM_HOST:
            J.pump_demod_s16(f[1], b[1], d, raw, nblk, psd[1], audio, ma, pk[1], ic=ic, qc=qc)
        else:
            bufs = [ctx.dev_alloc(x.nbytes) for x in (raw, psd[1], pk[1], audio, ma)]
            bufs[0].upload(raw)
            J.pump_demod_s16(f[1], b[1], d, bufs[0], nblk, bufs[1], bufs[3], bufs[4], bufs[2], mem=J.MEM_DEVICE,
                             ic=ic, qc=qc)
            ctx.sync()
            psd[1][:] = bufs[1].download(np.float32, psd[1].size).reshape(psd[1].shape)
            pk[1][:] = bufs[2].download(np.int32, pk[1].size)
            audio[:] = bufs[3].download(np.int16, audio.size).reshape(audio.shape)
            ma[:] = bufs[4].download(np.float32, ma.size).reshape(ma.shape)
            for x in bufs:
                x.free()
        assert same_bits(psd[0], psd[1]) and np.array_equal(pk[0], pk[1]), call
        assert same_bits(b[0].read_ds(), b[1].read_ds()), call
        b0, b1 = b[0].read_bits(), b[1].read_bits()
        for c in range(nchan):
            assert np.array_equal(b0[0][c], b1[0][c]) and np.array_equal(b0[1][c], b1[1][c]), (call, c)
        assert np.array_equal(b[0].counters(), b[1].counters()), call
        x = to_float(raw, ic, qc)
        for j in range(nblk):
            ra, rma = dref.receive_audio(x[:, 2 * j * n: 2 * (j + 1) * n])
            assert np.array_equal(audio[:, j * n: (j + 1) * n], ra), (call, j)
            assert same_bits(ma[:, j], rma), (call, j)
    for h in f + b + [d, dref]:
        h.close()


# ---------------------------------------------------------------------------- robustness
GUARD = 4096


def _guarded(ctx, nbytes):
    buf = ctx.dev_alloc(nbytes + GUARD)
    buf.upload(np.full(nbytes + GUARD, 0xA5, np.uint8))
    return buf


def _guard_intact(buf, nbytes):
    return bool(np.all(buf.download(np.uint8, GUARD, offset=nbytes) == 0xA5))


def test_device_outputs_stay_inside_their_buffers(ctx):
    L = J.lib()
    nchan, n, nblk = 3, 1024, 3
    S = n * nblk
    rng = np.random.default_rng(19)
    raw = raw_block(rng, nchan, S)
    d_raw = ctx.dev_alloc(raw.nbytes)
    d_raw.upload(raw)
    d = J.demod(ctx, J.AudioDescriptor(RATE), nchan=nchan, max_block=S)
    d.weights(3000, 9000)
    d.set_mode(J.demod.MODE_AM, True)
    for m in (777, S):
        out = _guarded(ctx, nchan * m * 8)
        J._ck(L.jsdr_demod_receive_s16(d.h, J._ptr(d_raw), m, S, 9, -9, J._ptr(out), J.MEM_DEVICE))
        aud, ma = _guarded(ctx, nchan * m * 2), _guarded(ctx, nchan * 8)
        J._ck(L.jsdr_demod_receive_audio_s16(d.h, J._ptr(d_raw), m, S, 9, -9, J._ptr(aud), J._ptr(ma), J.MEM_DEVICE))
        ctx.sync()
        assert _guard_intact(out, nchan * m * 8) and _guard_intact(aud, nchan * m * 2) and _guard_intact(ma, nchan * 8), m
        for x in (out, aud, ma):
            x.free()
    adsc = J.AudioDescriptor(RATE)
    f = J.fft(ctx, None, adsc, max_batch=nchan * nblk, n=n)
    b = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=[12000.0, 9000.0, 3000.0], max_block=S)
    psd, pk = _guarded(ctx, nchan * nblk * (n + 2) * 4), _guarded(ctx, nchan * nblk * 4)
    aud, ma = _guarded(ctx, nchan * S * 2), _guarded(ctx, nchan * nblk * 8)
    for max_avg in (ma, None):
        J.pump_demod_s16(f, b, d, d_raw, nblk, psd, aud, max_avg, pk, mem=J.MEM_DEVICE)
        ctx.sync()
        assert _guard_intact(aud, nchan * S * 2) and _guard_intact(ma, nchan * nblk * 8)
        assert _guard_intact(psd, nchan * nblk * (n + 2) * 4) and _guard_intact(pk, nchan * nblk * 4)
    # per block: a pump of one block writes one pair per channel and one block of audio per channel
    for x, nb in ((ma, nchan * nblk * 8), (aud, nchan * S * 2)):
        x.upload(np.full(nb + GUARD, 0xA5, np.uint8))
    J.pump_demod_s16(f, b, d, d_raw, 1, psd, aud, ma, pk, mem=J.MEM_DEVICE)
    ctx.sync()
    assert _guard_intact(ma, nchan * 8) and _guard_intact(aud, nchan * n * 2)
    for x in (psd, pk, aud, ma, d_raw):
        x.free()
    for h in (f, b, d):
        h.close()


def test_bad_arguments_are_refused(ctx):
    L = J.lib()
    nchan, n = 2, 1024
    adsc = J.AudioDescriptor(RATE)
    d = J.demod(ctx, adsc, nchan=nchan, max_block=2 * n)
    d.weights(3000, 9000)
    raw = np.zeros((nchan, 4 * n), np.int16)
    out = np.zeros((nchan, 4 * n), np.float32)
    aud = np.zeros((nchan, 2 * n), np.int16)
    ma = np.zeros((nchan, 2, 2), np.float32)
    P = J._ptr

    def refused(rc):
        assert rc == -1 and L.jsdr_last_error(), rc

    for fn, tail in ((L.jsdr_demod_receive_s16, (P(out), J.MEM_HOST)),
                     (L.jsdr_demod_receive_audio_s16, (P(aud), P(ma), J.MEM_HOST))):
        refused(fn(d.h, None, n, n, 0, 0, *tail))                          # null input
        refused(fn(d.h, P(raw), 2 * n + 1, 0, 0, 0, *tail))                # beyond max_block_samples
        refused(fn(d.h, P(raw), n, n - 1, 0, 0, *tail))                    # rows overlap
        refused(fn(d.h, P(raw), -1, 0, 0, 0, *tail))
        refused(fn(d.h, P(raw), n, n, 0, 0, *tail[:-1], 2))                # mem out of range
    refused(L.jsdr_demod_receive_s16(d.h, P(raw), n, n, 0, 0, None, J.MEM_HOST))
    refused(L.jsdr_demod_receive_audio_s16(d.h, P(raw), n, n, 0, 0, None, P(ma), J.MEM_HOST))

    f = J.fft(ctx, None, adsc, max_batch=4 * nchan, n=n)
    b = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=[12000.0, 9000.0], max_block=4 * n)
    b3 = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=[12000.0, 9000.0, 3000.0], max_block=4 * n)
    other = J.Context(0)
    d_other = J.demod(other, adsc, nchan=nchan, max_block=2 * n)
    psd = np.zeros((4 * nchan, n + 2), np.float32)
    pk = np.zeros(4 * nchan, np.int32)

    def pump(fh, bh, dh, nblk=2, r=P(raw), ps=P(psd), a=P(aud), mem=J.MEM_HOST):
        return L.jsdr_pump_demod_s16(fh, bh, dh, r, nblk, 0, 0, ps, P(pk), a, P(ma), mem)

    refused(pump(f.h, b.h, None))
    refused(pump(None, b.h, d.h))
    refused(pump(f.h, None, d.h))
    refused(pump(f.h, b.h, d.h, r=None))
    refused(pump(f.h, b.h, d.h, ps=None))
    refused(pump(f.h, b.h, d.h, a=None))
    refused(pump(f.h, b.h, d_other.h))                                     # another context
    refused(pump(f.h, b3.h, d.h))                                          # channel counts differ
    refused(pump(f.h, b.h, d.h, nblk=3))                                   # beyond the demod's max_block_samples
    refused(pump(f.h, b.h, d.h, nblk=0))
    refused(pump(f.h, b.h, d.h, nblk=-1))
    refused(pump(f.h, b.h, d.h, mem=2))
    refused(pump(f.h, b.h, d.h, mem=-1))
    # the handles still work and match a fresh twin
    rng = np.random.default_rng(20)
    x = raw_block(rng, nchan, n)
    d2 = J.demod(ctx, adsc, nchan=nchan, max_block=2 * n)
    d2.weights(3000, 9000)
    assert same_bits(d.receive_raw(x), d2.receive_raw(x))
    for h in (d, d2, f, b, b3, d_other):
        h.close()
    other.close()


def test_empty_calls_write_nothing(ctx):
    L = J.lib()
    nchan = 2
    d = J.demod(ctx, J.AudioDescriptor(RATE), nchan=nchan, max_block=1024)
    d.weights(3000, 9000)
    d.set_mode(J.demod.MODE_NFM, True)
    raw = np.ones((nchan, 64), np.int16)
    out = np.full((nchan, 64), 7.0, np.float32)
    aud = np.full((nchan, 32), 7, np.int16)
    ma = np.full((nchan, 2), 7.0, np.float32)
    assert L.jsdr_demod_receive_s16(d.h, J._ptr(raw), 0, 0, 0, 0, J._ptr(out), J.MEM_HOST) == 0
    assert L.jsdr_demod_receive_audio_s16(d.h, J._ptr(raw), 0, 32, 0, 0, J._ptr(aud), J._ptr(ma), J.MEM_HOST) == 0
    assert np.all(out == 7.0) and np.all(aud == 7) and np.all(ma == 7.0)
    # and the state did not move: the next block equals a fresh handle's first
    d2 = J.demod(ctx, J.AudioDescriptor(RATE), nchan=nchan, max_block=1024)
    d2.weights(3000, 9000)
    d2.set_mode(J.demod.MODE_NFM, True)
    rng = np.random.default_rng(21)
    x = raw_block(rng, nchan, 300)
    a1, m1 = d.receive_audio_raw(x)
    a2, m2 = d2.receive_audio_raw(x)
    assert np.array_equal(a1, a2) and same_bits(m1, m2)
    d.close()
    d2.close()
