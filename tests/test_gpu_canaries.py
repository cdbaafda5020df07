"""Out-of-bounds writes, checked with guard bands (compute-sanitizer is closed on the GPU pool).

Every device-resident output of the C-ABI is placed inside a larger allocation whose margins
hold a byte pattern; after the call the margins must be untouched and the payload must equal
what the same call returns through host buffers (which the parity tests tie to the oracle).
Sizes are ragged on purpose: batches that do not fill a wave, channel counts that do not fill a
warp, widths that do not divide N, block lengths that are not multiples of the decimation.
"""
import ctypes as C

import numpy as np
import pytest

import jsdrcuda as J

pytestmark = pytest.mark.gpu

PAD = 8192                                                   # bytes of margin on either side
FILL = 0xA5


class Guarded:
    """`nbytes` of device memory between two margins of FILL bytes."""

    def __init__(self, ctx, nbytes):
        self.nbytes = int(nbytes)
        self.buf = ctx.dev_alloc(self.nbytes + 2 * PAD)
        self.buf.upload(np.full(self.nbytes + 2 * PAD, FILL, dtype=np.uint8))
        self.ptr = self.buf.ptr + PAD

    def payload(self, dtype):
        return self.buf.download(np.uint8, self.nbytes, PAD).view(dtype)

    def check(self, what):
        lo = self.buf.download(np.uint8, PAD, 0)
        hi = self.buf.download(np.uint8, PAD, PAD + self.nbytes)
        assert np.all(lo == FILL), f"{what}: write below the buffer, first at byte {-PAD + int(np.argmax(lo != FILL))}"
        assert np.all(hi == FILL), f"{what}: write above the buffer, first at byte +{int(np.argmax(hi != FILL))}"

    def free(self):
        self.buf.free()


def _dev(ctx, a):
    d = ctx.dev_alloc(a.nbytes)
    d.upload(a)
    return d


@pytest.mark.parametrize("n,batch", [(128, 5), (256, 1), (777, 3), (1000, 3), (6000, 2), (4096, 7), (4410, 2), (9600, 3), (19200, 2),
                                     (32768, 3), (65536, 2)])
@pytest.mark.parametrize("fmt", ["s16", "f32"])
def test_fft_outputs_stay_inside(ctx, n, batch, fmt):
    if not J.fft_supported(n):                 # no plan (777 = 3 * 7 * 37): refused before anything is written
        with pytest.raises(J.JsdrError):
            J.fft(ctx, None, J.AudioDescriptor(96000), max_batch=batch, n=n)
        return
    rng = np.random.default_rng(n + batch)
    if fmt == "s16":
        x = rng.integers(-20000, 20000, (batch, 2 * n)).astype(np.int16)
    else:
        x = rng.uniform(-1, 1, (batch, 2 * n)).astype(np.float32)
    f = J.fft(ctx, None, J.AudioDescriptor(96000), max_batch=batch, n=n)
    psd_h, pk_h = f.receive_batch(x, s16=(fmt == "s16"))
    d_in = _dev(ctx, x)
    g_psd, g_pk = Guarded(ctx, batch * (n + 2) * 4), Guarded(ctx, batch * 4)
    f.receive_dev(d_in.ptr, batch, g_psd.ptr, g_pk.ptr, s16=(fmt == "s16"))
    ctx.sync()
    g_psd.check(f"psd n={n}")
    g_pk.check(f"peak n={n}")
    assert np.array_equal(g_psd.payload(np.float32).reshape(batch, n + 2), psd_h)
    assert np.array_equal(g_pk.payload(np.int32), pk_h)
    for b in (d_in, g_psd.buf, g_pk.buf):
        b.free()
    f.close()


@pytest.mark.parametrize("nchan,nblk,rate,n", [(37, 3, 96000, 4096), (5, 2, 192000, 19200), (64, 1, 96000, 4096)])
def test_pump_outputs_stay_inside(ctx, nchan, nblk, rate, n):
    rng = np.random.default_rng(nchan)
    raw = rng.integers(-12000, 12000, (nchan, nblk * n * 2)).astype(np.int16)
    tuning = np.linspace(-30000.0, 30000.0, nchan)
    adsc = J.AudioDescriptor(rate, blen=n * 4)

    def run(device):
        f = J.fft(ctx, None, adsc, max_batch=nchan * nblk, n=n)
        b = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tuning, max_block=nblk * n)
        if device:
            d_raw = _dev(ctx, raw)
            g_psd, g_pk = Guarded(ctx, nchan * nblk * (n + 2) * 4), Guarded(ctx, nchan * nblk * 4)
            J.pump_receive_s16(f, b, d_raw.ptr, nblk, g_psd.ptr, g_pk.ptr, mem=J.MEM_DEVICE)
            ctx.sync()
            nds = b.last_nds()
            g_ds, g_dm = Guarded(ctx, nchan * nds * 16), Guarded(ctx, nchan * nds * 16)
            J._ck(J.lib().jsdr_bpsk_read_ds(b.h, C.c_void_p(g_ds.ptr), J.MEM_DEVICE))
            J._ck(J.lib().jsdr_bpsk_read_dm(b.h, C.c_void_p(g_dm.ptr), J.MEM_DEVICE))
            ctx.sync()
            for g, what in ((g_psd, "psd"), (g_pk, "peak"), (g_ds, "ds"), (g_dm, "dm")):
                g.check(f"pump {what} nchan={nchan}")
            out = (g_psd.payload(np.float32).copy(), g_pk.payload(np.int32).copy(), g_ds.payload(np.float64).copy(),
                   g_dm.payload(np.float64).copy())
            for g in (g_psd, g_pk, g_ds, g_dm):
                g.free()
            d_raw.free()
        else:
            psd = np.zeros((nchan * nblk, n + 2), dtype=np.float32)
            pk = np.zeros(nchan * nblk, dtype=np.int32)
            J.pump_receive_s16(f, b, raw, nblk, psd, pk)
            out = (psd.ravel(), pk, b.read_ds().ravel(), b.read_dm().ravel())
        b.close()
        f.close()
        return out

    dev, host = run(True), run(False)
    for d, h, what in zip(dev, host, ("psd", "peak", "ds", "dm")):
        assert d.size == h.size and np.array_equal(d, h), what


@pytest.mark.parametrize("width", [1, 333, 1000, 4096])
def test_waterfall_outputs_stay_inside(ctx, width):
    nchan, nblk, n, rate = 9, 2, 4096, 96000
    rng = np.random.default_rng(width)
    raw = rng.integers(-12000, 12000, (nchan, nblk * n * 2)).astype(np.int16)
    adsc = J.AudioDescriptor(rate, blen=n * 4)
    f = J.fft(ctx, None, adsc, max_batch=nchan * nblk, n=n)
    b = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=np.linspace(1000.0, 20000.0, nchan), max_block=nblk * n)
    rows = nchan * nblk
    d_raw = _dev(ctx, raw)
    g_pix, g_peak, g_pk = Guarded(ctx, rows * width * 4), Guarded(ctx, rows * 8), Guarded(ctx, rows * 4)
    J.pump_waterfall_s16(f, b, d_raw.ptr, nblk, width, g_pix.ptr, g_peak.ptr, g_pk.ptr, mem=J.MEM_DEVICE)
    ctx.sync()
    for g, what in ((g_pix, "pixels"), (g_peak, "peak"), (g_pk, "peak bin")):
        g.check(f"waterfall {what} width={width}")
    pix_d, peak_d, pk_d = g_pix.payload(np.int32).copy(), g_peak.payload(np.float32).copy(), g_pk.payload(np.int32).copy()
    b.close()
    b = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=np.linspace(1000.0, 20000.0, nchan), max_block=nblk * n)
    pix = np.zeros((rows, width), dtype=np.int32)
    peak = np.zeros((rows, 2), dtype=np.float32)
    pk = np.zeros(rows, dtype=np.int32)
    J.pump_waterfall_s16(f, b, raw, nblk, width, pix, peak, pk)
    assert np.array_equal(pix_d, pix.ravel()) and np.array_equal(peak_d, peak.ravel()) and np.array_equal(pk_d, pk)
    for g in (g_pix, g_peak, g_pk):
        g.free()
    d_raw.free()
    b.close()
    f.close()


@pytest.mark.parametrize("nchan,S", [(1, 1), (3, 19), (44, 777), (33, 9601)])
def test_bank_outputs_stay_inside_at_ragged_block_lengths(ctx, nchan, S):
    """Block lengths that are not multiples of the decimation (96000 / 9600 = 10), three blocks
    in a row so that filter histories and the fractional output position carry over."""
    rng = np.random.default_rng(S)
    adsc = J.AudioDescriptor(96000, blen=S * 4)
    tuning = np.linspace(-20000.0, 20000.0, nchan) if nchan > 1 else np.array([12000.0])
    bd = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tuning, max_block=S)
    bh = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tuning, max_block=S)
    for blk in range(3):
        raw = rng.integers(-12000, 12000, (nchan, S * 2)).astype(np.int16)
        d_raw = _dev(ctx, raw)
        bd.receive_dev(d_raw.ptr, S, S, s16=True)
        ctx.sync()
        bh.receive_raw(raw, shared=False)
        nds = bd.last_nds()
        assert nds == bh.last_nds()
        g_ds, g_dm = Guarded(ctx, max(nchan * nds * 16, 16)), Guarded(ctx, max(nchan * nds * 16, 16))
        J._ck(J.lib().jsdr_bpsk_read_ds(bd.h, C.c_void_p(g_ds.ptr), J.MEM_DEVICE))
        J._ck(J.lib().jsdr_bpsk_read_dm(bd.h, C.c_void_p(g_dm.ptr), J.MEM_DEVICE))
        ctx.sync()
        g_ds.check(f"ds S={S} block {blk}")
        g_dm.check(f"dm S={S} block {blk}")
        if nds:
            assert np.array_equal(g_ds.payload(np.float64)[:nchan * nds * 2], bh.read_ds().ravel())
            assert np.array_equal(g_dm.payload(np.float64)[:nchan * nds * 2], bh.read_dm().ravel())
        g_ds.free()
        g_dm.free()
        d_raw.free()
    bd.close()
    bh.close()
