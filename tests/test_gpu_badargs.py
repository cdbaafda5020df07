"""Bad arguments on live handles: every call below must come back as a negative status with a
message — never a crash, a hang or a CUDA error left pending — and afterwards the same handles
must still produce exactly what they produced before (nothing throws through
IAudioHandler.receive, JavaAudio.java:321-323)."""
import ctypes as C

import numpy as np
import pytest

import jsdrcuda as J

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(300)]


ACCEPTED = []


def refused(fn, *args):
    rc = fn(*args)
    if rc >= 0:
        ACCEPTED.append((fn.__name__, [a.value if hasattr(a, "value") else a for a in args][1:], rc))
    else:
        assert J.lib().jsdr_last_error(), fn.__name__
    return rc


def p(a):
    return a.ctypes.data_as(C.c_void_p)


def test_bad_arguments_on_live_handles(ctx):
    L = J.lib()
    rng = np.random.default_rng(3)
    n, rate = 1024, 96000
    adsc = J.AudioDescriptor(rate, blen=4 * 2 * n)
    f = J.fft(ctx, None, adsc, max_batch=4, n=n)
    b = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=[12000.0, -7000.0, 30000.0], max_block=2 * n)
    d = J.demod(ctx, adsc, nchan=2, max_block=2 * n)
    r = J.fir(ctx, float(rate), nchan=2, max_block=2 * n)
    d.weights(3000, 6000)
    d.weights(3000, 6000, chan=1)
    r.weights(1000, 2000)
    iq = rng.uniform(-1, 1, (4, 2 * n)).astype(np.float32)
    raw = rng.integers(-9000, 9000, (3, 4 * n)).astype(np.int16)
    xi = rng.integers(-1000, 1000, (2, n)).astype(np.int32)

    def good():
        b2 = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=[12000.0, -7000.0, 30000.0], max_block=2 * n)
        psd = np.zeros((6, n + 2), np.float32)
        J.pump_receive_s16(f, b2, raw, 2, psd) if f.max_batch >= 6 else None
        out = (f.receive_batch(iq)[0].copy(), b2.receive_raw(raw, shared=False), b2.read_ds().copy(),
               J.demod(ctx, adsc, nchan=1, max_block=n).receive(iq[0])[0].copy(), r.complex_mod(xi.reshape(-1, 2), xi.reshape(-1, 2)))
        b2.close()
        return out

    before = good()
    psd = np.zeros((4, n + 2), np.float32)
    pk = np.zeros(4, np.int32)
    # ---- fft
    refused(L.jsdr_fft_receive_f32, f.h, None, 1, p(psd), p(pk), 0)
    refused(L.jsdr_fft_receive_f32, f.h, p(iq), 1, None, p(pk), 0)
    assert L.jsdr_fft_receive_f32(f.h, p(iq), 0, p(psd), p(pk), 0) == 0          # an empty batch is a no-op
    for batch in (-1, 5, 2**31 - 1):
        refused(L.jsdr_fft_receive_f32, f.h, p(iq), batch, p(psd), p(pk), 0)
        refused(L.jsdr_fft_receive_s16, f.h, p(raw), batch, 0, 0, p(psd), p(pk), 0)
        refused(L.jsdr_fft_forward_f32, f.h, p(iq), batch, p(psd), 0)
    for mem in (-1, 2, 7):
        refused(L.jsdr_fft_receive_f32, f.h, p(iq), 1, p(psd), p(pk), mem)
        refused(L.jsdr_bpsk_receive_f32, b.h, p(iq), n, 0, mem)
        refused(L.jsdr_demod_receive_f32, d.h, p(iq), n, 0, p(psd), mem)
    fh = C.c_void_p()
    for bad_n in (0, 1, -4096, 11 * 1024):
        refused(L.jsdr_fft_create, ctx.h, bad_n, rate, 1, C.byref(fh))
    refused(L.jsdr_fft_create, ctx.h, n, 0, 1, C.byref(fh))
    refused(L.jsdr_fft_create, ctx.h, n, rate, 0, C.byref(fh))
    # ---- tuner bank
    refused(L.jsdr_bpsk_receive_f32, b.h, None, n, 0, 0)
    for ns in (-1, 2 * n + 1, 2**31 - 1):
        refused(L.jsdr_bpsk_receive_f32, b.h, p(iq), ns, 0, 0)
        refused(L.jsdr_bpsk_receive_s16, b.h, p(raw), ns, 0, 0, 0, 0)
    refused(L.jsdr_bpsk_receive_f32, b.h, p(iq), n, -5, 0)
    for chan in (-1, 3, 2**31 - 1):
        refused(L.jsdr_bpsk_set_tuning, b.h, chan, C.c_double(1000.0))
    for hz in (float("nan"), float("inf"), -float("inf")):
        refused(L.jsdr_bpsk_set_tuning, b.h, 0, C.c_double(hz))
    bh = C.c_void_p()
    tun = np.array([1000.0, float("nan")])
    refused(L.jsdr_bpsk_create, ctx.h, rate, 2, p(tun), n, C.byref(bh))
    tun[1] = 2000.0
    for args in ((9599, 2, n), (rate, 0, n), (rate, 65536, n), (rate, 2, 0), (rate, 2, -1)):
        refused(L.jsdr_bpsk_create, ctx.h, args[0], args[1], p(tun), args[2], C.byref(bh))
    for st in (0, 4, -1):
        refused(L.jsdr_bpsk_set_stages, b.h, st)
    refused(L.jsdr_bpsk_set_precision, b.h, 2)
    for mode in (3, 9):
        refused(L.jsdr_bpsk_set_kernel, b.h, mode)
    taps = np.ones(200)
    for nt in (0, -1, 129):
        refused(L.jsdr_bpsk_set_ds_filter, b.h, p(taps), nt)
    refused(L.jsdr_bpsk_set_ds_filter, b.h, None, 27)
    refused(L.jsdr_bpsk_enable_fec, b.h, None, 4)
    refused(L.jsdr_bpsk_enable_fec, b.h, p(np.zeros(512, np.int16)), 0)
    refused(L.jsdr_bpsk_read_frames, b.h, None, None, None, None, None, 4)
    bits, at, nb = np.zeros((3, 8), np.int8), np.zeros((3, 8), np.int64), np.zeros(3, np.int32)
    refused(L.jsdr_bpsk_read_bits, b.h, None, p(at), p(nb), 8, 0)
    for mb in (0, -1):
        refused(L.jsdr_bpsk_read_bits, b.h, p(bits), p(at), p(nb), mb, 0)
    refused(L.jsdr_bpsk_read_ds, b.h, None, 0)
    refused(L.jsdr_bpsk_read_counters, b.h, None)
    # ---- demod / fir / waterfall
    for chan in (-1, 2):
        refused(L.jsdr_demod_weights, d.h, chan, 1000, 2000)
        refused(L.jsdr_fir_set_weights, r.h, chan, p(np.zeros(21)))
    for mode in (-1, 5):
        refused(L.jsdr_demod_set_mode, d.h, mode, 0)
    out = np.zeros((2, 4 * n), np.float32)
    refused(L.jsdr_demod_receive_f32, d.h, None, n, 0, p(out), 0)
    refused(L.jsdr_demod_receive_f32, d.h, p(iq), n, 0, None, 0)
    for ns in (-1, 2 * n + 1):
        refused(L.jsdr_demod_receive_f32, d.h, p(iq), ns, 0, p(out), 0)
        refused(L.jsdr_fir_filter_i32, r.h, p(xi), ns, 0, p(np.zeros((2, 2 * n + 1), np.int32)), 0)
    refused(L.jsdr_fir_filter_i32, r.h, None, n, 0, p(xi), 0)
    refused(L.jsdr_fir_complex_mod_i32, ctx.h, p(xi), p(xi), p(xi), -1, 0)
    pix = np.zeros((4, n), np.int32)
    assert L.jsdr_waterfall_rows(ctx.h, p(psd), n, 0, 10, 0xffff, p(pix), 0) == 0   # no rows: a no-op
    for rows, width in ((-1, 10), (4, 0), (4, -1), (4, n + 1)):
        refused(L.jsdr_waterfall_rows, ctx.h, p(psd), n, rows, width, 0xffff, p(pix), 0)
    refused(L.jsdr_waterfall_rows, ctx.h, p(psd), 0, 4, 10, 0xffff, p(pix), 0)
    # ---- pump
    big = np.zeros((12, n + 2), np.float32)
    for nblk in (0, -1, 3, 2**31 - 1):
        refused(L.jsdr_pump_receive_s16, f.h, b.h, p(raw), nblk, 0, 0, p(big), None, 0)
    refused(L.jsdr_pump_receive_s16, f.h, b.h, p(raw), 2, 0, 0, p(big), None, 0)      # 3 ch x 2 blocks > max_batch 4
    refused(L.jsdr_pump_receive_s16, f.h, b.h, None, 1, 0, 0, p(big), None, 0)
    refused(L.jsdr_pump_waterfall_s16, f.h, b.h, p(raw), 1, 0, 0, 0, 0xffff, p(pix), p(psd), None, 0)
    d3 = J.demod(ctx, adsc, nchan=3, max_block=2 * n)
    audio = np.zeros((3, n), np.int16)
    for mem in (-1, 2):                  # every other argument is valid: only mem is refused
        refused(L.jsdr_pump_receive_s16, f.h, b.h, p(raw), 1, 0, 0, p(big), None, mem)
        refused(L.jsdr_pump_waterfall_s16, f.h, b.h, p(raw), 1, 0, 0, 16, 0xffff, p(pix), p(psd), None, mem)
        refused(L.jsdr_pump_demod_s16, f.h, b.h, d3.h, p(raw), 1, 0, 0, p(big), None, p(audio), None, mem)
    d3.close()
    # ---- memory and context
    q = C.c_void_p()
    refused(L.jsdr_dev_alloc, ctx.h, 1 << 50, C.byref(q))
    refused(L.jsdr_host_alloc, ctx.h, 1 << 50, C.byref(q))
    refused(L.jsdr_memcpy_h2d, ctx.h, None, p(iq), 16)
    refused(L.jsdr_ctx_profile_read, ctx.h, p(np.zeros(3)), p(np.zeros(3, np.int64)), 3)
    ch = C.c_void_p()
    refused(L.jsdr_ctx_create, 10**6, C.byref(ch))
    refused(L.jsdr_ctx_create, -1, C.byref(ch))
    assert not ACCEPTED, "\n".join(map(str, ACCEPTED))
    # ---- nothing is left pending, and everything still works bit for bit
    ctx.sync()
    after = good()
    for x, y in zip(before, after):
        if x is not None:
            assert np.array_equal(x, y)
    for h in (f, b, d, r):
        h.close()


def test_profiling_left_on_and_never_read_is_bounded(ctx):
    """Switch per-kernel timing on, launch 70 000 kernels without ever reading: at most 65 536
    spans (event pairs) are kept, the rest simply is not timed, results are unaffected and the
    next read starts afresh."""
    n = 128
    f = J.fft(ctx, None, J.AudioDescriptor(44100, blen=4 * n), max_batch=1, n=n)
    d_in, d_psd = ctx.dev_alloc(8 * n), ctx.dev_alloc(4 * (n + 2))
    x = np.random.default_rng(0).uniform(-1, 1, 2 * n).astype(np.float32)
    d_in.upload(x)
    want = f.receive(x).copy()
    ctx.profile(True)
    for _ in range(70000):
        f.receive_dev(d_in.ptr, 1, d_psd.ptr, None, s16=False)
    prof = ctx.profile_read()
    total = sum(int(v[1]) for v in prof.values()) if isinstance(next(iter(prof.values())), (tuple, list)) else None
    L = J.lib()
    ms, cnt = np.zeros(12), np.zeros(12, np.int64)
    f.receive_dev(d_in.ptr, 1, d_psd.ptr, None, s16=False)
    assert L.jsdr_ctx_profile_read(ctx.h, p(ms), p(cnt), 12) == 0
    assert cnt.sum() == 1 and cnt[0] == 1                     # afresh: exactly the one launch since the read
    if total is not None:
        assert total == 65536, total
    ctx.profile(False)
    assert np.array_equal(d_psd.download(np.float32, n + 2), want)
    d_in.free()
    d_psd.free()
    f.close()
