"""Out of device memory in a create or in a lazily allocated workspace: the call answers
JSDR_ENOMEM with a message naming it, the handle (if any) still destroys, nothing leaks, and the
context goes on computing exactly what it computed before.

Each case asks for one allocation larger than the whole device, behind a few small ones, so the
test never holds memory that other work on the same GPU needs: a case is skipped unless its
failing request exceeds the device's total memory, and what it allocates before that request is
held under 64 MB.  (A four-step or split-plan FFT has no such case: its block maxima take 8 bytes
per max_batch up front, 17 GB at max_batch 2^31 - 1, which would succeed.)"""
import ctypes as C

import numpy as np
import pytest

import jsdrcuda as J

pytestmark = pytest.mark.gpu

ENOMEM = -3
BIG = 2**31 - 1          # max_block_samples / max_batch
NCHAN = 65535            # the most channels a bank or a demod takes
ROUNDS = 20


def free_bytes():
    import torch
    torch.cuda.synchronize()
    return torch.cuda.mem_get_info(0)[0]


def device_total():
    import torch
    return torch.cuda.mem_get_info(0)[1]


def needs_more_than_the_device(failing, before):
    if failing <= device_total():
        pytest.skip(f"the failing request ({failing} bytes) would fit this device")
    assert before < (64 << 20), f"{before} bytes allocated ahead of the failing request"


def last_error():
    return J.lib().jsdr_last_error().decode("utf-8", "replace")


def ordinary(ctx):
    """One ordinary handle of each kind on `ctx`, and what it computes."""
    rng = np.random.default_rng(11)
    adsc = J.AudioDescriptor(96000, blen=4 * 4096)
    iq = rng.uniform(-1, 1, (2, 2 * 1000)).astype(np.float32)
    f = J.fft(ctx, None, adsc, max_batch=2, n=1000)
    psd, pk = f.receive_batch(iq)
    f.close()
    raw = rng.integers(-9000, 9000, (3, 2 * 4096)).astype(np.int16)
    b = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=[12000.0, -7000.0, 30000.0], max_block=4096)
    b.receive_raw(raw, shared=False)
    ds = b.read_ds().copy()
    bits = b.read_bits()
    b.close()
    d = J.demod(ctx, adsc, nchan=2, max_block=4096)
    d.weights(3000, 6000)
    d.weights(3000, 6000, chan=1)
    out = d.receive(rng.uniform(-1, 1, (2, 2 * 4096)).astype(np.float32))
    d.close()
    return psd.copy(), pk.copy(), ds, bits, out.copy()


def same(a, b):
    if isinstance(a, (tuple, list)):
        return len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
    return np.array_equal(np.asarray(a), np.asarray(b))


def rounds(ctx, one):
    """`one` once to warm up, then ROUNDS times: the device's free memory ends where it started,
    and the context still computes what it computed before."""
    ref = ordinary(ctx)
    one()
    before = free_bytes()
    for _ in range(ROUNDS):
        one()
    after = free_bytes()
    assert before - after < (8 << 20), f"{(before - after) >> 20} MiB not returned after {ROUNDS} failures"
    assert same(ordinary(ctx), ref), "the context computes something else after the failures"


def test_bpsk_create_out_of_memory(ctx):
    rate = 192000
    nc = NCHAN
    max_words = (BIG + 31) // 32 + 1
    # nine small buffers (taps, matched filter, two sin/cos tables, four per-channel tuner
    # arrays of 8 bytes and one of 32), then the first plan's phase checkpoints
    needs_more_than_the_device(8 * nc * max_words, 8 * 128 + 8 * 65 + 8 * 512 + 16 * 257 + nc * (4 * 8 + 32))
    tuning = np.linspace(1000.0, 90000.0, nc)

    def one():
        h = C.c_void_p()
        rc = J.lib().jsdr_bpsk_create(ctx.h, rate, nc, tuning.ctypes.data_as(C.c_void_p), BIG, C.byref(h))
        assert rc == ENOMEM, (rc, last_error())
        assert "jsdr_bpsk_create" in last_error()
        assert not h.value
        assert J.lib().jsdr_bpsk_destroy(h) == 0

    rounds(ctx, one)


def test_demod_create_out_of_memory(ctx):
    nc = NCHAN
    max_chunks = (BIG + 31) // 32 + 1
    # taps, phi and car, then the chunk-carry checkpoints
    needs_more_than_the_device(4 * nc * max_chunks, 4 * 21 * nc + 4 * nc + 4 * nc)

    def one():
        h = C.c_void_p()
        rc = J.lib().jsdr_demod_create(ctx.h, 96000, nc, BIG, C.byref(h))
        assert rc == ENOMEM, (rc, last_error())
        assert "jsdr_demod_create" in last_error()
        assert not h.value
        assert J.lib().jsdr_demod_destroy(h) == 0

    rounds(ctx, one)


def test_fft_staged_workspace_out_of_memory(ctx):
    n = 1000                                         # no single-CTA plan: the staged path
    assert J.lib().jsdr_fft_supported(n) == 2
    # device pointers: the host path would first stage a 4-byte peak per max_batch (8.6 GB)
    needs_more_than_the_device(8 * n * BIG, 8 * n)
    d_in = ctx.dev_alloc(8 * n)
    d_psd = ctx.dev_alloc(4 * (n + 2))
    d_in.upload(np.random.default_rng(5).uniform(-1, 1, 2 * n).astype(np.float32))

    def one():
        h = C.c_void_p()
        assert J.lib().jsdr_fft_create(ctx.h, n, 96000, BIG, C.byref(h)) == 0, last_error()
        for _ in range(2):                           # a failed workspace is not half there on the retry
            rc = J.lib().jsdr_fft_receive_f32(h, C.c_void_p(d_in.ptr), 1, C.c_void_p(d_psd.ptr), None, J.MEM_DEVICE)
            assert rc == ENOMEM, (rc, last_error())
            assert "fft workspace" in last_error()
        assert J.lib().jsdr_fft_destroy(h) == 0

    try:
        rounds(ctx, one)
    finally:
        d_in.free()
        d_psd.free()
