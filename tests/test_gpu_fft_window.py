"""The fft handle's optional window (jsdr_fft_set_window) on every path the dispatcher can pick:
every block of every batch within the binary64 bound B(N) of tests/fft_accuracy.py, taken of the
exactly rebuilt windowed input (tests/fft_window.py); an all-ones window and a removed window are
bitwise the unwindowed handle; a window change is ordered with the work already enqueued; the
reference's sine fixtures under fft.java's Hamming table; the three pumps, whose bank and demod
handler must not see the window; and the refusals."""
import numpy as np
import pytest

import fft_accuracy as A
import fft_window as W
import test_gpu_fft_accuracy as G
from conftest import load_s16

import jsdrcuda as J

pytestmark = pytest.mark.gpu

RATE = G.RATE
EINVAL = -1


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def check_rows(psd, pk, X, s16, what):
    A.check_psd(psd, X, s16, what=what)
    A.check_peak(psd, pk, X, RATE, what=what)


def forward_dev(f, d_in, batch, d_out):
    J._ck(J.lib().jsdr_fft_forward_f32(f.h, J._ptr(d_in), batch, J._ptr(d_out), J.MEM_DEVICE))


def bits_of(psd):
    return np.ascontiguousarray(psd).view(np.uint32)


# ------------------------------------------------------------------ every block, every path
@pytest.mark.parametrize("n", A.LENGTHS)
def test_window_every_block(ctx, sms, n):
    """s16 (with wrapping ic / qc) and f32, host and device memory, PSD and forward spectra, over
    the batch sizes of test_fft_batch_geometry (both sides of a CTA's block group and of the
    resident CTAs); every block within B(N) of the windowed input and every peak its own."""
    sizes = G.geometry(n, sms)
    top = sizes[-1]
    win = W.random_window(n, n)
    raw = G.noise_s16(n, top, 11 * n)
    raw[:, 0] = np.arange(top) * 37 % 30000                    # neighbours differ at sample 0
    x = G.floats_of(raw)
    Rs = A.PsdRef(A.reference(W.s16_input(raw, n, win)), s16=True)
    Xf = A.reference(W.f32_input(x, n, win))
    Rf = A.PsdRef(Xf, s16=False)
    f = J.fft(ctx, None, J.AudioDescriptor(RATE), max_batch=top, n=n)
    f.set_window(win)
    bufs = []
    try:
        for b in sizes:
            psd, pk = f.receive_batch(raw[:b], s16=True)
            check_rows(psd, pk, Rs[:b], True, f"windowed PSD s16 batch {b}")
            psd, pk = f.receive_batch(x[:b])
            check_rows(psd, pk, Rf[:b], False, f"windowed PSD f32 batch {b}")
            A.check_spectrum(f.forward(x[:b]), Xf[:b], what=f"windowed forward f32 batch {b}")
        ext = G.extremes_s16(n, top, n + 1)
        for ic, qc in G.WRAPS:
            psd, pk = f.receive_batch(ext, s16=True, ic=ic, qc=qc)
            check_rows(psd, pk, A.reference(W.s16_input(ext, n, win, ic, qc)), True, f"windowed PSD s16 ic={ic} qc={qc}")
        # device-resident buffers (the pump's and the benchmark's entry)
        ic, qc = G.WRAPS[1]
        d_in, d_psd, d_pk, d_spec = bufs = [ctx.dev_alloc(x.nbytes), ctx.dev_alloc(top * (n + 2) * 4),
                                            ctx.dev_alloc(top * 4), ctx.dev_alloc(x.nbytes)]
        for s16, src, X in ((True, ext, A.reference(W.s16_input(ext, n, win, ic, qc))), (False, x, Rf)):
            d_in.upload(src)
            f.receive_dev(d_in, top, d_psd, d_pk, s16=s16, ic=ic, qc=qc)
            psd = d_psd.download(np.float32, top * (n + 2)).reshape(top, n + 2)
            check_rows(psd, d_pk.download(np.int32, top), X, s16, f"windowed device PSD s16={s16}")
        forward_dev(f, d_in, top, d_spec)
        A.check_spectrum(d_spec.download(np.complex64, top * n).reshape(top, n), Xf, what="windowed device forward f32")
    finally:
        for d in bufs:
            d.free()
        f.close()


@pytest.mark.parametrize("n", A.LENGTHS)
def test_all_ones_and_removed_window_are_bitwise_unwindowed(ctx, n):
    """x * 1.0f is x: an all-ones window publishes the unwindowed handle's PSD, peaks and spectra
    bit for bit on every path; set_window(None) after a real window does the same."""
    batch = 2 * G.blocks_per_cta(n) + 3
    raw = G.extremes_s16(n, batch, n + 7)
    x = G.floats_of(G.noise_s16(n, batch, n + 8))
    ic, qc = G.WRAPS[2]
    adsc = J.AudioDescriptor(RATE)
    plain = J.fft(ctx, None, adsc, max_batch=batch, n=n)
    f = J.fft(ctx, None, adsc, max_batch=batch, n=n)

    def outputs(h):
        ps, ks = h.receive_batch(raw, s16=True, ic=ic, qc=qc)
        pf, kf = h.receive_batch(x)
        return bits_of(ps), ks, bits_of(pf), kf, h.forward(x).view(np.uint32)

    try:
        want = outputs(plain)
        f.set_window(np.ones(n, np.float32))
        for k, (got, ref) in enumerate(zip(outputs(f), want)):
            assert np.array_equal(got, ref), f"all-ones window: output {k} differs from the unwindowed handle"
        f.set_window(W.random_window(n, n))
        assert not np.array_equal(outputs(f)[0], want[0])
        f.set_window(None)
        for k, (got, ref) in enumerate(zip(outputs(f), want)):
            assert np.array_equal(got, ref), f"removed window: output {k} differs from the unwindowed handle"
    finally:
        plain.close()
        f.close()


# ------------------------------------------------------------------ ordering
@pytest.mark.parametrize("n", [4096, 16384, 19200, 32768, 65536, 1000])
def test_window_change_is_stream_ordered(ctx, n):
    """Device receive under window A, set_window(B), device receive, then one sync: the first
    result is A's and the second B's, bit for bit as host calls under each window give them
    (the last blocks are the ones still in flight when the window changes)."""
    batch = max(8, (1 << 25) // n)
    tail = 4
    rng = np.random.default_rng(n)
    tile = rng.integers(-20000, 20000, (64, 2 * n)).astype(np.int16)
    a, b = W.random_window(n, 1), W.random_window(n, 2)
    f = J.fft(ctx, None, J.AudioDescriptor(RATE), max_batch=batch, n=n)
    d_in = ctx.dev_alloc(batch * n * 4)
    d_psd = [ctx.dev_alloc(batch * (n + 2) * 4) for _ in range(2)]
    d_pk = [ctx.dev_alloc(batch * 4) for _ in range(2)]
    try:
        for b0 in range(0, batch, 64):
            d_in.upload(tile[: min(64, batch - b0)], offset=b0 * n * 4)
        last = tile[[(batch - tail + i) % 64 for i in range(tail)]]
        f.set_window(a)
        ctx.sync()
        f.receive_dev(d_in, batch, d_psd[0], d_pk[0])
        f.set_window(b)
        f.receive_dev(d_in, batch, d_psd[1], d_pk[1])
        ctx.sync()
        got = [d.download(np.float32, tail * (n + 2), offset=(batch - tail) * (n + 2) * 4).reshape(tail, n + 2) for d in d_psd]
        pks = [d.download(np.int32, tail, offset=(batch - tail) * 4) for d in d_pk]
        for k, win in enumerate((a, b)):
            f.set_window(win)
            psd, pk = f.receive_batch(last, s16=True)
            assert np.array_equal(bits_of(got[k]), bits_of(psd)) and np.array_equal(pks[k], pk), f"call {k} under window {'AB'[k]}"
            check_rows(got[k], pks[k], A.reference(W.s16_input(last, n, win)), True, f"call {k}")
    finally:
        for d in [d_in] + d_psd + d_pk:
            d.free()
        f.close()


# ------------------------------------------------------------------ the reference's fixtures
@pytest.mark.parametrize("name,n,tone,mirror", [("sine4410.raw", 4096, 410, 3686), ("sine4410-short.raw", 128, 13, 115)])
def test_hamming_on_the_reference_fixtures(ctx, name, n, tone, mirror):
    """fft.java's Hamming table on the 4410 Hz fixtures at 44100 S/s: within the bound, the peak
    on the tone or its near-tied mirror (SURVEY Q3), and the leakage 20 bins away below the
    unwindowed spectrum's."""
    raw = load_s16(name)
    assert raw.size == 2 * n
    win = W.hamming(n)
    x = G.floats_of(raw).reshape(1, 2 * n)
    adsc = J.AudioDescriptor(44100, blen=4 * n)
    plain = J.fft(ctx, None, adsc)
    f = J.fft(ctx, None, adsc)
    f.set_window(win)
    try:
        for s16 in (True, False):
            src = raw.reshape(1, 2 * n) if s16 else x
            X = A.reference(W.s16_input(src, n, win) if s16 else W.f32_input(src, n, win))
            psd, pk = f.receive_batch(src, s16=s16)
            A.check_psd(psd, X, s16, what=f"{name} s16={s16}")
            A.check_peak(psd, pk, X, 44100, what=f"{name} s16={s16}")
            assert pk[0] in (tone, mirror), f"{name} s16={s16}: peak bin {pk[0]}"
            p0, _ = plain.receive_batch(src, s16=s16)
            far = [k % n for k in (tone + 20, tone - 20, mirror + 20, mirror - 20)
                   if min(abs(k - tone), abs(k - mirror), abs(k - tone - n), abs(k - mirror + n)) >= 20]
            assert far and np.all(psd[0, far] < p0[0, far]), (name, s16, far, psd[0, far], p0[0, far])
    finally:
        plain.close()
        f.close()


# ------------------------------------------------------------------ the pumps
@pytest.mark.parametrize("n", [4096, 19200])
def test_pumps_window_only_the_spectrum(ctx, n):
    """jsdr_pump_receive_s16, _waterfall_s16 and _demod_s16 on a windowed fft handle: PSD, pixel
    rows and peaks are the windowed ones (within the bound), while the bank's decimated rows and
    bits and the demod's audio equal, bit for bit, the same calls with an unwindowed handle."""
    nchan, nblk, width = 3, 2, 700
    ic, qc = G.WRAPS[1]
    raw = G.extremes_s16(n, nchan * nblk, n + 3).reshape(nchan, nblk * 2 * n)
    win = W.random_window(n, n + 3)
    X = A.PsdRef(A.reference(W.s16_input(raw.reshape(nchan * nblk, 2 * n), n, win, ic, qc)), s16=True)
    adsc = J.AudioDescriptor(RATE)

    def handles(windowed):
        f = J.fft(ctx, None, adsc, max_batch=nchan * nblk, n=n)
        if windowed:
            f.set_window(win)
        b = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=np.linspace(5000.0, 60000.0, nchan), max_block=nblk * n, stages=3)
        d = J.demod(ctx, adsc, nchan=nchan, max_block=nblk * n)
        for c in range(nchan):
            d.weights(3000, 9000, chan=c)
        d.set_mode(J.demod.MODE_NFM, True)
        return f, b, d

    def run(f, b, d):
        out = {}
        psd = np.empty((nchan * nblk, n + 2), np.float32)
        pk = np.empty(nchan * nblk, np.int32)
        J.pump_receive_s16(f, b, raw, nblk, psd, pk, ic=ic, qc=qc)
        out["receive"] = (psd, pk, b.read_ds(), b.read_bits()[0])
        pix = np.empty((nchan * nblk, width), np.int32)
        peak = np.empty((nchan * nblk, 2), np.float32)
        pk2 = np.empty(nchan * nblk, np.int32)
        J.pump_waterfall_s16(f, b, raw, nblk, width, pix, peak, pk2, ic=ic, qc=qc)
        out["waterfall"] = (pix, peak, pk2, b.read_ds(), b.read_bits()[0])
        psd3 = np.empty_like(psd)
        pk3 = np.empty_like(pk)
        aud = np.empty((nchan, nblk * n), np.int16)
        ma = np.empty((nchan, nblk, 2), np.float32)
        J.pump_demod_s16(f, b, d, raw, nblk, psd3, aud, ma, pk3, ic=ic, qc=qc)
        out["demod"] = (psd3, pk3, aud, ma, b.read_ds(), b.read_bits()[0])
        return out

    hw, h0 = handles(True), handles(False)
    try:
        w, u = run(*hw), run(*h0)
    finally:
        for h in hw + h0:
            h.close()
    psd, pk, ds, bits = w["receive"]
    check_rows(psd, pk, X, True, "pump_receive_s16")
    assert not np.array_equal(psd, u["receive"][0]), "the pump's PSD is not windowed"
    pix, peak, pk2, ds2, bits2 = w["waterfall"]
    assert np.array_equal(pix, J.waterfall_rows(ctx, psd, width)), "pixel rows are not those of the windowed PSD"
    assert np.array_equal(bits_of(peak), bits_of(psd[:, n:])) and np.array_equal(pk2, pk)
    psd3, pk3, aud, ma, ds3, bits3 = w["demod"]
    assert np.array_equal(bits_of(psd3), bits_of(psd)) and np.array_equal(pk3, pk)
    # the handlers beside the fft see unwindowed samples
    for (leg, i) in (("receive", 2), ("waterfall", 3), ("demod", 4)):
        assert np.array_equal(w[leg][i].view(np.uint64), u[leg][i].view(np.uint64)), f"{leg}: decimated rows differ"
        assert all(np.array_equal(p, q) for p, q in zip(w[leg][i + 1], u[leg][i + 1])), f"{leg}: bits differ"
    assert np.array_equal(aud, u["demod"][2]) and np.array_equal(bits_of(ma), bits_of(u["demod"][3])), "demod audio differs"


# ------------------------------------------------------------------ refusals and leaks
def test_nonfinite_window_is_refused_and_the_old_one_stays(ctx):
    n, batch = 4096, 5
    raw = G.noise_s16(n, batch, 3)
    win = W.random_window(n, 3)
    f = J.fft(ctx, None, J.AudioDescriptor(RATE), max_batch=batch, n=n)
    plain = J.fft(ctx, None, J.AudioDescriptor(RATE), max_batch=batch, n=n)
    try:
        p_plain, _ = plain.receive_batch(raw, s16=True)
        for bad in (np.nan, np.inf, -np.inf):                  # no window in force: none stays
            w = win.copy()
            w[[77, 200]] = bad
            with pytest.raises(J.JsdrError) as e:
                f.set_window(w)
            assert e.value.code == EINVAL and "win[77]" in str(e.value), str(e.value)
            assert np.array_equal(bits_of(f.receive_batch(raw, s16=True)[0]), bits_of(p_plain))
        f.set_window(win)
        want, _ = f.receive_batch(raw, s16=True)
        for bad in (np.nan, np.inf, -np.inf):
            w = W.random_window(n, 4)
            w[n - 1] = bad
            with pytest.raises(J.JsdrError) as e:
                f.set_window(w)
            assert e.value.code == EINVAL and f"win[{n - 1}]" in str(e.value), str(e.value)
            assert np.array_equal(bits_of(f.receive_batch(raw, s16=True)[0]), bits_of(want)), "the old window is gone"
        with pytest.raises(ValueError):
            f.set_window(win[:-1])
    finally:
        f.close()
        plain.close()


def test_windowed_handles_return_their_device_memory(ctx):
    import torch

    def free_bytes():
        torch.cuda.synchronize()
        return torch.cuda.mem_get_info(0)[0]

    rng = np.random.default_rng(6)

    def one_round(k):
        n = [4096, 19200, 65536, 32768, 1000][k % 5]
        f = J.fft(ctx, None, J.AudioDescriptor(RATE), max_batch=3, n=n)
        f.set_window(W.random_window(n, k))
        f.receive_batch(rng.integers(-9000, 9000, (3, 2 * n)).astype(np.int16), s16=True)
        f.set_window(None)
        f.set_window(W.hamming(n))
        f.forward(rng.uniform(-1, 1, (3, 2 * n)).astype(np.float32))
        f.close()

    for k in range(5):
        one_round(k)
    before = free_bytes()
    for k in range(40):
        one_round(k)
    after = free_bytes()
    assert before - after < (8 << 20), f"{(before - after) >> 20} MiB of device memory not returned after 40 rounds"
