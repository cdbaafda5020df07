"""Every FFT / PSD path the dispatcher can pick, held to the binary64 error bound of
tests/fft_accuracy.py on every block: each input format and entry point, batch sizes on both
sides of a CTA's block group and of the resident CTA count, dynamic range, the published peak,
maxima that must not leak from one call into the next, and non-finite input.

The 1e-4-of-full-scale parity bar (tests/test_gpu_parity.py) cannot see one wrong sample at
N >= 16384; the normwise bound here sees it at every length with a margin of 40x or more."""
import numpy as np
import pytest

import fft_accuracy as A
import oracle as O

import jsdrcuda as J

pytestmark = pytest.mark.gpu

RATE = 192000
PLANS = A.plans()                                    # fft_plans.h: N -> (threads, blocks per CTA, radices)
WRAPS = ((9, -9), (-9, 9), (70000, -32768))          # ic / qc that wrap on extreme samples


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def blocks_per_cta(n):
    return PLANS[n][1] if n in PLANS else 1


def plan_smem(n):
    """Plan::SMEM: G blocks of RL rows of ML + PAD float2."""
    _, g, r = PLANS[n]
    rl = r[-1]
    ml = n // rl
    return g * rl * (ml + (2 if ml % 4 == 0 else 4)) * 8


def resident_blocks(n, s16, sms):
    """Blocks in flight when every SM holds as many CTAs as it can: one per SM for the persistent
    plans (s16 input; exact, the persistent grid is min(blocks, SMs)), otherwise what shared memory
    and threads allow.  Registers are not counted, so for the ordinary plans this can overestimate
    the real wave; 2r+1 crosses it either way."""
    if n in A.SPLIT:
        return sms // 2                               # two 16384-point CTAs of 131 KB per block
    t, g, _ = PLANS[n]
    smem = plan_smem(n)
    if s16 and n in A.PERSISTENT:
        return sms
    per_sm = max(1, min((228 * 1024) // (smem + 1024), 2048 // t, 32))
    return sms * per_sm * g


def geometry(n, sms):
    if n in A.FOUR_STEP:
        return [1, 63, 64, 65, 129]                   # 64 blocks per chunk: boundary and both streams
    if n in A.STAGED:
        return [1, 2, 17]
    g = blocks_per_cta(n)
    r = resident_blocks(n, True, sms)
    sizes = {1, g + 1, r - 1, r, r + 1, 2 * r + 1}
    if g > 1:
        sizes.add(g - 1)
    if n in (9600, 16384, 19200):
        sizes.add(700)                                # many blocks per persistent CTA
    return sorted(s for s in sizes if s >= 1)


def noise_s16(n, batch, seed):
    return np.random.default_rng(seed).integers(-32768, 32768, (batch, 2 * n)).astype(np.int16)


def extremes_s16(n, batch, seed):
    """Moderate noise with a sixteenth of the samples at -32768, -32767 or 32767: these are the
    ones an ic / qc correction wraps."""
    rng = np.random.default_rng(seed)
    raw = rng.integers(-8000, 8000, (batch, 2 * n)).astype(np.int16)
    hit = rng.random((batch, 2 * n)) < 1.0 / 16
    raw[hit] = rng.choice(np.array([-32768, -32767, 32767], np.int16), int(hit.sum()))
    return raw


def floats_of(raw):
    return (raw.astype(np.float32) / np.float32(32767.0)).astype(np.float32)


def check_rows(psd, pk, X, s16, what):
    A.check_psd(psd, X, s16, what=what)
    A.check_peak(psd, pk, X, RATE, what=what)


# ------------------------------------------------------------------ formats and entry points
@pytest.mark.parametrize("n", A.LENGTHS)
def test_fft_formats_every_block(ctx, n):
    assert J.lib().jsdr_fft_supported(n) == (2 if n in A.STAGED else 3 if n in A.FOUR_STEP else 1)
    batch = blocks_per_cta(n) + 2
    raw = noise_s16(n, batch, n)
    x = floats_of(raw)
    Xs = A.reference(A.s16_input(raw, n))
    Xf = A.reference(A.f32_input(x, n))
    f = J.fft(ctx, None, J.AudioDescriptor(RATE), max_batch=batch, n=n)
    try:
        A.check_spectrum(f.forward(x), Xf, what="forward f32")
        psd, pk = f.receive_batch(x)
        check_rows(psd, pk, Xf, False, "PSD f32")
        psd, pk = f.receive_batch(raw, s16=True)
        check_rows(psd, pk, Xs, True, "PSD s16")
        ext = extremes_s16(n, batch, n + 1)
        for ic, qc in WRAPS:
            psd, pk = f.receive_batch(ext, s16=True, ic=ic, qc=qc)
            check_rows(psd, pk, A.reference(A.s16_input(ext, n, ic, qc)), True, f"PSD s16 ic={ic} qc={qc}")
        # device-resident buffers (the pump's and the benchmark's entry)
        ic, qc = WRAPS[1]
        d_in = ctx.dev_alloc(x.nbytes)
        d_psd = ctx.dev_alloc(batch * (n + 2) * 4)
        d_pk = ctx.dev_alloc(batch * 4)
        try:
            for s16, src, X in ((True, ext, A.reference(A.s16_input(ext, n, ic, qc))), (False, x, Xf)):
                d_in.upload(src)
                f.receive_dev(d_in, batch, d_psd, d_pk, s16=s16, ic=ic, qc=qc)
                psd = d_psd.download(np.float32, batch * (n + 2)).reshape(batch, n + 2)
                check_rows(psd, d_pk.download(np.int32, batch), X, s16, f"device PSD s16={s16}")
        finally:
            for d in (d_in, d_psd, d_pk):
                d.free()
    finally:
        f.close()


# ------------------------------------------------------------------ batch geometry
@pytest.mark.parametrize("n", A.LENGTHS)
def test_fft_batch_geometry(ctx, sms, n):
    """Batches of 1, G-1, G+1 blocks and around one and two waves of resident CTAs (700 blocks,
    several per persistent CTA, at 9600 / 16384 / 19200); every block of every batch."""
    sizes = geometry(n, sms)
    top = sizes[-1]
    raw = noise_s16(n, top, 7 * n)
    raw[:, 0] = np.arange(top) * 37 % 30000              # neighbours differ at sample 0
    x = floats_of(raw)
    Rs = A.PsdRef(A.reference(A.s16_input(raw, n)), s16=True)
    Xf = A.reference(A.f32_input(x, n))
    Rf = A.PsdRef(Xf, s16=False)
    f = J.fft(ctx, None, J.AudioDescriptor(RATE), max_batch=top, n=n)
    try:
        for b in sizes:
            psd, pk = f.receive_batch(raw[:b], s16=True)
            check_rows(psd, pk, Rs[:b], True, f"PSD s16 batch {b}")
            psd, pk = f.receive_batch(x[:b])
            check_rows(psd, pk, Rf[:b], False, f"PSD f32 batch {b}")
            A.check_spectrum(f.forward(x[:b]), Xf[:b], what=f"forward f32 batch {b}")
    finally:
        f.close()


@pytest.mark.parametrize("n", [4096, 16384, 19200])
def test_fft_pump_every_block(ctx, sms, n):
    """The pump's FFT (jsdr_pump_receive_s16) over nchan x nblocks just beyond the resident CTAs."""
    nblk = 2
    nchan = resident_blocks(n, True, sms) // nblk + 1
    raw = extremes_s16(n, nchan * nblk, n + 5).reshape(nchan, nblk * 2 * n)
    ic, qc = WRAPS[1]
    adsc = J.AudioDescriptor(RATE)
    f = J.fft(ctx, None, adsc, max_batch=nchan * nblk, n=n)
    bank = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=np.linspace(2000.0, 90000.0, nchan), max_block=nblk * n, stages=1)
    try:
        psd = np.empty((nchan * nblk, n + 2), np.float32)
        pk = np.empty(nchan * nblk, np.int32)
        J.pump_receive_s16(f, bank, raw, nblk, psd, pk, ic=ic, qc=qc)
        check_rows(psd, pk, A.reference(A.s16_input(raw, n, ic, qc)), True, "pump")
    finally:
        f.close()
        bank.close()


# ------------------------------------------------------------------ dynamic range and peak
def tone_bins(n):
    """Carrier at bin 0, N/2 (p = -N, and -N * 192000 wraps int32 for N >= 11185), N-1 (p = -2) and
    an odd bin (the second CTA of the split plan); the weak tone a third of the band away."""
    odd = 2 * (n // 3) + 1 if 2 * (n // 3) + 1 < n else 1
    k0 = sorted({0, n // 2, n - 1, odd})
    return k0, [(k + max(1, n // 3)) % n for k in k0]


@pytest.mark.parametrize("n", A.LENGTHS)
def test_fft_dynamic_range_and_peak(ctx, n):
    k0, kw = tone_bins(n)
    nt = len(k0)
    x = np.stack([A.two_tones_f32(n, a, b) for a, b in zip(k0, kw)] + [np.zeros(2 * n, np.float32)])
    x[nt, 0] = 1.0                                       # impulse: every bin exactly 1
    raw = np.stack([A.two_tones_s16(n, a, b) for a, b in zip(k0, kw)] + [np.zeros(2 * n, np.int16)])
    raw[nt, 0] = 32767
    Xf = A.reference(A.f32_input(x, n))
    Xs = A.reference(A.s16_input(raw, n))
    f = J.fft(ctx, None, J.AudioDescriptor(RATE), max_batch=nt + 1, n=n)
    try:
        S = f.forward(x)
        A.check_spectrum(S, Xf, what="forward")
        A.check_dynamic_range(np.abs(S[:nt]).astype(np.float64), Xf[:nt], 1.0, kw, s16=False, psd=False, what="forward")
        for s16, src, X, amp in ((False, x, Xf, 1.0), (True, raw, Xs, 32766.0 / 32767.0)):
            what = f"PSD s16={s16}"
            psd, pk = f.receive_batch(src, s16=s16)
            check_rows(psd, pk, X, s16, what)
            A.check_dynamic_range(A.amplitude(psd[:nt], n), X[:nt], amp, kw, s16=s16, psd=True, what=what)
            assert np.array_equal(pk[:nt], k0), what
            assert pk[nt] == 0 and np.all(psd[nt, :n] == psd[nt, 0]), f"{what}: impulse"
    finally:
        f.close()


@pytest.mark.parametrize("n", A.LENGTHS)
def test_fft_maxima_do_not_leak_between_calls(ctx, n):
    """Back-to-back calls on one handle: large maxima, then smaller ones in a smaller batch, then
    a batch of one.  Each call publishes its own peaks (the split plan's best / cnt and the
    four-step's d_best are per launch)."""
    f = J.fft(ctx, None, J.AudioDescriptor(RATE), max_batch=5, n=n)
    t = np.arange(n)
    try:
        for s16 in (False, True):
            for call, (batch, amp) in enumerate(((5, 0.9), (3, 0.05), (1, 0.002))):
                bins = (np.arange(batch) * 7 + 3 * call + 1) % n
                z = amp * np.exp(2j * np.pi * ((bins[:, None] * t[None, :]) % n) / n)
                if s16:
                    src = np.empty((batch, 2 * n), np.int16)
                    src[:, 0::2], src[:, 1::2] = np.rint(32767 * z.real), np.rint(32767 * z.imag)
                    X = A.reference(A.s16_input(src, n))
                else:
                    src = z.astype(np.complex64).view(np.float32)
                    X = A.reference(A.f32_input(src, n))
                psd, pk = f.receive_batch(src, s16=s16)
                check_rows(psd, pk, X, s16, f"s16={s16} call {call}")
                assert np.array_equal(pk, bins), f"s16={s16} call {call}"
    finally:
        f.close()


# ------------------------------------------------------------------ non-finite input
@pytest.mark.parametrize("n", A.MULTI_BLOCK + [16384])
def test_fft_nonfinite_block(ctx, n):
    """One block with NaN and +-inf inside a multi-block CTA (and in a batch of the 16384 float
    path): the other blocks are bit-identical to a run without it; its row is all NaN, and its
    published peak follows the strict '>' of fft.java:208-211 (NaN never wins), as the oracle's."""
    g = blocks_per_cta(n)
    batch, bad = 2 * g + 3, g + 1
    rng = np.random.default_rng(n)
    x = rng.uniform(-1, 1, (batch, 2 * n)).astype(np.float32)
    y = x.copy()
    y[bad, 10], y[bad, 21], y[bad, 2 * n - 1] = np.nan, np.inf, -np.inf
    f = J.fft(ctx, None, J.AudioDescriptor(RATE), max_batch=batch, n=n)
    try:
        p0, k0 = f.receive_batch(x)
        p1, k1 = f.receive_batch(y)
    finally:
        f.close()
    keep = np.arange(batch) != bad
    assert np.array_equal(p1[keep].view(np.uint32), p0[keep].view(np.uint32)) and np.array_equal(k1[keep], k0[keep])
    assert np.all(np.isnan(p1[bad, :n]))
    o, opk = O.fft_receive(y[bad], RATE)
    assert np.all(np.isnan(o[:n]))
    assert p1[bad, n] == o[n] and p1[bad, n + 1] == o[n + 1] and k1[bad] == opk == -1
