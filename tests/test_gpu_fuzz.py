"""Seeded differential runs of the tuner bank against the oracle (FUNcubeBPSKDemod.java:366-595).

Each seed draws a whole scenario — rate, number of tuners (both sides of the 32-channel switch
between the tile kernel and the streaming kernel), per-channel streams or one shared stream,
s16 or float blocks, a sequence of ragged block lengths (including 0 and 1), tunings of either
sign, retunes between blocks, the kernel mode — and every output of every block of a few
channels must be bit-identical to the oracle's: decimator rows, matched-filter rows, bits, the
sample index of every bit, the counters.
"""
import os

import numpy as np
import pytest

import jsdrcuda as J
import oracle as O

pytestmark = pytest.mark.gpu


def scenario(seed):
    rng = np.random.default_rng(1000 + seed)
    rate = int(rng.choice([48000, 96000, 192000]))
    nchan = int(rng.choice([1, 2, 5, 31, 32, 33, 47, 64, 96]))
    shared = bool(rng.integers(0, 2)) and nchan > 1
    s16 = bool(rng.integers(0, 2))
    nblocks = int(rng.integers(3, 7))
    max_block = int(rng.choice([700, 4096, 9600, 20000]))
    lens = [int(rng.integers(0, max_block + 1)) for _ in range(nblocks)]
    lens[int(rng.integers(0, nblocks))] = max_block
    if seed % 4 == 0:
        lens[0] = 1
    if seed % 5 == 0:
        lens[1] = 0
    lim = rate / 2.2
    tuning = rng.uniform(-lim, lim, nchan)
    tuning[rng.integers(0, nchan)] = 12000.0
    kernel = int(rng.choice([J.KERNEL_AUTO, J.KERNEL_AUTO, J.KERNEL_TILE, J.KERNEL_STREAM]))
    retunes = {}                                              # block index -> [(chan, hz)]
    for _ in range(int(rng.integers(0, 4))):
        retunes.setdefault(int(rng.integers(1, nblocks)), []).append((int(rng.integers(0, nchan)), float(rng.uniform(-lim, lim))))
    return rng, rate, nchan, shared, s16, lens, max_block, tuning, kernel, retunes


@pytest.mark.parametrize("seed", range(int(os.environ.get("JSDR_FUZZ_SEEDS", "24"))))   # more seeds: a soak run
def test_bank_scenarios_bit_exact(ctx, seed):
    rng, rate, nchan, shared, s16, lens, max_block, tuning, kernel, retunes = scenario(seed)
    adsc = J.AudioDescriptor(rate, blen=max_block * 4)
    bank = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tuning, max_block=max_block)
    bank.set_kernel(kernel)
    watch = sorted(set([0, nchan - 1, int(rng.integers(0, nchan))] + [c for v in retunes.values() for c, _ in v]))
    orcs = {c: O.Bpsk(rate, float(tuning[c])) for c in watch}
    what = f"seed {seed}: rate {rate}, {nchan} tuners, shared={shared}, s16={s16}, kernel {kernel}, blocks {lens}"
    for k, n in enumerate(lens):
        for c, hz in retunes.get(k, []):
            bank.set_tuning(c, hz)
            orcs[c].set_tuning(hz)
        rows = 1 if shared else nchan
        if s16:
            raw = rng.integers(-32768, 32768, (rows, 2 * n)).astype(np.int16)
            if n:
                bank.receive_raw(raw if not shared else raw[0], shared=shared)
            else:
                bank.receive_raw(np.zeros(0, np.int16), shared=True)
            fl = O.s16_to_float(raw.ravel()).reshape(rows, 2 * n)
        else:
            fl = rng.uniform(-1, 1, (rows, 2 * n)).astype(np.float32)
            if n:
                bank.receive(fl if not shared else fl[0], shared=shared)
            else:
                bank.receive(np.zeros(0, np.float32), shared=True)
        nds = bank.last_nds()
        ds, dm = bank.read_ds(), bank.read_dm()
        bits, at = bank.read_bits()
        for c in watch:
            r = orcs[c].receive(fl[0 if shared else c])
            assert nds == r["ds"].shape[0], f"{what}: block {k} channel {c} output count"
            assert np.array_equal(ds[c], r["ds"]), f"{what}: block {k} channel {c} decimator"
            assert np.array_equal(dm[c], r["dm"]), f"{what}: block {k} channel {c} matched filter"
            assert np.array_equal(bits[c], r["bits"]), f"{what}: block {k} channel {c} bits"
            assert np.array_equal(at[c], r["bit_at"]), f"{what}: block {k} channel {c} bit positions"
    cnt = bank.counters()
    for c in watch:
        oc = orcs[c].counters()
        assert (cnt[c, 0], cnt[c, 1], cnt[c, 2]) == (oc["raw"], oc["ds"], oc["bit"]), f"{what}: counters of channel {c}"
    bank.close()


FFT_N = [2, 3, 16, 100, 128, 256, 500, 512, 1000, 1024, 2048, 4096, 4410, 4800, 6000, 8192, 9600, 16384, 19200, 32768, 65536]


@pytest.mark.parametrize("seed", range(int(os.environ.get("JSDR_FUZZ_SEEDS", "24"))))
def test_fft_scenarios_against_the_binary64_oracle(ctx, seed):
    """fft.java:190-224 on drawn shapes: any supported length (single-CTA, split, staged and
    four-step paths), ragged batches, s16 blocks with a drawn I/Q correction or float blocks,
    noise plus a tone of drawn level and bin (on or off the grid, either half, DC and Nyquist
    included); every block's dB row within 1e-4 of full scale of the binary64 restatement, the
    published maximum and its wrapping-int32 frequency exact."""
    from test_gpu_parity import check_psd
    rng = np.random.default_rng(5000 + seed)
    n = int(rng.choice(FFT_N))
    if not J.fft_supported(n):
        pytest.skip(f"no plan for N={n}")
    rate = int(rng.choice([44100, 96000, 192000]))
    batch = int(rng.integers(1, 10)) if n <= 19200 else int(rng.integers(1, 4))
    s16 = bool(rng.integers(0, 2))
    t = np.arange(n)
    x = np.empty((batch, 2 * n), dtype=np.float64)
    for b in range(batch):
        k = rng.choice([0.0, n / 2, float(rng.integers(0, n)), float(rng.uniform(0, n))])
        tone = rng.uniform(0.01, 0.7) * np.exp(2j * np.pi * (k * t / n + rng.uniform()))
        noise = rng.uniform(-0.2, 0.2, (n, 2))
        x[b, 0::2], x[b, 1::2] = tone.real + noise[:, 0], tone.imag + noise[:, 1]
    f = J.fft(ctx, None, J.AudioDescriptor(rate), max_batch=batch, n=n)
    if s16:
        ic, qc = (int(rng.integers(-300, 300)), int(rng.integers(-300, 300))) if rng.integers(0, 2) else (0, 0)
        raw = np.round(x * 32767).astype(np.int16)
        psd, pk = f.receive_batch(raw, s16=True, ic=ic, qc=qc)
        fl = np.stack([O.s16_to_float(raw[b], ic=ic, qc=qc) for b in range(batch)])
    else:
        fl = x.astype(np.float32)
        psd, pk = f.receive_batch(fl)
    f.close()
    for b in range(batch):
        check_psd(psd[b], fl[b], rate, n)
        row = psd[b, :n]
        assert pk[b] == int(np.argmax(row)) and psd[b, n + 1] == row.max()


@pytest.mark.parametrize("seed", range(int(os.environ.get("JSDR_FUZZ_SEEDS", "24"))))
def test_demod_scenarios_bit_exact_without_nco(ctx, seed):
    """demod.java:378-396,405-481 on drawn shapes: channels, band edges (the all-pass included),
    detector mode, AGC, ragged blocks with carried FIR history / running mean / discriminator
    state.  NCO off, so nothing transcendental enters and every float and every s16 is exact."""
    rng = np.random.default_rng(9000 + seed)
    rate = int(rng.choice([44100, 48000, 96000, 192000]))
    nchan = int(rng.choice([1, 2, 3, 7, 33]))
    mode = int(rng.integers(0, 5))
    doagc = bool(rng.integers(0, 2))
    max_block = int(rng.choice([333, 2048, 9600]))
    lens = [int(rng.integers(1, max_block + 1)) for _ in range(int(rng.integers(2, 6)))] + [max_block]
    d = J.demod(ctx, J.AudioDescriptor(rate), nchan=nchan, max_block=max_block, dofir=True, dodwn=False)
    d.set_mode(mode, doagc)
    os_, lilq = [], [np.zeros(2, np.float32) for _ in range(nchan)]
    for c in range(nchan):
        if rng.integers(0, 6) == 0:
            lo, hi = J.INT_MIN, 0                                 # all-pass (demod.java:343-346)
        else:
            lo = int(rng.integers(-rate // 2, rate // 2 - 200))
            hi = int(rng.integers(lo + 100, rate // 2))
        d.weights(lo, hi, chan=c)
        o = O.Demod(rate, True, False)
        o.weights(O.INT_MIN if lo == J.INT_MIN else lo, hi)
        os_.append(o)
    scale = float(rng.choice([0.01, 0.3, 1.0]))
    for n in lens:
        x = (rng.standard_normal((nchan, 2 * n)) * scale).astype(np.float32)
        audio, ma = d.receive_audio(x)
        for c in range(nchan):
            ref_a, ref_ma = O.demod_detect(os_[c].receive(x[c]), mode, rate, doagc, lilq[c])
            assert np.array_equal(audio[c], ref_a), (seed, rate, nchan, mode, doagc, n, c)
            assert np.array_equal(ma[c], ref_ma, equal_nan=True), (seed, rate, nchan, mode, doagc, n, c)
    d.close()


@pytest.mark.parametrize("seed", range(int(os.environ.get("JSDR_FUZZ_SEEDS", "24"))))
def test_fir_and_waterfall_scenarios_bit_exact(ctx, seed):
    """fir.java:169-228 (int samples x double taps, (int) truncation and saturation, carried
    delay line, wrapping complex multiply) and waterfall.java:90-107 on drawn shapes."""
    rng = np.random.default_rng(13000 + seed)
    rate = float(rng.choice([8000.0, 44100.0, 96000.0]))
    f, o = J.fir(ctx, rate), O.Fir(rate)
    f1 = int(rng.integers(0, int(rate) // 2 - 200))
    f2 = int(rng.integers(f1 + 100, int(rate) // 2))
    assert np.array_equal(f.weights(f1, f2), o.weights(f1, f2))
    for _ in range(int(rng.integers(2, 6))):
        n = int(rng.integers(1, 20000))
        span = int(rng.choice([100, 32768, 1 << 31]))
        x = rng.integers(-span, span, n).astype(np.int32)
        assert np.array_equal(f.filter(x)[0], o.filter(x)), (seed, n, span)
    m = int(rng.integers(1, 5000))
    a = rng.integers(-(1 << 31), 1 << 31, (m, 2)).astype(np.int32)
    b = rng.integers(-(1 << 31), 1 << 31, (m, 2)).astype(np.int32)
    assert np.array_equal(f.complex_mod(a, b), O.complex_mod(a, b))
    f.close()
    n = int(rng.choice([128, 1000, 4096, 9600, 19200]))
    width = int(rng.integers(1, n + 1))
    rows = int(rng.integers(1, 9))
    psd = rng.uniform(-140, 10, (rows, n + 2)).astype(np.float32)
    psd[rng.integers(0, rows), rng.integers(0, n)] = -np.inf
    pix = J.waterfall_rows(ctx, psd, width)
    for r in range(rows):
        assert np.array_equal(pix[r], O.waterfall_row(psd[r], width)), (seed, n, width, r)


@pytest.mark.parametrize("seed", range(max(1, int(os.environ.get("JSDR_FUZZ_SEEDS", "24")) // 4)))
def test_frame_stage_scenarios(ctx, seed):
    """Sync correlator + FECDecode (FUNcubeBPSKDemod.java:553-574, FECDecoder.java:703-852) on
    drawn damage: two frames whose RS blocks carry 0..22 symbol errors behind the convolutional
    code AND whose channel symbols are flipped in 0..300 places in front of it, so Viterbi, both
    RS outcomes (corrected / -1 / miscorrected) and the channel-error count are all exercised.
    Frame list, return values, payloads and cntFEC / cntDec equal the oracle's."""
    import rs_warp_model as M
    from oracle import siggen
    from test_gpu_fec import mettab, oracle_frames
    alpha, index, poly = (J.probe_table(t).tolist() for t in ("ALPHA_TO", "INDEX_OF", "RS_poly"))
    gf = M.GF(alpha, index)
    par = M.rs_parity_map(alpha, index, poly)
    scr, sync = J.probe_table("Scrambler").tolist(), J.probe_table("SYNC_VECTOR").tolist()
    rng = np.random.default_rng(17000 + seed)
    frames = []
    for _ in range(2):
        blocks = []
        for r in range(2):
            d = rng.integers(0, 256, 128).tolist()
            cw = d + M.rs_parity(d, par, gf)
            for q in rng.choice(160, int(rng.integers(0, 23)), replace=False):
                cw[q] ^= int(rng.integers(1, 256))
            blocks.append(cw)
        sym = M.symbols_from_blocks(blocks, scr, sync)
        flips = rng.choice(sym.size, int(rng.choice([0, 10, 100, 300])), replace=False)
        sym[flips] ^= 1
        frames.append(sym)
    sig = siggen.make_iq_s16(None, rate=96000, ebn0_db=None, pad_to=9600, symbols=frames)
    fbuf = O.s16_to_float(sig)
    adsc = J.AudioDescriptor(96000)
    bank = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=[12000.0])
    bank.enable_fec(mettab(), max_frames=8)
    orc = O.Bpsk(96000, 12000.0, do_fec=True)
    got, allbits = [], []
    for k in range(fbuf.size // (2 * adsc.samples)):
        blk = fbuf[2 * k * adsc.samples: 2 * (k + 1) * adsc.samples]
        bank.receive(blk)
        got += bank.read_frames()
        allbits.append(orc.receive(blk)["bits"])
    ref = oracle_frames(np.concatenate(allbits))
    assert len(got) == len(ref), (seed, len(got), len(ref))
    for (ch, at, err, data), (rat, rerr, rdata) in zip(got, ref):
        assert at == rat and err == rerr, (seed, at, rat, err, rerr)
        if rerr >= 0:
            assert np.array_equal(data, rdata)
    fec, dec = bank.fec_counters()
    oc = orc.counters()
    assert (int(fec[0]), int(dec[0])) == (oc["fec"], oc["dec"]), seed
    bank.close()


@pytest.mark.parametrize("seed", range(max(1, int(os.environ.get("JSDR_FUZZ_SEEDS", "24")) // 6)))
def test_autotune_scenarios(ctx, seed):
    """doBufferFFT (FUNcubeBPSKDemod.java:406-464) on drawn carriers in either scanned band, with
    and without noise: the centre bin and every bit identical to the oracle, samples within
    1e-9 of full scale (the two sides transform with different binary64 FFTs)."""
    from oracle import siggen
    rng = np.random.default_rng(21000 + seed)
    rate = int(rng.choice([96000, 192000]))
    adsc = J.AudioDescriptor(rate)
    n = adsc.samples
    upper = bool(rng.integers(0, 2))
    lo_bin, hi_bin = (n // 4 + 300, n // 2 - 300) if upper else (300, n // 4 - 300)
    carrier = float(rng.uniform(lo_bin, hi_bin)) * rate / n
    ebn0 = [None, 16.0, 20.0][int(rng.integers(0, 3))]
    sig = siggen.make_iq_s16(siggen.random_payloads(1), rate=rate, carrier_hz=carrier, ebn0_db=ebn0,
                             noise_seed=int(rng.integers(1, 1 << 30)), pad_to=n)
    fbuf = O.s16_to_float(sig)
    bank = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=[12000.0])
    bank.set_autotune(True, upper)
    orc = O.Bpsk(rate, 12000.0)
    orc.s.doUp = int(upper)
    worst, nbits = 0.0, 0
    for k in range(min(fbuf.size // (2 * n), 12)):
        blk = fbuf[2 * k * n: 2 * (k + 1) * n]
        bank.receive(blk)
        r = orc.receive(blk, autotune=True)
        assert int(bank.centre_bins()[0]) == r["centre_bin"], (seed, k)
        ds = bank.read_ds()[0]
        assert ds.shape == r["ds"].shape
        worst = max(worst, float(np.max(np.abs(ds - r["ds"]))) / (0.9 * 32768.0))
        assert np.array_equal(bank.read_bits()[0][0], r["bits"]), (seed, k)
        nbits += r["bits"].size
    assert worst <= 1e-9 and nbits > 300, (seed, worst, nbits)
    bank.close()


@pytest.mark.parametrize("seed", range(int(os.environ.get("JSDR_FUZZ_SEEDS", "24"))))
def test_pump_scenarios_equal_the_separate_handlers(ctx, seed):
    """jsdr_pump_receive_s16 / jsdr_pump_waterfall_s16 (JavaAudio.java:262-304) on drawn shapes —
    channel counts on both sides of every chunk boundary of the pipelined host path, blocks per
    call, FFT length, I/Q correction, host or device buffers, PSD or pixel rows — against the
    spectrum handler and the tuner bank called one after the other on the same bytes (each of
    which the tests above tie to the oracle): identical PSD rows / pixel rows, peak bins,
    decimator rows and bits."""
    rng = np.random.default_rng(25000 + seed)
    rate = int(rng.choice([96000, 192000]))
    n = int(rng.choice([128, 1000, 1024, 4096, 4800]))
    nchan = int(rng.choice([1, 7, 8, 15, 16, 17, 33, 37, 130, 200]))
    nblk = int(rng.integers(1, 4))
    ic, qc = (int(rng.integers(-500, 500)), int(rng.integers(-500, 500))) if rng.integers(0, 2) else (0, 0)
    device = bool(rng.integers(0, 2))
    pixels = bool(rng.integers(0, 2))
    width = int(rng.integers(1, n + 1))
    S, rows = nblk * n, nchan * nblk
    raw = rng.integers(-32768, 32768, (nchan, 2 * S)).astype(np.int16)
    tuning = rng.uniform(-rate / 2.2, rate / 2.2, nchan)
    adsc = J.AudioDescriptor(rate, blen=S * 4)
    what = (seed, rate, n, nchan, nblk, ic, qc, device, pixels, width)
    # the two handlers, separately
    f1 = J.fft(ctx, None, adsc, max_batch=rows, n=n)
    b1 = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tuning, max_block=S)
    psd1, pk1 = f1.receive_batch(raw.reshape(rows, 2 * n), s16=True, ic=ic, qc=qc)
    b1.receive_raw(raw, ic=ic, qc=qc, shared=False)
    ds1, bits1 = b1.read_ds(), b1.read_bits()[0]
    # the pump
    f2 = J.fft(ctx, None, adsc, max_batch=rows, n=n)
    b2 = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tuning, max_block=S)
    if device:
        d_raw = ctx.dev_alloc(raw.nbytes)
        d_raw.upload(raw)
        d_pk = ctx.dev_alloc(rows * 4)
        if pixels:
            d_pix, d_peak = ctx.dev_alloc(rows * width * 4), ctx.dev_alloc(rows * 8)
            J.pump_waterfall_s16(f2, b2, d_raw.ptr, nblk, width, d_pix.ptr, d_peak.ptr, d_pk.ptr, mem=J.MEM_DEVICE, ic=ic, qc=qc)
            ctx.sync()
            pix2 = d_pix.download(np.int32, rows * width).reshape(rows, width)
            peak2 = d_peak.download(np.float32, rows * 2).reshape(rows, 2)
            d_pix.free()
            d_peak.free()
        else:
            d_psd = ctx.dev_alloc(rows * (n + 2) * 4)
            J.pump_receive_s16(f2, b2, d_raw.ptr, nblk, d_psd.ptr, d_pk.ptr, mem=J.MEM_DEVICE, ic=ic, qc=qc)
            ctx.sync()
            psd2 = d_psd.download(np.float32, rows * (n + 2)).reshape(rows, n + 2)
            d_psd.free()
        pk2 = d_pk.download(np.int32, rows)
        d_pk.free()
        d_raw.free()
    else:
        pk2 = np.zeros(rows, np.int32)
        if pixels:
            pix2, peak2 = np.zeros((rows, width), np.int32), np.zeros((rows, 2), np.float32)
            J.pump_waterfall_s16(f2, b2, raw, nblk, width, pix2, peak2, pk2, ic=ic, qc=qc)
        else:
            psd2 = np.zeros((rows, n + 2), np.float32)
            J.pump_receive_s16(f2, b2, raw, nblk, psd2, pk2, ic=ic, qc=qc)
    assert np.array_equal(pk2, pk1), what
    if pixels:
        assert np.array_equal(pix2, J.waterfall_rows(ctx, psd1, width)), what
        assert np.array_equal(peak2, psd1[:, n:]), what
    else:
        assert np.array_equal(psd2, psd1), what
    assert np.array_equal(b2.read_ds(), ds1), what
    bits2 = b2.read_bits()[0]
    assert all(np.array_equal(x, y) for x, y in zip(bits2, bits1)), what
    for h in (f1, f2, b1, b2):
        h.close()


@pytest.mark.parametrize("kernel,s16", [(J.KERNEL_TILE, False), (J.KERNEL_STREAM, True), (J.KERNEL_STREAM, False)])
def test_bank_absurd_but_finite_tunings_follow_the_reference(ctx, kernel, s16):
    """Tunings far outside the band are finite numbers the reference would take from its dialog
    (FUNcubeBPSKDemod.java:175-188): the phase then grows without bound and the table index comes
    from Java's saturating (int) cast.  The bank must neither hang nor differ."""
    rate, n = 96000, 4800
    tuning = [1e300, 250000.0, -1e9, 0.75 * rate, 0.0, -0.0, 1e-300, 47999.9, 96000.0, 96001.0, 1e7] + list(np.linspace(500.0, 40000.0, 29))
    bank = J.FUNcubeBPSKDemod(ctx, None, J.AudioDescriptor(rate, blen=4 * n), tuning=tuning, max_block=n)
    bank.set_kernel(kernel)
    orcs = [O.Bpsk(rate, t) for t in tuning[:13]]
    rng = np.random.default_rng(77)
    for k in range(3):
        if s16:
            raw = rng.integers(-32768, 32768, 2 * n).astype(np.int16)
            bank.receive_raw(raw, shared=True)
            x = O.s16_to_float(raw)
        else:
            x = rng.uniform(-1, 1, 2 * n).astype(np.float32)
            bank.receive(x, shared=True)
        ds, bits = bank.read_ds(), bank.read_bits()[0]
        for c, o in enumerate(orcs):
            r = o.receive(x)
            assert np.array_equal(ds[c], r["ds"], equal_nan=True), (k, tuning[c])
            assert np.array_equal(bits[c], r["bits"]), (k, tuning[c])
    bank.close()


@pytest.mark.parametrize("seed", range(int(os.environ.get("JSDR_FUZZ_SEEDS", "24"))))
def test_bank_filter_and_rate_shapes(ctx, seed):
    """Every decimation the rate rule allows (rate / 9600 from 1 to 64, FUNcubeBPSKDemod.java:476)
    with drawn decimator filters of 1..128 taps (jsdr_bpsk_set_ds_filter): the compiled shapes and
    the generic loop, the tile and the streaming kernel, against the oracle with the same taps."""
    rng = np.random.default_rng(31000 + seed)
    D = int(rng.choice([1, 2, 3, 5, 7, 10, 20, 33, 64]))
    rate = min(9600 * D + int(rng.integers(0, 9600)) * int(rng.integers(0, 2)), 614400)   # integer division :476
    ntaps = int(rng.choice([1, 2, 3, 26, 27, 28, 63, 64, 65, 127, 128]))
    taps = rng.uniform(-1, 1, ntaps) if rng.integers(0, 2) else np.hamming(ntaps + 2)[1:-1] / max(ntaps, 1)
    nchan = int(rng.choice([1, 3, 32, 45]))
    max_block = int(rng.choice([1, 50, 999, 6400]))
    lens = [int(rng.integers(0, max_block + 1)) for _ in range(int(rng.integers(2, 6)))] + [max_block]
    tuning = rng.uniform(-rate / 2.2, rate / 2.2, nchan)
    bank = J.FUNcubeBPSKDemod(ctx, None, J.AudioDescriptor(rate, blen=4 * max_block), tuning=tuning, max_block=max_block)
    bank.set_ds_filter(taps)
    bank.set_kernel(int(rng.choice([J.KERNEL_AUTO, J.KERNEL_TILE, J.KERNEL_STREAM])))
    watch = sorted({0, nchan - 1, int(rng.integers(0, nchan))})
    orcs = {c: O.Bpsk(rate, float(tuning[c]), ds_taps=taps) for c in watch}
    what = (seed, rate, D, ntaps, nchan, lens)
    for k, n in enumerate(lens):
        x = rng.uniform(-1, 1, (nchan, 2 * n)).astype(np.float32)
        bank.receive(x if n else np.zeros(0, np.float32), shared=(n == 0))
        ds, dm = bank.read_ds(), bank.read_dm()
        bits = bank.read_bits()[0]
        for c in watch:
            r = orcs[c].receive(x[c])
            assert ds[c].shape == r["ds"].shape, (what, k, c)
            assert np.array_equal(ds[c], r["ds"]), (what, k, c)
            assert np.array_equal(dm[c], r["dm"]), (what, k, c)
            assert np.array_equal(bits[c], r["bits"]), (what, k, c)
    bank.close()


def test_long_runs_do_not_drift(ctx):
    """Recurrences that run for the life of a handle — the tuner phase and its fixed-point
    shadow (re-anchored at exact checkpoints), the VCO phase, the 65-slot matched-filter rotation
    (cntDS % 65), the bit-timing IIRs, demod.java's float NCO phase (:424-433) — over 1500 blocks
    (14.4 M samples per channel): still bit-identical (bank) / within 1e-6 (demod NCO, whose
    cos/sin come from a different libm) at the end, every block checked on the way."""
    rate, n, nblk = 96000, 9600, 1500
    tuning = [12000.0, -31234.5, 47000.0, 3.0]
    bank = J.FUNcubeBPSKDemod(ctx, None, J.AudioDescriptor(rate), tuning=tuning)
    orcs = [O.Bpsk(rate, t) for t in tuning]
    d = J.demod(ctx, J.AudioDescriptor(rate), nchan=1, max_block=n)
    d.weights(9000, 15000)
    od = O.Demod(rate, True, True)
    od.weights(9000, 15000)
    rng = np.random.default_rng(99)
    nbits = 0
    for k in range(nblk):
        x = rng.uniform(-0.5, 0.5, 2 * n).astype(np.float32)
        bank.receive(x, shared=True)
        ds, bits = bank.read_ds(), bank.read_bits()[0]
        for c, o in enumerate(orcs):
            r = o.receive(x)
            assert np.array_equal(ds[c], r["ds"]), (k, c)
            assert np.array_equal(bits[c], r["bits"]), (k, c)
            nbits += r["bits"].size
        y = d.receive(x)[0]
        assert np.max(np.abs(y - od.receive(x))) <= 1e-6, k
    cnt = bank.counters()
    for c, o in enumerate(orcs):
        oc = o.counters()
        assert (cnt[c, 0], cnt[c, 1], cnt[c, 2]) == (oc["raw"], oc["ds"], oc["bit"]) and oc["raw"] == nblk * n
    assert nbits > 10000
    bank.close()
    d.close()


@pytest.mark.parametrize("seed", range(max(1, int(os.environ.get("JSDR_FUZZ_SEEDS", "24")) // 3)))
def test_binary32_decimator_stays_within_tolerance(ctx, seed):
    """JSDR_PREC_F32 (channeliser use, stages == 1): same exact table index sequence, mix and FIR
    in binary32 — every output of every channel within the bound derived from the kernel's arithmetic
    (tests/f32_bound.py, which one wrong table index at a tap of 3e-4 or more leaves), and within 1e-4
    of full scale of the binary64 oracle (the north_star's bar; measured ~2e-6), on drawn shapes, s16
    and float input, compiled (27/10, 27/20, 64/20) and generic taps."""
    import f32_bound as F
    rng = np.random.default_rng(37000 + seed)
    D, ntaps = [(10, 27), (20, 27), (20, 64), (10, 40), (5, 27)][int(rng.integers(0, 5))]
    rate = 9600 * D
    nchan = int(rng.choice([8, 40, 70]))
    n = int(rng.choice([999, 4800, 19200]))
    taps = np.sinc((np.arange(ntaps) - (ntaps - 1) / 2) * 0.9 / D) * np.hamming(ntaps)
    taps /= taps.sum()
    tuning = rng.uniform(500.0, rate / 2.2, nchan)
    bank = J.FUNcubeBPSKDemod(ctx, None, J.AudioDescriptor(rate, blen=4 * n), tuning=tuning, max_block=n, stages=1)
    if ntaps != 27 or rng.integers(0, 2):
        bank.set_ds_filter(taps)
        otaps = taps
    else:
        otaps = None
    bank.set_precision(J.PREC_F32)
    rng.integers(0, nchan)                                   # (the draw that once picked a watched channel)
    orcs = {c: O.Bpsk(rate, float(tuning[c]), ds_taps=otaps, stages=1) for c in range(nchan)}
    s16 = bool(rng.integers(0, 2))
    bounds = {c: F.Bound(O.default_taps()[0] if otaps is None else otaps, D, s16) for c in orcs}
    worst = 0.0
    for k in range(3):
        if s16:
            raw = rng.integers(-32768, 32768, (nchan, 2 * n)).astype(np.int16)
            bank.receive_raw(raw, shared=False)
            x = O.s16_to_float(raw.ravel()).reshape(nchan, 2 * n)
        else:
            x = rng.uniform(-1, 1, (nchan, 2 * n)).astype(np.float32)
            bank.receive(x, shared=False)
        ds = bank.read_ds()
        for c in orcs:
            r = orcs[c].receive(x[c])["ds"]
            assert ds[c].shape == r.shape
            assert np.all(np.abs(ds[c] - r) <= bounds[c].block(x[c])), (seed, D, ntaps, nchan, n, s16, k, c)
            worst = max(worst, float(np.max(np.abs(ds[c] - r))) / (0.9 * 32768.0))
    assert worst <= 1e-4, (seed, D, ntaps, nchan, n, s16, worst)
    bank.close()


def test_frame_capacity_overflow_is_counted_not_written(ctx):
    """More frames in one call than max_frames: *nframes says how many were detected, only
    max_frames are returned, nothing is written past the caller's arrays, cntFEC / cntDec still
    count every one (FUNcubeBPSKDemod.java:563-571)."""
    from oracle import siggen
    from test_gpu_fec import mettab
    pl = siggen.random_payloads(3)
    sig = siggen.make_iq_s16(pl, rate=96000, ebn0_db=None, pad_to=9600)
    fbuf = O.s16_to_float(sig)
    n = fbuf.size // 2                                       # the whole signal as ONE block: 3 frames per channel
    nchan = 5
    bank = J.FUNcubeBPSKDemod(ctx, None, J.AudioDescriptor(96000, blen=4 * n), tuning=[12000.0] * nchan, max_block=n)
    bank.enable_fec(mettab(), max_frames=1)
    bank.receive(fbuf, shared=True)
    cap = 4                                                  # fewer than the 15 detected
    nf = C_int32 = np.zeros(1, np.int32)
    chan = np.full(cap + 2, -7, np.int32)
    at = np.full(cap + 2, -7, np.int64)
    err = np.full(cap + 2, -7, np.int32)
    data = np.full((cap + 2, 256), 0xEE, np.uint8)
    J._ck(J.lib().jsdr_bpsk_read_frames(bank.h, J._ptr(nf), J._ptr(chan), J._ptr(at), J._ptr(err), J._ptr(data), cap))
    assert nf[0] == 3 * nchan, nf
    assert np.all(chan[cap:] == -7) and np.all(at[cap:] == -7) and np.all(err[cap:] == -7) and np.all(data[cap:] == 0xEE)
    assert list(chan[:cap]) == [0, 0, 0, 1] and np.all(err[:cap] >= 0)
    for i in range(cap):
        assert np.array_equal(data[i], pl[i % 3])
    fec, dec = bank.fec_counters()
    assert list(fec) == [3] * nchan and list(dec) == [3] * nchan
    bank.close()
    assert C_int32 is nf


@pytest.mark.parametrize("seed", range(max(1, int(os.environ.get("JSDR_FUZZ_SEEDS", "24")) // 3)))
def test_many_handles_interleaved_on_one_context(ctx, seed):
    """Handles of one context share its streams and fork / join events: several banks (tile and
    streaming kernel, with and without the frame stage, asynchronous reads), spectrum handlers and
    a demod called in a drawn order, per-kernel profiling switched on and off in between — every
    handle still equals its own oracle, as if it were alone."""
    from test_gpu_parity import check_psd
    rng = np.random.default_rng(41000 + seed)
    rate = int(rng.choice([96000, 192000]))
    n = rate // 10
    adsc = J.AudioDescriptor(rate)
    banks = []
    for _ in range(int(rng.integers(2, 5))):
        nchan = int(rng.choice([1, 2, 33, 64]))
        tuning = rng.uniform(-rate / 2.2, rate / 2.2, nchan)
        b = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tuning, stages=int(rng.choice([1, 3, 3])))
        watch = sorted({0, nchan - 1})
        banks.append((b, nchan, {c: O.Bpsk(rate, float(tuning[c]), stages=b.stages) for c in watch}))
    ffts = [J.fft(ctx, None, adsc, max_batch=3, n=int(m)) for m in rng.choice([1024, 4096, n], 2)]
    d = J.demod(ctx, adsc, nchan=2, max_block=n, dofir=True, dodwn=False)
    d.weights(2000, 9000)
    d.weights(-9000, -2000, chan=1)
    od = [O.Demod(rate, True, False), O.Demod(rate, True, False)]
    od[0].weights(2000, 9000)
    od[1].weights(-9000, -2000)
    pinned = ctx.host_alloc((64 * (n // (rate // 9600) + 2) * 2,), np.float64)
    profiling = False
    for step in range(int(rng.integers(8, 20))):
        if rng.integers(0, 4) == 0:
            profiling = not profiling
            ctx.profile(profiling)
            if not profiling:
                ctx.profile_read()
        kind = int(rng.integers(0, 4))
        if kind <= 1:
            b, nchan, orcs = banks[int(rng.integers(0, len(banks)))]
            m = int(rng.choice([n, n, n // 2, 777]))
            x = rng.uniform(-1, 1, (nchan, 2 * m)).astype(np.float32)
            b.receive(x, shared=False)
            if rng.integers(0, 2):
                nds = b.read_ds_async(pinned)
                ctx.sync()
                ds = pinned[:nchan * nds * 2].reshape(nchan, nds, 2).copy()
            else:
                ds = b.read_ds()
            for c, o in orcs.items():
                r = o.receive(x[c])
                assert np.array_equal(ds[c], r["ds"]), (seed, step, c)
                if b.stages == 3:
                    assert np.array_equal(b.read_bits()[0][c], r["bits"]), (seed, step, c)
        elif kind == 2:
            f = ffts[int(rng.integers(0, 2))]
            batch = int(rng.integers(1, 4))
            x = rng.uniform(-1, 1, (batch, 2 * f.n)).astype(np.float32)
            psd, _ = f.receive_batch(x)
            for k in range(batch):
                check_psd(psd[k], x[k], rate, f.n)
        else:
            m = int(rng.integers(1, n + 1))
            x = rng.uniform(-1, 1, (2, 2 * m)).astype(np.float32)
            y = d.receive(x)
            for c in range(2):
                assert np.array_equal(y[c], od[c].receive(x[c])), (seed, step, c)
    ctx.profile(False)
    ctx.profile_read()
    ctx.host_free(pinned)
    for b, _, _ in banks:
        b.close()
    for f in ffts:
        f.close()
    d.close()
