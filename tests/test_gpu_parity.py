"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle
on the same seeded inputs, against the committed golden vectors, and through
size-independent properties at larger sizes.

Tolerances (BASELINE north_star): spectra and float-filtered samples within 1e-4 of
full scale against the double-precision path; everything computed in binary64 or
integers (tuner/decimator/matched filter outputs, bits, int FIR) is compared
bit-exactly.
"""
import numpy as np
import pytest

import oracle as O
from oracle import siggen
from conftest import load_s16

import jsdrcuda as J

pytestmark = pytest.mark.gpu

FS_TOL = 1e-4          # fraction of full scale


def amp_from_db(psd):
    return np.power(10.0, np.asarray(psd, dtype=np.float64) / 20.0)


def check_psd(psd_gpu, buf, rate, n):
    """psd_gpu[n+2] against the double-precision oracle path for one block."""
    pw = O.fft_power_f64(buf)                      # (re^2+im^2)*(2/N)^2 in binary64
    amp_ref = np.sqrt(pw)                          # = 2|X|/N; full scale (|X|/N = 1) is 2
    amp_gpu = amp_from_db(psd_gpu[:n])
    assert np.max(np.abs(amp_gpu - amp_ref)) <= FS_TOL * 2.0
    strong = amp_ref > 1e-3
    if strong.any():
        db_ref = 10 * np.log10(pw[strong])
        assert np.max(np.abs(psd_gpu[:n][strong] - db_ref)) < 0.05
    # published maximum: value equals the largest bin, frequency follows fft.java:214-221
    m = np.max(psd_gpu[:n][np.isfinite(psd_gpu[:n])]) if np.isfinite(psd_gpu[:n]).any() else None
    if m is not None:
        assert psd_gpu[n + 1] == m
        k = int(np.argmax(psd_gpu[:n] == m))       # first strict maximum
        p = 2 * k if 2 * k < n else 2 * k - 2 * n
        p = (p * rate) & 0xffffffff
        p = p - (1 << 32) if p >= (1 << 31) else p
        assert psd_gpu[n] == np.float32(int(p / (2 * n)))


# ------------------------------------------------------------------ fft.java
ALL_N = [128, 256, 512, 1024, 2048, 4096, 8192, 16384, 4410, 4800, 9600, 19200]


@pytest.mark.parametrize("n", ALL_N)
def test_fft_spectrum_matches_dft(ctx, n):
    rng = np.random.default_rng(n)
    batch = 5
    x = (rng.uniform(-1, 1, (batch, n)) + 1j * rng.uniform(-1, 1, (batch, n))).astype(np.complex64)
    f = J.fft(ctx, None, J.AudioDescriptor(96000), max_batch=batch, n=n)
    X = f.forward(x.view(np.float32))
    f.close()
    for b in range(batch):
        ref = O.dft_f64(x[b].astype(np.complex128))
        assert np.max(np.abs(X[b] - ref)) / n <= FS_TOL, f"block {b}"
        # and it is far better than the tolerance
        assert np.max(np.abs(X[b] - ref)) / n <= 2e-6


@pytest.mark.parametrize("n", ALL_N)
def test_fft_psd_config3_known_answers_and_random(ctx, n):
    """BASELINE config 3 shape: block 0 impulse, 1 DC, 2 on-bin tone, rest uniform noise."""
    rate = 192000
    rng = np.random.default_rng(42)
    batch = 37                                     # not a multiple of any blocks-per-CTA
    x = np.zeros((batch, n), np.complex64)
    x[0, 0] = 1.0
    x[1, :] = 1.0
    k0 = n - n // 8                                # negative frequency, wraps int32 at 192 kS/s for large n
    x[2, :] = 0.5 * np.exp(2j * np.pi * k0 * np.arange(n) / n)
    x[3:] = rng.uniform(-1, 1, (batch - 3, n)) + 1j * rng.uniform(-1, 1, (batch - 3, n))
    f = J.fft(ctx, None, J.AudioDescriptor(rate), max_batch=batch, n=n)
    psd, pk = f.receive_batch(x.view(np.float32))
    f.close()
    assert pk[0] == 0 and np.allclose(psd[0, :n], 10 * np.log10((2.0 / n) ** 2), atol=1e-3)
    assert pk[1] == 0 and abs(psd[1, 0] - 10 * np.log10(4.0)) < 1e-3
    assert pk[2] == k0 and abs(psd[2, k0] - 0.0) < 1e-3          # amplitude 0.5 complex tone reads 0 dB
    for b in range(batch):
        check_psd(psd[b], x[b].view(np.float32), rate, n)
    for b in (3, 17, batch - 1):                   # the oracle's own float path agrees on the arg-max
        _, opk = O.fft_receive(x[b].view(np.float32), rate)
        assert pk[b] == opk


def test_fft_config1_fixtures(ctx, golden):
    """BASELINE config 1: the reference's sine4410 fixtures, one block each."""
    for name, n, fn in (("raw4096", 4096, "sine4410.raw"), ("raw128", 128, "sine4410-short.raw"),
                        ("wav4410", 4410, "sine4410-wav4410.raw")):
        raw = load_s16(fn)
        buf = O.s16_to_float(raw)
        pub = J.Publish()
        seen = []
        pub.listen(lambda k, v: seen.append((k, v.copy())))
        h = J.fft(ctx, pub, J.AudioDescriptor(44100, blen=4 * n))
        psd = h.receive(buf).copy()
        assert seen and seen[0][0] == "fft-psd" and seen[0][1].size == n + 2     # fft.java:226
        check_psd(psd, buf, 44100, n)
        g = golden[f"psd_{name}"]
        fin = np.isfinite(g[:n]) & (g[:n] > -80)
        assert np.max(np.abs(psd[:n][fin] - g[:n][fin])) < 0.02
        # Q3: real input -> the +f/-f bins tie to ~1e-4 dB; peak frequency is equal up to sign
        assert abs(abs(psd[n]) - abs(g[n])) <= 44100 / n + 1 and abs(psd[n + 1] - g[n + 1]) < 1e-3
        # IRawHandler path: same block as s16 bytes, converted on the device
        psd2 = h.receive_raw(raw).copy()
        check_psd(psd2, buf, 44100, n)
        assert np.max(np.abs(amp_from_db(psd2[:n]) - amp_from_db(psd[:n]))) < 2e-5
        h.close()


def test_fft_s16_ingest_with_iq_correction(ctx):
    """JavaAudio.java:281-288: s += (short)ic with 16-bit wrap before scaling."""
    n = 1024
    rng = np.random.default_rng(5)
    raw = rng.integers(-32768, 32768, (3, 2 * n)).astype(np.int16)
    raw[0, :8] = [32767, 32767, -32768, -32768, 32760, 32760, 0, 0]       # these wrap with ic=+9/qc=-9
    f = J.fft(ctx, None, J.AudioDescriptor(96000), max_batch=3, n=n)
    psd, _ = f.receive_batch(raw, s16=True, ic=9, qc=-9)
    f.close()
    for b in range(3):
        check_psd(psd[b], O.s16_to_float(raw[b], ic=9, qc=-9), 96000, n)


def test_fft_edge_cases(ctx):
    n = 256
    f = J.fft(ctx, None, J.AudioDescriptor(96000), max_batch=4, n=n)
    psd, pk = f.receive_batch(np.zeros((0, 2 * n), np.float32))           # empty batch
    assert psd.shape == (0, n + 2)
    psd, pk = f.receive_batch(np.zeros((2, 2 * n), np.float32))           # log10(0) published as -inf (Q4)
    assert np.all(np.isneginf(psd[:, :n])) and np.all(pk == -1)
    o, _ = O.fft_receive(np.zeros(2 * n, np.float32), 96000)
    assert psd[0, n] == o[n] and psd[0, n + 1] == o[n + 1]
    with pytest.raises(J.JsdrError):
        f.receive_batch(np.zeros((5, 2 * n), np.float32))                 # beyond max_batch
    f.close()
    with pytest.raises(J.JsdrError):
        J.fft(ctx, None, J.AudioDescriptor(96000), n=4097)                # no plan: loud, not a fallback


def test_fft_large_batch_linearity_and_parseval(ctx):
    """Size-independent properties on a config-3 sized launch (10^4 blocks)."""
    n, batch = 1024, 10000
    rng = np.random.default_rng(9)
    a = (rng.uniform(-1, 1, (batch, n)) + 1j * rng.uniform(-1, 1, (batch, n))).astype(np.complex64)
    f = J.fft(ctx, None, J.AudioDescriptor(96000), max_batch=batch, n=n)
    A = f.forward(a.view(np.float32))
    # Parseval per block
    e_t = np.sum(np.abs(a.astype(np.complex128)) ** 2, axis=1)
    e_f = np.sum(np.abs(A.astype(np.complex128)) ** 2, axis=1) / n
    assert np.max(np.abs(e_f / e_t - 1)) < 1e-5
    # linearity: F(a + i*roll(a)) = F(a) + i*F(roll(a)); a circular shift is a phase ramp
    sh = np.roll(a, 1, axis=1)
    S = f.forward(sh.view(np.float32))
    ramp = np.exp(-2j * np.pi * np.arange(n) / n)
    assert np.max(np.abs(S - A * ramp)) / n < 2e-6
    psd, pk = f.receive_batch(a.view(np.float32))
    idx = rng.choice(batch, 8, replace=False)
    for b in idx:
        check_psd(psd[b], a[b].view(np.float32), 96000, n)
    f.close()


# ------------------------------------------------------------------ FUNcubeBPSKDemod.java
def run_blocks(bank, orc, fbuf, nblock):
    """Feed identical blocks to the GPU bank (one channel) and the oracle; compare everything bit-exactly."""
    gb, ob = [], []
    for k in range(fbuf.size // 2 // nblock):
        blk = fbuf[2 * k * nblock:2 * (k + 1) * nblock]
        bank.receive(blk)
        r = orc.receive(blk)
        assert np.array_equal(bank.read_ds()[0], r["ds"]), f"decimator differs in block {k}"
        assert np.array_equal(bank.read_dm()[0], r["dm"]), f"matched filter differs in block {k}"
        bits, at = bank.read_bits()
        assert np.array_equal(bits[0], r["bits"]) and np.array_equal(at[0], r["bit_at"]), f"bits differ in block {k}"
        gb.append(bits[0])
        ob.append(r["bits"])
    return np.concatenate(gb), np.concatenate(ob)


def test_bpsk_config2_bits_exact_and_frames_decode(ctx, golden):
    """BASELINE config 2: 96 kS/s, three FUNcube frames, tuner -> decimator -> matched
    filter -> bits; every stage bit-identical to the oracle, frames decode to the payload."""
    pl = siggen.random_payloads(3)
    sig = siggen.make_iq_s16(pl, rate=96000, pad_to=9600)
    fbuf = O.s16_to_float(sig)
    adsc = J.AudioDescriptor(96000)
    pub = J.Publish()
    bank = J.FUNcubeBPSKDemod(ctx, pub, adsc, tuning=[12000.0])
    orc = O.Bpsk(96000, 12000.0)
    gbits, obits = run_blocks(bank, orc, fbuf, adsc.samples)
    assert np.array_equal(gbits, golden["cfg2_bits"])
    assert pub.getPublish("FUNcube0-bpsk-tune") == 12000 and pub.getPublish("FUNcube0-bpsk-centre") == -1
    c = bank.counters()[0]
    assert c[0] == sig.size // 2 and c[1] == c[0] // 10 and c[2] == gbits.size
    bank.close()
    # the GPU's bit stream through the sync correlator + FEC (oracle side, :553-574) gives the payloads
    frames = []
    corr = np.zeros(5200, np.int8)
    sync = O.sync_vector().astype(np.int32)
    for bit in gbits:
        corr[:-1] = corr[1:]
        corr[-1] = bit
        if int(np.dot(corr[::80].astype(np.int32), sync)) >= 45:
            rc, out = O.fec_decode(np.where(corr == 1, 0xc0, 0x40).astype(np.uint8))
            if rc >= 0:
                frames.append(out)
    assert len(frames) == 3 and all(np.array_equal(f, p) for f, p in zip(frames, pl))


def test_bpsk_raw_s16_ingest_matches_float_path(ctx):
    sig = siggen.make_iq_s16(siggen.random_payloads(1), rate=96000, pad_to=9600)[: 2 * 9600 * 6]
    adsc = J.AudioDescriptor(96000)
    bank = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=[12000.0])
    orc = O.Bpsk(96000, 12000.0)
    for k in range(6):
        raw = sig[k * 19200:(k + 1) * 19200]
        bank.receive_raw(raw, ic=3, qc=-2)
        r = orc.receive(O.s16_to_float(raw, ic=3, qc=-2))
        assert np.array_equal(bank.read_ds()[0], r["ds"])
        assert np.array_equal(bank.read_bits()[0][0], r["bits"])
    bank.close()


def test_bpsk_ragged_blocks_and_state_carry(ctx):
    """Edge cases: empty, tiny and odd block sizes (dsCnt and both FIR histories carry)."""
    sig = siggen.make_iq_s16(siggen.random_payloads(1), rate=96000, pad_to=9600)[: 2 * 70000]
    fbuf = O.s16_to_float(sig)
    bank = J.FUNcubeBPSKDemod(ctx, None, J.AudioDescriptor(96000), tuning=[12000.0], max_block=30000)
    orc = O.Bpsk(96000, 12000.0)
    pos = 0
    for n in (1, 7, 9600, 0, 13, 4410, 3, 26, 27, 25000, 9, 30000):
        blk = fbuf[2 * pos:2 * (pos + n)]
        pos += n
        bank.receive(blk)
        r = orc.receive(blk)
        assert bank.last_nds() == r["ds"].shape[0]
        assert np.array_equal(bank.read_ds()[0], r["ds"]), n
        assert np.array_equal(bank.read_dm()[0], r["dm"]), n
        assert np.array_equal(bank.read_bits()[0][0], r["bits"]), n
    bank.close()


def test_bpsk_one_stream_many_tuners(ctx):
    """The reference's own model (jsdr.java:479-483): one stream, several tuners.
    Includes the two carriers that decode (tuning +-1200), a zero and a negative tuning
    (mixer bypass, FUNcubeBPSKDemod.java:388) and arbitrary ones."""
    sig = siggen.make_iq_s16(siggen.random_payloads(1), rate=96000, pad_to=9600)[: 2 * 9600 * 8]
    fbuf = O.s16_to_float(sig)
    tun = [12000.0, 14400.0, 0.0, -5000.0, 47999.0, 3.7, 31234.5]
    adsc = J.AudioDescriptor(96000)
    bank = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tun)
    orcs = [O.Bpsk(96000, t) for t in tun]
    for k in range(8):
        blk = fbuf[k * 19200:(k + 1) * 19200]
        bank.receive(blk)
        ds, dm = bank.read_ds(), bank.read_dm()
        bits, _ = bank.read_bits()
        for c, o in enumerate(orcs):
            r = o.receive(blk)
            assert np.array_equal(ds[c], r["ds"]), (k, c)
            assert np.array_equal(dm[c], r["dm"]), (k, c)
            assert np.array_equal(bits[c], r["bits"]), (k, c)
    # retune one channel mid-stream (actionPerformed, :174-189): the phase keeps accumulating
    bank.set_tuning(5, 13200.0)
    orcs[5].set_tuning(13200.0)
    blk = fbuf[:19200]
    bank.receive(blk)
    assert np.array_equal(bank.read_ds()[5], orcs[5].receive(blk)["ds"])
    bank.close()


def test_bpsk_config4_shape_many_streams_64_taps(ctx):
    """BASELINE config 4 shape at test size: independent streams at 192 kS/s, D=20,
    64-tap Hamming low-pass (cut-off 4800 Hz), per-channel tuning in [2000, 90000]."""
    rate, nchan, S = 192000, 24, 19200
    rng = np.random.default_rng(7)
    tun = rng.uniform(2000, 90000, nchan)
    taps = siggen.lowpass_taps(64, 4800.0, rate)
    raw = rng.integers(-20000, 20000, (nchan, 2 * S * 2)).astype(np.int16)
    adsc = J.AudioDescriptor(rate)
    bank = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tun, stages=1)
    bank.set_ds_filter(taps)
    orcs = [O.Bpsk(rate, t, ds_taps=taps) for t in tun]
    for k in range(2):
        blk = np.ascontiguousarray(raw[:, k * 2 * S:(k + 1) * 2 * S])
        bank.receive_raw(blk)
        ds = bank.read_ds()
        assert ds.shape == (nchan, S // 20, 2)
        for c, o in enumerate(orcs):
            assert np.array_equal(ds[c], o.receive(O.s16_to_float(blk[c]))["ds"]), (k, c)
    bank.close()


def test_bpsk_decimator_impulse_response_is_taps(ctx):
    ds27, _ = O.default_taps()
    bank = J.FUNcubeBPSKDemod(ctx, None, J.AudioDescriptor(96000), tuning=[0.0], stages=1)
    x = np.zeros(2 * 9600, np.float32)
    x[2 * 9] = 1.0
    bank.receive(x)
    got = bank.read_ds()[0][:3, 0]
    assert np.array_equal(got, np.array([ds27[0], ds27[10], ds27[20]]) * (0.9 * 32768.0))
    bank.close()


# ------------------------------------------------------------------ demod.java
def test_demod_fir_and_nco(ctx, golden):
    raw = load_s16("sine4410.raw")
    buf = O.s16_to_float(raw)
    adsc = J.AudioDescriptor(44100, blen=4 * 4096)
    d = J.demod(ctx, adsc)
    x = np.random.default_rng(1).standard_normal(2 * 4096).astype(np.float32)
    d.set_flags(True, False)
    assert np.all(d.receive(x) == 0)                              # Q5: zero taps until weights()
    w = d.weights(3000, 6000)
    assert np.array_equal(w, golden["demod_w"])                   # host formula, demod.java:356-366
    d.set_flags(True, True)
    o = O.Demod(44100, True, True)
    o.weights(3000, 6000)
    for k in range(3):                                            # carried FIR history and NCO phase
        y = d.receive(buf)[0]
        r = o.receive(buf)
        assert np.max(np.abs(y - r)) <= 1e-6                      # float path; full scale is 1
        if k < 2:
            assert np.max(np.abs(y - golden[f"demod_out{k + 1}"])) <= 1e-6
    # FIR alone is exact (no transcendental): float mul/add in the reference order
    d2 = J.demod(ctx, adsc, dofir=True, dodwn=False)
    d2.weights(3000, 6000)
    o2 = O.Demod(44100, True, False)
    o2.weights(3000, 6000)
    for _ in range(2):
        assert np.array_equal(d2.receive(x)[0], o2.receive(x))
    d2.weights(J.INT_MIN, 0)                                      # all-pass: unit tap at 10
    y = d2.receive(x)[0]
    assert np.array_equal(y[20:], x[:-20])
    d.close()
    d2.close()


def test_demod_many_channels_ragged(ctx):
    rate, nchan = 96000, 5
    rng = np.random.default_rng(2)
    d = J.demod(ctx, J.AudioDescriptor(rate), nchan=nchan, max_block=5000)
    os_ = []
    for c in range(nchan):
        lo = -20000 + 9000 * c
        d.weights(lo, lo + 6000, chan=c)
        o = O.Demod(rate, True, True)
        o.weights(lo, lo + 6000)
        os_.append(o)
    for n in (5000, 1, 19, 20, 21, 1023, 1024, 1025, 33):
        x = rng.uniform(-1, 1, (nchan, 2 * n)).astype(np.float32)
        y = d.receive(x)
        for c in range(nchan):
            assert np.max(np.abs(y[c] - os_[c].receive(x[c]))) <= 1e-6, (n, c)
    d.close()


# ------------------------------------------------------------------ fir.java
def test_fir_int_filter_exact(ctx):
    raw = load_s16("sine4410.raw")
    x = raw[0::2].astype(np.int32)
    f = J.fir(ctx, 44100.0)
    o = O.Fir(44100.0)
    assert np.array_equal(f.weights(3000, 6000), o.weights(3000, 6000))
    for _ in range(2):                                            # second call: carried delay line
        assert np.array_equal(f.filter(x)[0], o.filter(x))
    rng = np.random.default_rng(3)
    big = rng.integers(-(1 << 31), 1 << 31, 5000).astype(np.int32)       # saturating (int) cast
    assert np.array_equal(f.filter(big)[0], o.filter(big))
    for n in (1, 19, 20, 21, 255, 256, 257):
        xs = rng.integers(-4096, 4096, n).astype(np.int32)
        assert np.array_equal(f.filter(xs)[0], o.filter(xs))
    assert np.array_equal(f.weights(J.INT_MIN, J.INT_MIN), o.weights(O.INT_MIN, O.INT_MIN))
    f.close()


def test_fir_nco_and_complex_mod_exact(ctx):
    f = J.fir(ctx, 44100.0)
    o = O.Fir(44100.0)
    g1 = f.complex_gen(1000)
    g2 = f.complex_gen(500)
    assert np.array_equal(g1[:300], o.complex_gen(1000, 0, 300))
    assert np.array_equal(f.complex_mod(g1[:2000], g2[:2000]), O.complex_mod(g1[:2000], g2[:2000]))
    rng = np.random.default_rng(4)
    a = rng.integers(-(1 << 31), 1 << 31, (1000, 2)).astype(np.int32)    # int32 wrap
    b = rng.integers(-(1 << 31), 1 << 31, (1000, 2)).astype(np.int32)
    assert np.array_equal(f.complex_mod(a, b), O.complex_mod(a, b))
    f.close()


# ------------------------------------------------------------------ pump
def test_pump_equals_separate_handlers(ctx):
    rate, nchan, n, nblk = 192000, 6, 4096, 3
    rng = np.random.default_rng(11)
    tun = rng.uniform(2000, 90000, nchan)
    raw = rng.integers(-30000, 30000, (nchan, nblk * n * 2)).astype(np.int16)
    adsc = J.AudioDescriptor(rate)
    f = J.fft(ctx, None, adsc, max_batch=nchan * nblk, n=n)
    b1 = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tun, max_block=nblk * n, stages=1)
    b2 = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=tun, max_block=nblk * n, stages=1)
    psd = np.empty((nchan * nblk, n + 2), np.float32)
    pk = np.empty(nchan * nblk, np.int32)
    J.pump_receive_s16(f, b1, raw, nblk, psd, pk)
    psd2, pk2 = f.receive_batch(raw.reshape(nchan * nblk, 2 * n), s16=True)
    assert np.array_equal(psd, psd2) and np.array_equal(pk, pk2)
    b2.receive_raw(raw)
    assert np.array_equal(b1.read_ds(), b2.read_ds())
    o = O.Bpsk(rate, tun[2])
    assert np.array_equal(b1.read_ds()[2], o.receive(O.s16_to_float(raw[2]))["ds"])
    for h in (f, b1, b2):
        h.close()


def test_error_paths_return_codes_not_crashes(ctx):
    """Nothing may throw through IAudioHandler.receive (JavaAudio.java:321-323): bad calls come
    back as status codes with a message, and the handles stay usable."""
    adsc = J.AudioDescriptor(96000)
    with pytest.raises(J.JsdrError) as e:
        J.fft(ctx, None, adsc, n=11 * 1024)                       # a prime factor outside 2, 3, 5, 7
    assert e.value.code == -4                                     # JSDR_EUNSUPPORTED
    f = J.fft(ctx, None, adsc, max_batch=2, n=1024)
    with pytest.raises(J.JsdrError) as e:
        f.receive_batch(np.zeros((3, 2048), np.float32))          # batch > max_batch
    assert e.value.code == -1
    assert f.receive(np.zeros(2048, np.float32))[1024 + 1] == np.float32(-3.4028234663852886e38)   # still works (Q4: all -inf)
    f.close()
    bank = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=[12000.0], max_block=4800)
    with pytest.raises(J.JsdrError):
        bank.receive(np.zeros(2 * 9600, np.float32))              # nsamples > max_block_samples
    with pytest.raises(J.JsdrError):
        bank.read_frames() if hasattr(bank, "_max_frames") else J._ck(J.lib().jsdr_bpsk_read_frames(bank.h, None, None, None, None, None, 0))
    bank.receive(np.zeros(2 * 4800, np.float32))                  # and the bank is still usable
    assert bank.read_ds().shape == (1, 480, 2)
    bank.close()
