"""demod.java's down-shift (:423-433) on the GPU held to the CPU model of tests/nco_phase.py with no
tolerance: every mixed float of k_demod / k_demod_s16 equal to mix_reference (the oracle's bit-exact
FIR output, the reference's float phase replayed in C, nco_sincos emulated bit for bit, the
correctly rounded float on the library path), every s16 audio sample and max/avg pair equal to the
oracle's detectors on that reference.

Inputs (tests/test_nco_model.py checks that they reach what is claimed): tunings whose phase
returns exactly to 0.0, placed at every chunk / tile / call seam of the car replay; tunings with
phi = 0, phi just below and at 2 pi and above (car runs negative) and below 0 (car grows onto the
library path); banks on both sides of k_car_scout's 128 channels per CTA; ragged call lengths;
f32 and s16 entry points from host and device memory, shared input and chan_stride > nsamples; the
state changes of weights() and set_flags(); the pump's demod handler; and one run of 2^24 samples
into the stall, where car - phi rounds back to car."""
import numpy as np
import pytest

import jsdrcuda as J
import nco_phase as N
import oracle as O

pytestmark = pytest.mark.gpu

KINDS = ("f32", "f32_dev", "s16", "s16_dev")
IC, QC = 9, -9


# ------------------------------------------------------------------ the GPU side, in one place
def gpu_receive(ctx, d, kind, x, S, stride):
    """The FIR + NCO output [nchan][2 S] of one call: x is float32 or int16 IQ rows (or one shared
    row when stride is 0), `kind` picks the entry point and where the data lives."""
    L = J.lib()
    nchan = d.nchan
    out = np.empty((nchan, 2 * S), np.float32)
    s16 = kind.startswith("s16")
    a = np.ascontiguousarray(x, np.int16 if s16 else np.float32)
    if kind.endswith("_dev"):
        d_in, d_out = ctx.dev_alloc(a.nbytes), ctx.dev_alloc(out.nbytes)
        d_in.upload(a)
        args = (J._ptr(d_in), S, stride) + ((IC, QC) if s16 else ()) + (J._ptr(d_out), J.MEM_DEVICE)
        J._ck((L.jsdr_demod_receive_s16 if s16 else L.jsdr_demod_receive_f32)(d.h, *args))
        ctx.sync()
        out[:] = d_out.download(np.float32, out.size).reshape(out.shape)
        d_in.free()
        d_out.free()
    else:
        args = (J._ptr(a), S, stride) + ((IC, QC) if s16 else ()) + (J._ptr(out), J.MEM_HOST)
        J._ck((L.jsdr_demod_receive_s16 if s16 else L.jsdr_demod_receive_f32)(d.h, *args))
    return out


def make_input(rng, kind, rows, width, scale=0.5):
    if kind.startswith("s16"):
        raw = rng.integers(-32768, 32768, (rows, 2 * width)).astype(np.int16)
        raw[:, :4] = np.array([32767, -32768, 32760, -32760], np.int16)[: min(4, 2 * width)]    # wrap under ic/qc
        return raw
    return (rng.uniform(-1, 1, (rows, 2 * width)) * scale).astype(np.float32)


def as_float(kind, row):
    return O.s16_to_float(row, IC, QC) if kind.startswith("s16") else row


class Pair:
    """A GPU demod handle and one RefDemod per channel, fed the same calls."""

    def __init__(self, ctx, rate, nchan, max_block, dofir=True, dodwn=True):
        self.ctx, self.rate, self.nchan = ctx, rate, nchan
        self.d = J.demod(ctx, J.AudioDescriptor(rate), nchan=nchan, max_block=max_block, dofir=dofir, dodwn=dodwn)
        self.ref = [N.RefDemod(rate, dofir, dodwn) for _ in range(nchan)]

    def weights(self, c, flo, fhi):
        self.d.weights(flo, fhi, chan=c)
        self.ref[c].weights(flo, fhi)

    def set_flags(self, dofir, dodwn):
        self.d.set_flags(dofir, dodwn)
        for r in self.ref:
            r.set_flags(dofir, dodwn)

    def call(self, rng, kind, S, shared=False, stride=None):
        """One call of S samples per channel; asserts every float equal; returns the references."""
        width = S if stride is None else stride
        x = make_input(rng, kind, 1 if shared else self.nchan, width)
        got = gpu_receive(self.ctx, self.d, kind, x[0] if shared else x, S, 0 if shared else width)
        refs = []
        for c in range(self.nchan):
            row = as_float(kind, x[0 if shared else c])[: 2 * S]
            ref, allowed = self.ref[c].receive(row)
            assert N.matches(got[c], ref, allowed), (kind, S, c, float(self.ref[c].phi))
            refs.append((ref, allowed))
        return refs

    def close(self):
        self.d.close()


def bank_tunings(rate, nchan, rng):
    """Distinct tunings: every zero-return and planned one first, then drawn ones over (-rate, 2 rate)."""
    fl = [f for f, _ in N.zero_returns(rate)] + N.planned_tunings(rate)
    seen = set(fl)
    while len(fl) < nchan:
        f = int(rng.integers(-rate + 1, 2 * rate))
        if f not in seen:
            seen.add(f)
            fl.append(f)
    return fl[:nchan]


# ------------------------------------------------------------------ tests
@pytest.mark.parametrize("rate", [44100, 96000, 192000])
def test_zero_returns_at_every_seam(ctx, rate):
    """Each tuning whose phase returns exactly to 0.0, the return placed by a prefix call at every
    seam: samples 0, 31, 32, 33 of the call (first and last of the first chunk, first two of the
    next), the last sample of the first tile and the first of the second, and (prefix only) the
    first sample of a call, which the carried car_ feeds."""
    rng = np.random.default_rng(rate)
    p = Pair(ctx, rate, 1, 4200)
    for i, (flo, m) in enumerate(N.zero_returns(rate)):
        for j, q in enumerate(N.SEAMS):
            kind = KINDS[(i + j) % len(KINDS)]
            p.weights(0, flo, flo + 3000)                       # car back to 0, delay line cleared
            pre = N.placement(m, q)
            if pre:
                p.call(rng, kind, pre)
            assert N.phases(p.ref[0].phi, p.ref[0].car, q + 1)[q] == 0.0
            p.call(rng, KINDS[(i + j + 1) % len(KINDS)], N.TILE + 76)
    p.close()


@pytest.mark.parametrize("nchan", [1, 127, 128, 129, 300])
def test_banks_and_ragged_calls(ctx, nchan):
    """Distinct tunings per channel (the zero-return and out-of-range ones among them) through
    k_car_scout's 128-channel CTAs and the [chunk][nchan] checkpoints; ragged call lengths, the
    largest max_block (not a multiple of 32); every entry point, shared input, chan_stride > S."""
    rate, max_block = 96000, 4133
    rng = np.random.default_rng(1000 + nchan)
    p = Pair(ctx, rate, nchan, max_block)
    for c, flo in enumerate(bank_tunings(rate, nchan, rng)):
        p.weights(c, flo, flo + 4000)
    lengths = (1, 31, 32, 33, 1023, 1024, 1025, 4100, max_block)
    for i, S in enumerate(lengths):
        p.call(rng, KINDS[i % len(KINDS)], S)
    for i, kind in enumerate(KINDS):
        p.call(rng, kind, 1025 + i, shared=True)
        p.call(rng, kind, 777, stride=1100)
    p.close()


@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("doagc", [False, True])
def test_audio_equals_the_detectors_on_the_reference(ctx, mode, doagc):
    """receive_audio / receive_audio_raw: every s16 sample and max/avg pair equal to O.demod_detect
    on mix_reference, with the li/lq pair carried across calls."""
    rate, nchan = 96000, 4
    rng = np.random.default_rng(50 + 2 * mode + doagc)
    d = J.demod(ctx, J.AudioDescriptor(rate), nchan=nchan, max_block=4100)
    d.set_mode(mode, doagc)
    ref = [N.RefDemod(rate) for _ in range(nchan)]
    lilq = [np.zeros(2, np.float32) for _ in range(nchan)]
    for c, flo in enumerate((16000, -8000, rate + 3, 6400)):
        d.weights(flo, flo + 6000, chan=c)
        ref[c].weights(flo, flo + 6000)
    for i, S in enumerate((1, 33, 1025, 4100, 31)):
        s16 = i % 2 == 1
        x = make_input(rng, "s16" if s16 else "f32", nchan, S)
        audio, ma = d.receive_audio_raw(x, ic=IC, qc=QC) if s16 else d.receive_audio(x)
        for c in range(nchan):
            mixed, allowed = ref[c].receive(as_float("s16" if s16 else "f32", x[c]))
            assert not allowed, (S, c)                  # no library-path value near a midpoint here
            ra, rma = O.demod_detect(mixed, mode, rate, doagc, lilq[c])
            assert np.array_equal(audio[c], ra), (S, c)
            assert np.array_equal(ma[c], rma, equal_nan=True), (S, c)
    d.close()


def test_weights_and_flags_between_calls(ctx):
    """weights(INT_MIN, ..) keeps phi and car (demod.java:343), any other weights() puts car back
    to 0 and clears the delay line (:369-374), and with dodwn off car does not move."""
    rate = 96000
    rng = np.random.default_rng(7)
    p = Pair(ctx, rate, 3, 2100)
    for c, flo in enumerate((19200, -20000, rate + 1)):
        p.weights(c, flo, flo + 5000)
    p.call(rng, "f32", 1000)
    p.weights(1, J.INT_MIN, 0)
    p.call(rng, "s16", 77)
    p.weights(0, 6400, 9000)
    p.call(rng, "f32_dev", 1030)
    p.set_flags(True, False)
    p.call(rng, "s16_dev", 500)
    p.call(rng, "f32", 33)
    p.set_flags(True, True)
    p.call(rng, "f32", 2100)
    p.set_flags(False, True)
    p.call(rng, "s16", 64)
    p.weights(2, J.INT_MIN, 0)
    p.set_flags(True, True)
    p.call(rng, "f32", 1)
    p.call(rng, "f32", 1999)
    p.close()


@pytest.mark.parametrize("nblk", [1, 3])
@pytest.mark.parametrize("mode", [2, 3])
def test_pump_demod_against_the_oracle(ctx, nblk, mode):
    """jsdr_pump_demod_s16 (the car replay on side2 behind ev_car_ready, one FIR + NCO launch over
    the row, k_detect per block), two calls in a row: every audio sample and max/avg pair equal to
    the detectors on mix_reference, block by block."""
    rate, n, nchan = 96000, 1024, 3
    S = nblk * n
    rng = np.random.default_rng(400 + 10 * mode + nblk)
    adsc = J.AudioDescriptor(rate)
    f = J.fft(ctx, None, adsc, max_batch=nchan * nblk, n=n)
    b = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=[12000.0, -7000.0, 30000.0], max_block=S, stages=3)
    d = J.demod(ctx, adsc, nchan=nchan, max_block=S)
    d.set_mode(mode, True)
    ref = [N.RefDemod(rate) for _ in range(nchan)]
    lilq = [np.zeros(2, np.float32) for _ in range(nchan)]
    for c, flo in enumerate((19200, -9000, rate + 7)):
        d.weights(flo, flo + 5000, chan=c)
        ref[c].weights(flo, flo + 5000)
    for call in range(2):
        raw = make_input(rng, "s16", nchan, S)
        psd = np.zeros((nchan * nblk, n + 2), np.float32)
        pk = np.zeros(nchan * nblk, np.int32)
        audio = np.zeros((nchan, S), np.int16)
        ma = np.zeros((nchan, nblk, 2), np.float32)
        J.pump_demod_s16(f, b, d, raw, nblk, psd, audio, ma, pk, ic=IC, qc=QC)
        for c in range(nchan):
            x = O.s16_to_float(raw[c], IC, QC)
            for j in range(nblk):
                mixed, allowed = ref[c].receive(x[2 * j * n: 2 * (j + 1) * n])
                assert not allowed, (call, c, j)
                ra, rma = O.demod_detect(mixed, mode, rate, True, lilq[c])
                assert np.array_equal(audio[c, j * n: (j + 1) * n], ra), (call, c, j)
                assert np.array_equal(ma[c, j], rma, equal_nan=True), (call, c, j)
    for h in (f, b, d):
        h.close()


def test_long_run_into_the_stall(ctx):
    """One channel with phi just inside -1 for 2^24 + 1024 samples in four calls: car leaves the
    fast path after 8 samples, climbs to 2^24 and stops there (car - phi == car) at sample
    2^24 + 1.  Every float equal to the reference; the library-path samples within SLOW_DOUBT
    binary64 ulps of a float midpoint may take either neighbour, and there are few of them."""
    rate = 96000
    rng = np.random.default_rng(24)
    p = Pair(ctx, rate, 1, max(N.LONG_CALLS))
    p.weights(0, N.LONG_FLO, N.LONG_FLO + 6000)
    for i, S in enumerate(N.LONG_CALLS):
        p.call(rng, ("f32", "s16_dev")[i % 2], S)
    st = p.ref[0].stats
    print(f"long run: {sum(N.LONG_CALLS)} samples, {st.get('slow', 0)} on the library path, "
          f"{st.get('slow_doubt', 0)} within {N.SLOW_DOUBT} ulps of a float midpoint")
    assert p.ref[0].car == np.float32(2.0 ** 24)
    assert st.get("slow_doubt", 0) <= 64
    p.close()
