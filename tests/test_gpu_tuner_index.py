"""The tuner bank against the oracle on tunings whose phases sweep through every table boundary band
(tests/tuner_phase.py, bank_plan): near-grid and on-grid tunings from phase 0, retunes between ragged
blocks, and climbs from negative phase through 0 placed at the streaming kernel's seams, including exact
returns to 0.0.  Every channel is compared bit for bit (tests/test_tuner_index_model.py shows that these
inputs see a wrong guard in any of the three index paths)."""
import numpy as np
import pytest

import f32_bound as F
import jsdrcuda as J
import oracle as O
import tuner_phase as T

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sm_count():
    """The device's SM count: the streaming kernel's segment length, and so the seams the plan's
    crossings are placed at, follow from it."""
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count

# (rate, taps or None for the default 27, kernel mode, s16, shared input, (ic, qc), stages)
CASES = {
    "stream-27x10-s16": (96000, None, J.KERNEL_STREAM, True, False, (0, 0), 3),
    "stream-27x20-f32": (192000, None, J.KERNEL_STREAM, False, False, (0, 0), 1),
    "stream-64x20-s16-shared": (192000, 64, J.KERNEL_STREAM, True, True, (0, 0), 1),
    "auto-27x10-s16-iqcorr": (96000, None, J.KERNEL_AUTO, True, False, (-300, 211), 1),
    "auto-27x20-f32-shared": (192000, None, J.KERNEL_AUTO, False, True, (0, 0), 1),
    "tile-27x10-f32": (96000, None, J.KERNEL_TILE, False, False, (0, 0), 3),
    "tile-generic-40x5-s16-iqcorr": (48000, 40, J.KERNEL_TILE, True, False, (57, -999), 1),
}


def lowpass(ntaps, D):
    h = np.sinc((np.arange(ntaps) - (ntaps - 1) / 2) * 0.9 / D) * np.hamming(ntaps)
    return h / h.sum()


def input_block(rng, rows, n, s16, ic, qc):
    if s16:
        raw = rng.integers(-32768, 32768, (rows, 2 * n)).astype(np.int16)
        return raw, np.stack([O.s16_to_float(r, ic=ic, qc=qc) for r in raw]) if n else np.zeros((rows, 0), np.float32)
    x = rng.uniform(-1, 1, (rows, 2 * n)).astype(np.float32)
    return x, x


def check_block(bank, orcs, fl, shared, stages, what):
    nds = bank.last_nds()
    ds = bank.read_ds()
    dm = bank.read_dm() if stages >= 2 else None
    bits, at = bank.read_bits() if stages >= 3 else (None, None)
    for c, o in enumerate(orcs):
        r = o.receive(fl[0 if shared else c])
        assert nds == r["ds"].shape[0], f"{what}: channel {c} output count"
        assert np.array_equal(ds[c], r["ds"]), f"{what}: channel {c} (tuning {bank.tuning[c]!r} Hz) decimator"
        if stages >= 2:
            assert np.array_equal(dm[c], r["dm"]), f"{what}: channel {c} matched filter"
        if stages >= 3:
            assert np.array_equal(bits[c], r["bits"]), f"{what}: channel {c} bits"
            assert np.array_equal(at[c], r["bit_at"]), f"{what}: channel {c} bit positions"


def retune(bank, orcs, plan, k):
    if k == 0:
        return
    for c in np.nonzero(plan.tunings[k] != plan.tunings[k - 1])[0]:
        bank.set_tuning(int(c), float(plan.tunings[k][c]))
        orcs[c].set_tuning(float(plan.tunings[k][c]))


def check_counters(bank, orcs, what):
    cnt = bank.counters()
    for c, o in enumerate(orcs):
        oc = o.counters()
        assert (cnt[c, 0], cnt[c, 1], cnt[c, 2]) == (oc["raw"], oc["ds"], oc["bit"]), f"{what}: counters of channel {c}"


@pytest.mark.parametrize("case", list(CASES))
def test_every_channel_equals_the_oracle_through_the_boundaries(ctx, sm_count, case):
    rate, ntaps, mode, s16, shared, (ic, qc), stages = CASES[case]
    D = rate // 9600
    plan = T.bank_plan(rate, s16=s16, sm_count=sm_count)
    max_block = max(plan.lens)
    bank = J.FUNcubeBPSKDemod(ctx, None, J.AudioDescriptor(rate, blen=4 * max_block), tuning=plan.tunings[0],
                              max_block=max_block, stages=stages)
    taps = None
    if ntaps is not None:
        taps = lowpass(ntaps, D)
        bank.set_ds_filter(taps)
    bank.set_kernel(mode)
    orcs = [O.Bpsk(rate, float(t), ds_taps=taps, stages=stages) for t in plan.tunings[0]]
    rng = np.random.default_rng(sum(map(ord, case)))
    rows = 1 if shared else plan.nchan
    for k, n in enumerate(plan.lens):
        retune(bank, orcs, plan, k)
        data, fl = input_block(rng, rows, n, s16, ic, qc)
        if s16:
            bank.receive_raw(data[0] if shared else data, ic=ic, qc=qc, shared=shared)
        else:
            bank.receive(data[0] if shared else data, shared=shared)
        check_block(bank, orcs, fl, shared, stages, f"{case}, {plan.what}: block {k}")
    check_counters(bank, orcs, f"{case}, {plan.what}")
    bank.close()


def test_pump_with_device_buffers_through_the_boundaries(ctx, sm_count):
    """jsdr_pump_receive_s16 from device memory (the pump places the phase replay itself), three calls of
    two 4096-sample blocks with the climbs through 0 in the second call."""
    rate, n, nblk = 96000, 4096, 2
    S = n * nblk
    plan = T.bank_plan(rate, lens=(S, S, S), pump=True, sm_count=sm_count)
    adsc = J.AudioDescriptor(rate, blen=4 * S)
    rows = plan.nchan * nblk
    f = J.fft(ctx, None, adsc, max_batch=rows, n=n)
    bank = J.FUNcubeBPSKDemod(ctx, None, adsc, tuning=plan.tunings[0], max_block=S, stages=1)
    orcs = [O.Bpsk(rate, float(t), stages=1) for t in plan.tunings[0]]
    rng = np.random.default_rng(4711)
    d_raw = ctx.dev_alloc(plan.nchan * 2 * S * 2)
    d_psd = ctx.dev_alloc(rows * (n + 2) * 4)
    d_pk = ctx.dev_alloc(rows * 4)
    for k in range(len(plan.lens)):
        retune(bank, orcs, plan, k)
        raw = rng.integers(-32768, 32768, (plan.nchan, 2 * S)).astype(np.int16)
        d_raw.upload(raw)
        J.pump_receive_s16(f, bank, d_raw.ptr, nblk, d_psd.ptr, d_pk.ptr, mem=J.MEM_DEVICE)
        ctx.sync()
        fl = np.stack([O.s16_to_float(r) for r in raw])
        check_block(bank, orcs, fl, False, 1, f"pump, {plan.what}: call {k}")
    check_counters(bank, orcs, f"pump, {plan.what}")
    for b in (d_raw, d_psd, d_pk):
        b.free()
    f.close()
    bank.close()


# (rate, taps or None, s16, shared input): binary32 banks go to the streaming kernel (8 or more channels)
F32_CASES = {
    "f32-27x10-s16": (96000, None, True, False),
    "f32-27x20-float": (192000, None, False, False),
    "f32-64x20-s16-shared": (192000, 64, True, True),
}


@pytest.mark.parametrize("case", list(F32_CASES))
def test_binary32_decimator_within_its_bound_through_the_boundaries(ctx, sm_count, case):
    """JSDR_PREC_F32 keeps the reference's table index sequence and mixes and filters in binary32: every
    output of every channel within the bound derived in tests/f32_bound.py, which a wrong index at any
    tap of 3e-4 or more would leave."""
    rate, ntaps, s16, shared = F32_CASES[case]
    D = rate // 9600
    plan = T.bank_plan(rate, s16=s16, sm_count=sm_count)
    max_block = max(plan.lens)
    bank = J.FUNcubeBPSKDemod(ctx, None, J.AudioDescriptor(rate, blen=4 * max_block), tuning=plan.tunings[0],
                              max_block=max_block, stages=1)
    taps = O.default_taps()[0] if ntaps is None else lowpass(ntaps, D)
    if ntaps is not None:
        bank.set_ds_filter(taps)
    bank.set_precision(J.PREC_F32)
    orcs = [O.Bpsk(rate, float(t), ds_taps=None if ntaps is None else taps, stages=1) for t in plan.tunings[0]]
    bounds = [F.Bound(taps, D, s16) for _ in orcs]
    rng = np.random.default_rng(sum(map(ord, case)))
    rows = 1 if shared else plan.nchan
    worst = 0.0
    for k, n in enumerate(plan.lens):
        retune(bank, orcs, plan, k)
        data, fl = input_block(rng, rows, n, s16, 0, 0)
        if s16:
            bank.receive_raw(data[0] if shared else data, shared=shared)
        else:
            bank.receive(data[0] if shared else data, shared=shared)
        ds = bank.read_ds()
        for c, o in enumerate(orcs):
            x = fl[0 if shared else c]
            ref = o.receive(x)["ds"]
            b = bounds[c].block(x)
            assert ds[c].shape == ref.shape == b.shape, (case, k, c)
            r = np.abs(ds[c] - ref) / b
            worst = max(worst, float(r.max(initial=0.0)))
            assert np.all(r <= 1.0), f"{case}, {plan.what}: block {k} channel {c} (tuning {bank.tuning[c]!r} Hz), {r.max()} of the bound"
    print(f"\n{case}: worst error {worst:.3f} of the bound")
    bank.close()
