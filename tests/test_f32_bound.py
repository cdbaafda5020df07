"""The binary32 decimator's per-output bound (tests/f32_bound.py): it accepts a numpy binary32 emulation of
the kernel's arithmetic and rejects one wrong table index at every tap above a stated size.  No GPU
needed; tests/test_gpu_tuner_index.py, test_gpu_stream.py and test_gpu_fuzz.py hold the GPU to it."""
import numpy as np
import pytest

import f32_bound as F
import oracle as O

THRESHOLD = 3e-4          # |h_k| above which one wrong index at tap k is outside the bound (|x| >= 1/2)


def lowpass(ntaps, D):
    h = np.sinc((np.arange(ntaps) - (ntaps - 1) / 2) * 0.9 / D) * np.hamming(ntaps)
    return h / h.sum()


def drawn(rng, n, s16, lo=0.0):
    """n IQ samples with |I|, |Q| in [lo, 1]: (kernel input, the reference's floats)."""
    mag = rng.uniform(lo, 1.0, (n, 2)) * rng.choice([-1.0, 1.0], (n, 2))
    if s16:
        raw = np.round(mag * 32767).astype(np.int16)
        return raw.astype(np.float64), O.s16_to_float(raw.ravel()).reshape(n, 2).astype(np.float64)
    x = mag.astype(np.float32)
    return x, x.astype(np.float64)


SHAPES = [(27, 10, None), (27, 20, None), (64, 20, "lowpass"), (40, 5, "lowpass")]


@pytest.mark.parametrize("s16", [True, False])
@pytest.mark.parametrize("ntaps,D,kind", SHAPES)
def test_bound_accepts_the_binary32_emulation(ntaps, D, kind, s16):
    taps = O.default_taps()[0] if kind is None else lowpass(ntaps, D)
    rng = np.random.default_rng(ntaps * 100 + D + s16)
    n = 40000
    x, xref = drawn(rng, n, s16)
    idx = rng.integers(0, 257, n)
    y = F.reference(xref, idx, taps, D)
    got = F.kernel_f32(x, idx, taps, D, s16)
    b = F.Bound(taps, D, s16)
    bound = np.vstack([b.block(xref[i:i + 7777].ravel()) for i in range(0, n, 7777)])   # carried across blocks
    assert bound.shape == y.shape
    ratio = np.abs(got - y) / bound
    print(f"\n{ntaps} taps, D = {D}, s16 = {s16}: worst error / bound = {ratio.max():.3f}")
    assert ratio.max() <= 1.0
    assert ratio.max() > 0.01           # the bound is not loose by orders of magnitude


@pytest.mark.parametrize("s16", [True, False])
@pytest.mark.parametrize("ntaps,D,kind", SHAPES)
def test_bound_rejects_one_wrong_index_at_every_tap_above_the_threshold(ntaps, D, kind, s16):
    """One output in every NQ + 1 gets a wrong index (the next table entry) at tap k and nowhere else;
    every such output must leave the bound, for every tap with |h_k| >= THRESHOLD."""
    taps = O.default_taps()[0] if kind is None else lowpass(ntaps, D)
    rng = np.random.default_rng(7 + ntaps + D + s16)
    n = 30000
    x, xref = drawn(rng, n, s16, lo=0.5)
    idx = rng.integers(0, 256, n)
    y = F.reference(xref, idx, taps, D)
    b = F.Bound(taps, D, s16).block(xref.ravel())
    outs = np.arange(D - 1, n, D)
    step = (ntaps + D - 1) // D + 1
    big = np.nonzero(np.abs(taps) >= THRESHOLD)[0]
    for k in big:
        sel = np.arange(step, outs.size, step)
        bad = idx.copy()
        bad[outs[sel] - k] = (bad[outs[sel] - k] + 1) % 256
        got = F.kernel_f32(x, bad, taps, D, s16)
        out = np.any(np.abs(got[sel] - y[sel]) > b[sel], axis=1)
        assert out.all(), (k, taps[k], int((~out).sum()))
    print(f"\n{ntaps} taps: a wrong index is seen at {big.size} of {ntaps} taps (|h_k| >= {THRESHOLD})")
    if kind is None:
        assert big.size == 25
