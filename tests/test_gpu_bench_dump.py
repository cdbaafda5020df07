"""bench.py --dump-outputs: the same arguments give the same inputs and so the same files, the
files hold what the last timed step computed (the decimated channels against the oracle, the PSD
rows against the fft handler), and --steps sets the number of timed steps.  The size bound is
checked without a GPU (test_bench_dump_plan.py)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import jsdrcuda as J
import oracle as O
from jsdrcuda import sharding

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NCH, NBLK, N, WARMUP = 64, 2, 4096, 1


def run_bench(steps, dump=None):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--main-only", "--channels", str(NCH), "--blocks", str(NBLK),
           "--fft-n", str(N), "--steps", str(steps), "--warmup", str(WARMUP)]
    if dump is not None:
        cmd += ["--dump-outputs", str(dump)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])


def test_dump_is_reproducible_and_from_the_last_step(ctx, tmp_path):
    a, b = tmp_path / "a", tmp_path / "b"
    l2 = run_bench(2, a)
    run_bench(2, b)
    l4 = run_bench(4)
    assert l4["gpu_launches"] == 2 * l2["gpu_launches"] > 0
    names = sorted(os.listdir(a))
    assert names == sorted(os.listdir(b)) == ["ds.npy", "peak_bin.npy", "psd.npy"]
    out = {f[:-4]: np.load(a / f) for f in names}
    for f in names:
        assert out[f[:-4]].dtype in (np.float32, np.float64)
        assert np.array_equal(out[f[:-4]], np.load(b / f)), f

    S = NBLK * N
    tile = bench.synth_tile(NCH, S, 1000)
    tuning = sharding.channel_tuning(0, NCH)
    taps = J.design_lowpass(64, 4800.0, bench.RATE)
    # the decimator's state runs on through the warm-up and timed steps over the same batch, so
    # these rows tell the last step from any other
    orc = {}
    for c in range(NCH):
        o = O.Bpsk(bench.RATE, tuning[c], ds_taps=taps, stages=1)
        for _ in range(WARMUP + 2):
            orc[c] = o.receive(O.s16_to_float(tile[c]))["ds"]
    plan = bench.dump_plan(NCH * NBLK, N, NCH, orc[0].shape[0])
    rows, cols, _ = plan["ds"]
    assert out["ds"].shape == (rows.size, cols, 2)
    for i, c in enumerate(rows):
        assert np.array_equal(out["ds"][i], orc[int(c)][:cols]), int(c)
    # PSD rows [channel * NBLK + block] and peak bins against the fft handler on the host path: this
    # shows the right rows were taken, not which step they came from (the PSD keeps no state)
    f = J.fft(ctx, None, J.AudioDescriptor(bench.RATE), max_batch=NCH * NBLK, n=N)
    psd, pk = f.receive_batch(tile.reshape(NCH * NBLK, 2 * N), s16=True)
    f.close()
    rows, cols, _ = plan["psd"]
    assert np.array_equal(out["psd"], psd[rows, :cols])
    rows, _, _ = plan["peak_bin"]
    assert np.array_equal(out["peak_bin"], pk[rows].astype(np.float64))
