"""The sample bench.py --dump-outputs takes (no GPU): at the benchmark's default shape and at
shapes whose single rows exceed a file's budget, every file stays inside its budget, the budgets
with their .npy headers stay under 64 MB, and the sample is the same on every call."""
import numpy as np
import pytest

import bench


def test_budgets_leave_room_for_the_headers():
    assert sum(bench.DUMP_BUDGET.values()) + 3 * 4096 <= 64e6


# (channels, blocks, N): the default step, the reference's N = rate/10, one long block per channel,
# and single blocks whose PSD row alone is larger than the whole dump
@pytest.mark.parametrize("nchan,nblk,n", [(4096, 128, 4096), (4096, 27, 19200), (256, 1, 1 << 21),
                                          (1, 1, 1 << 28), (2, 1, 1 << 27)])
def test_dump_plan_stays_inside_its_budget(nchan, nblk, n):
    batch, nds = nchan * nblk, nblk * n // bench.D + 1
    plan = bench.dump_plan(batch, n, nchan, nds)
    again = bench.dump_plan(batch, n, nchan, nds)
    full = {"psd": (batch, n + 2), "peak_bin": (batch, 1), "ds": (nchan, nds)}
    for k, (rows, cols, size) in plan.items():
        nrows, ncols = full[k]
        assert rows.size >= 1 and 1 <= cols <= ncols, k
        assert rows.size * cols * size <= bench.DUMP_BUDGET[k], k
        assert np.all(np.diff(rows) > 0) and 0 <= rows[0] and rows[-1] < nrows, k
        assert np.array_equal(rows, again[k][0]) and cols == again[k][1], k
    if (nchan, nblk, n) == (4096, 128, 4096):      # the default shape fills every budget
        assert plan["peak_bin"][0].size == batch and plan["psd"][1] == n + 2 and plan["ds"][1] == nds
        for k, (rows, cols, size) in plan.items():
            assert rows.size * cols * size > 0.95 * bench.DUMP_BUDGET[k], k
