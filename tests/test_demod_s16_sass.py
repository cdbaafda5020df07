"""k_demod_s16 runs the same FIR as k_demod after its conversion, so it keeps the same rule: the two
products of a tap as one packed multiply (FMUL2), no packed fused multiply-add or packed add that
would round once where demod.java's filter() (:385-389) rounds twice.  Reads the built library;
no device needed."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "java-sdr_b200", "libjsdrcuda.so")


def kernel_sass(symbol):
    if not shutil.which("cuobjdump"):
        pytest.skip("cuobjdump not on PATH")
    if not os.path.exists(SO):
        pytest.skip("libjsdrcuda.so is not built")
    return subprocess.run(["cuobjdump", "-sass", "-fun", symbol, SO], capture_output=True, text=True, timeout=300).stdout


def test_s16_fir_keeps_products_and_sums_separately_rounded():
    sass = kernel_sass("_ZN4jsdr3dsp11k_demod_s16ENS0_11DemodParamsE")
    assert "Function" in sass, "k_demod_s16 is missing from the library"
    assert sass.count("FMUL2") >= 21 * 4, "k_demod_s16's packed tap products are missing"
    assert "FFMA2" not in sass and "FADD2" not in sass
