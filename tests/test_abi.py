"""CPU tests of the boundary: libjsdrcuda.so loads, exports every symbol
include/jsdrcuda.h declares, and fails loudly without a device (no compute calls)."""
import ctypes
import os
import re

import pytest

import jsdrcuda


def _declared():
    src = open(jsdrcuda.HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(jsdr_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = jsdrcuda.lib()
    names = _declared()
    assert len(names) >= 45
    for n in names:
        assert hasattr(lib, n), f"{n} declared in jsdrcuda.h but not exported"
    assert names == jsdrcuda.EXPORTS, "python binding and header disagree on the symbol list"
    assert lib.jsdr_abi_version() == 2


def test_no_cpu_fallback():
    """Without a CUDA device context creation must fail, not fall back.  In a child process
    that sees no device (CUDA_VISIBLE_DEVICES empty), so that a machine with a GPU checks it too."""
    import subprocess
    import sys
    code = r"""
import jsdrcuda as J
try:
    J.Context(0)
except J.JsdrError as e:
    print("REFUSED", e)
"""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="",
               PYTHONPATH=os.pathsep.join([os.path.dirname(os.path.dirname(jsdrcuda.__file__)), os.environ.get("PYTHONPATH", "")]))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0 and "REFUSED" in r.stdout, (r.returncode, r.stdout[-2000:], r.stderr[-2000:])


def test_host_side_helpers_need_no_device():
    import numpy as np
    assert jsdrcuda.fft_supported(4096) and jsdrcuda.fft_supported(19200) and not jsdrcuda.fft_supported(4097)
    w = np.empty(21)
    assert jsdrcuda.lib().jsdr_fir_design(500, 1500, ctypes.c_float(44100.0), w.ctypes.data_as(ctypes.c_void_p)) == 0
    import oracle as O
    assert np.array_equal(w, O.Fir(44100.0).weights(500, 1500))
    t = np.empty((44100, 2), dtype=np.int32)
    assert jsdrcuda.lib().jsdr_fir_nco_table(1000, ctypes.c_float(44100.0), t.ctypes.data_as(ctypes.c_void_p)) == 0
    assert np.array_equal(t[:64], O.Fir(44100.0).complex_gen(1000, 0, 64))


def test_product_does_not_touch_the_oracle():
    """The product path must not import, link or call anything under oracle/."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pkg = os.path.join(root, "java-sdr_b200")
    for dp, _, files in os.walk(pkg):
        if "build" in dp:
            continue
        for f in files:
            if f.endswith((".cu", ".cuh", ".h", ".hpp", ".cpp", ".py", ".java")):
                txt = open(os.path.join(dp, f), errors="replace").read()
                assert "orc_" not in txt and "jsdr_oracle" not in txt and "import oracle" not in txt, f


def test_null_handles_and_pointers_come_back_as_status_codes():
    """Every entry point called with null handles / null pointers and a range of scalar values
    answers a negative status (destroy of a null handle is a no-op): nothing dereferences before
    it checks.  In a child process, so that a crash is a failed assertion and not a dead run."""
    import subprocess
    import sys
    code = r"""
import ctypes as C, sys
import jsdrcuda as J
lib = J.lib()
bad = []
for iv in (0, 1, 2, 3, 21, 4096, -1, 2**31 - 1):
    for name, args in sorted(J._SIGS.items()):
        if name in ("jsdr_abi_version", "jsdr_fft_supported"):
            continue
        vals = []
        for a in args:
            if a in (C.c_float, C.c_double):
                vals.append(a(1000.0))
            elif a in (C.c_int, C.c_int64, C.c_uint32, C.c_size_t):
                vals.append(a(iv & 0xffffffff) if a is C.c_uint32 else a(max(iv, 0)) if a is C.c_size_t else a(iv))
            else:
                vals.append(None)
        rc = getattr(lib, name)(*vals)
        if not (rc < 0 or (rc == 0 and name.endswith("_destroy"))):
            bad.append((name, iv, rc))
        elif rc < 0 and not lib.jsdr_last_error():
            bad.append((name, iv, "no message"))
print("BAD", bad)
sys.exit(1 if bad else 0)
"""
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.dirname(os.path.dirname(jsdrcuda.__file__)), os.environ.get("PYTHONPATH", "")]))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, (r.returncode, r.stdout[-2000:], r.stderr[-2000:])


def test_demod_fir_multiply_and_add_stay_separately_rounded():
    """demod.java's filter() (:385-389) rounds the product and the sum of every tap separately.
    k_demod forms the two products of a tap with one packed multiply; ptxas contracts a packed
    multiply that feeds a packed add into FFMA2 (one rounding) whatever the flags, so the kernel
    adds in scalar form -- and this looks at the built library: packed multiplies present, no
    packed fused multiply-add anywhere in the kernel."""
    import shutil
    import subprocess
    if not shutil.which("cuobjdump"):
        pytest.skip("cuobjdump not on PATH")
    so = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "java-sdr_b200", "libjsdrcuda.so")
    sass = subprocess.run(["cuobjdump", "-sass", "-fun", "_ZN4jsdr3dsp7k_demodENS0_11DemodParamsE", so],
                          capture_output=True, text=True, timeout=300).stdout
    assert sass.count("FMUL2") >= 21 * 4, "k_demod's packed tap products are missing"
    assert "FFMA2" not in sass and "FADD2" not in sass
