"""The Java side cannot be compiled here (no JDK), so what can be checked mechanically is:
every FFM downcall descriptor in JsdrCuda.java names an exported symbol and has the argument
count and the scalar/pointer kinds of the C ABI (taken from the ctypes signatures, which
tests/test_abi.py ties to include/jsdrcuda.h); the patches against the reference are
insert-only and well-formed; and, given a java-sdr checkout in JAVA_SDR_REFERENCE, they apply
cleanly.  The upstream sources themselves are not vendored in this repository."""
import os
import re
import shutil
import subprocess

import pytest

import jsdrcuda as J

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
JAVA = os.path.join(ROOT, "java-sdr_b200", "java")
SRC = os.path.join(JAVA, "com", "ashbysoft", "java_sdr")
REF = os.environ.get("JAVA_SDR_REFERENCE", "")


def _descriptors():
    txt = open(os.path.join(SRC, "JsdrCuda.java")).read()
    out = {}
    for m in re.finditer(r'h\("(jsdr_\w+)",\s*FunctionDescriptor\.of\(([^;]*?)\)\)\s*;', txt, flags=re.S):
        args = [a.strip() for a in m.group(2).split(",")]
        out[m.group(1)] = args
    return out


def test_ffm_descriptors_match_the_c_abi():
    import ctypes as C
    desc = _descriptors()
    assert len(desc) >= 25
    kind = {C.c_int: "JAVA_INT", C.c_int64: "JAVA_LONG", C.c_double: "JAVA_DOUBLE", C.c_float: "JAVA_FLOAT",
            C.c_size_t: "JAVA_LONG", C.c_uint32: "JAVA_INT"}
    for name, args in desc.items():
        assert name in J.EXPORTS, f"{name} is not an exported symbol"
        if name == "jsdr_last_error":
            assert args == ["ADDRESS"]
            continue
        sig = J._SIGS[name]
        assert args[0] == "JAVA_INT", f"{name}: status return"
        assert len(args) - 1 == len(sig), f"{name}: {len(args) - 1} Java arguments, {len(sig)} in the ABI"
        for a, c in zip(args[1:], sig):
            assert a == kind.get(c, "ADDRESS"), f"{name}: {a} vs {c}"


def test_helpers_only_call_bound_entry_points():
    bound = {m for m in re.findall(r"static final MethodHandle (\w+) =", open(os.path.join(SRC, "JsdrCuda.java")).read())}
    for f in ("CudaFft.java", "CudaFUNcubeBPSKDemod.java"):
        used = set(re.findall(r"JsdrCuda\.([A-Z][A-Z0-9_]+)\.invokeExact", open(os.path.join(SRC, f)).read()))
        assert used and used <= bound, f"{f}: unbound {used - bound}"


def test_patches_are_insert_only():
    for f in ("fft.java.patch", "FUNcubeBPSKDemod.java.patch", "FECDecoder.java.patch"):
        body = [l for l in open(os.path.join(JAVA, "patches", f)).read().splitlines() if not l.startswith(("---", "+++"))]
        assert any(l.startswith("+") for l in body)
        assert not any(l.startswith("-") for l in body), f"{f} removes reference lines"


def test_patch_hunks_are_well_formed():
    """What patch(1) checks before it reads the file it patches: every hunk holds exactly the
    lines its header counts, and each hunk's new start is its old start shifted by the lines
    the hunks before it insert."""
    for f in ("fft.java.patch", "FUNcubeBPSKDemod.java.patch", "FECDecoder.java.patch"):
        lines = open(os.path.join(JAVA, "patches", f)).read().splitlines()
        assert lines[0].startswith("--- ") and lines[1].startswith("+++ "), f
        i, shift, hunks = 2, 0, 0
        while i < len(lines):
            m = re.fullmatch(r"@@ -(\d+)(?:,(\d+))? \+(\d+)(?:,(\d+))? @@.*", lines[i])
            assert m, f"{f}:{i + 1}: expected a hunk header"
            o0, oc, n0, nc = int(m[1]), int(m[2] or 1), int(m[3]), int(m[4] or 1)
            assert n0 == o0 + shift, f"{f}:{i + 1}: new start {n0}, expected {o0 + shift}"
            i += 1
            ro, rn = oc, nc
            while ro > 0 or rn > 0:
                assert i < len(lines), f"{f}: hunk ends early"
                tag = lines[i][:1] or " "            # an empty line is blank context
                assert tag in " +-", f"{f}:{i + 1}: not a hunk line"
                ro -= tag != "+"
                rn -= tag != "-"
                assert ro >= 0 and rn >= 0, f"{f}:{i + 1}: more lines than the header counts"
                i += 1
            shift += nc - oc
            hunks += 1
        assert hunks, f


@pytest.mark.skipif(not os.path.isdir(REF) or shutil.which("patch") is None, reason="needs a java-sdr checkout in JAVA_SDR_REFERENCE")
def test_patches_apply_to_the_reference(tmp_path):
    for f in ("fft.java", "FUNcubeBPSKDemod.java", "FECDecoder.java"):
        shutil.copy(os.path.join(REF, f), tmp_path / f)
        r = subprocess.run(["patch", "-p1", "-i", os.path.join(JAVA, "patches", f + ".patch")], cwd=tmp_path,
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        txt = (tmp_path / f).read_text()
        assert txt.count("{") == txt.count("}")
    # every private field cudaFetch() assigns is declared by the reference class
    fun = (tmp_path / "FUNcubeBPSKDemod.java").read_text()
    fetch = fun[fun.index("private void cudaFetch()"):fun.index("private void doBufferTune")]
    for field in set(re.findall(r"^\s*(\w+)(?:\[[^\]]*\])?\s*=[^=]", fetch, flags=re.M)):
        if field in ("int", "nds", "at"):
            continue
        assert re.search(r"\b(private|int|double|boolean)\b[^;\n]*\b" + field + r"\b", fun.replace(fetch, "")), field
