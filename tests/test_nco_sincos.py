"""The NCO's sine / cosine as k_demod evaluates them (java-sdr_b200/csrc/demod_fir.cu, nco_sincos):
one Cody-Waite step by k*pi/2 and two minimax kernels on [-pi/4, pi/4] in binary64, rounded to float
as demod.java:425-426 does with Math.cos / Math.sin.  The coefficients are read out of the CUDA
source, the routine is restated in numpy binary64 (fused multiply-adds become a multiply and an add:
a difference of an ulp of binary64, far below the float rounding this test looks at) and compared
with libm over the phase range of the recurrence (:427-429) and beyond it up to the routine's own
limit.  No GPU needed; tests/test_nco_model.py holds the same routine to exact arithmetic and the
correctly rounded float, and tests/test_gpu_nco.py the kernel to that model."""
import os
import re

import numpy as np

SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "java-sdr_b200", "csrc", "demod_fir.cu")


def coefficients():
    txt = open(SRC).read()
    body = re.search(r"__constant__ double c_trig\[15\] = \{(.*?)\};", txt, re.S).group(1)
    c = [float(x) for x in re.findall(r"-?\d+\.\d+(?:e[+-]?\d+)?", body)]
    assert len(c) == 15
    return c


def nco_sincos(car: np.ndarray):
    c = coefficients()
    x = car.astype(np.float64)
    magic = 6755399441055744.0
    t = x * c[12] + magic
    kd = t - magic
    k = kd.astype(np.int64)
    r = (x - kd * c[13]) - kd * c[14]
    z = r * r
    ps = np.full_like(z, c[5])
    for i in (4, 3, 2, 1, 0):
        ps = ps * z + c[i]
    pc = np.full_like(z, c[11])
    for i in (10, 9, 8, 7, 6):
        pc = pc * z + c[i]
    fs = (r + (z * r) * ps).astype(np.float32)
    fc = ((1.0 - 0.5 * z) + (z * z) * pc).astype(np.float32)
    a = np.where(k & 1, fc, fs)
    b = np.where(k & 1, fs, fc)
    return np.where(k & 2, -a, a), np.where((k + 1) & 2, -b, b), np.abs(r).max()


def test_coefficients_are_the_classic_kernels():
    c = coefficients()
    assert c[0] == -1.66666666666666324348e-01 and c[5] == 1.58969099521155010221e-10
    assert c[6] == 4.16666666666666019037e-02 and c[11] == -1.13596475577881948265e-11
    assert c[12] == 2.0 / np.pi and c[13] == np.pi / 2 and abs(c[13] + c[14] - np.pi / 2) < 1e-16


def test_float_results_equal_libm():
    rng = np.random.default_rng(425)
    twopi = np.float32(2 * np.pi)
    car = np.concatenate([
        rng.uniform(0, float(twopi), 1_500_000).astype(np.float32),           # the recurrence's range
        rng.uniform(-8, 8, 500_000).astype(np.float32),                       # the routine's whole domain
        np.array([0.0, twopi, np.pi / 2, np.pi, 3 * np.pi / 2, np.pi / 4, 8.0, -8.0, 1e-30, 1e-6], np.float32),
        (np.arange(0, 21, dtype=np.float32) * np.float32(np.pi / 4)).astype(np.float32)[:11],
    ])
    sn, cs, rmax = nco_sincos(car)
    assert rmax <= np.pi / 4 + 1e-7
    ref_s = np.sin(car.astype(np.float64)).astype(np.float32)
    ref_c = np.cos(car.astype(np.float64)).astype(np.float32)
    # binary64 results within an ulp of libm's can round to different floats about once in 2^28
    # samples; on these two million they do not
    assert np.array_equal(sn, ref_s)
    assert np.array_equal(cs, ref_c)
