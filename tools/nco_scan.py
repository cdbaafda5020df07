"""Exhaustive check of the NCO's own sine / cosine (nco_sincos, csrc/demod_fir.cu) over every float
in [-8, 8], the whole range it evaluates itself (beyond, it calls the CUDA library).

For every float: the kernel's float (tests/nco_phase.py: the binary64 chain with each FMA as a
multiply and an add, and every FMA exact for the values within BAND binary64 ulps of a float
midpoint) against the correctly rounded float (numpy's binary64 value, and mpmath at 200 bits for
the values within LIBM_BAND ulps of a midpoint).  Also counts the floats whose result changes when
the Cody-Waite reduction drops its second step (c_trig[14]).  Prints one summary; the result is
recorded in DESIGN.md section 4.5.  About 2.1e9 floats: a few minutes on 8 cores.

    python tools/nco_scan.py [--procs 8]
"""
import argparse
import os
import sys
import time
from multiprocessing import Pool

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "java-sdr_b200"), os.path.join(ROOT, "tests")]

import nco_phase as N  # noqa: E402

STEP = 1 << 22
TOP = int(np.float32(8.0).view(np.int32))


def no_tail(car):
    c = N.coefficients()
    x = car.astype(np.float64)
    kd = (x * c[12] + N.MAGIC) - N.MAGIC
    r = x - kd * c[13]
    z = r * r
    ps = np.full_like(z, c[5])
    for i in (4, 3, 2, 1, 0):
        ps = ps * z + c[i]
    pc = np.full_like(z, c[11])
    for i in (10, 9, 8, 7, 6):
        pc = pc * z + c[i]
    return N._quadrant(kd, r + (z * r) * ps, (1.0 - 0.5 * z) + (z * z) * pc)


def scan(job):
    lo, sign = job
    bits = np.arange(lo, min(lo + STEP, TOP + 1), dtype=np.int32)
    car = bits.view(np.float32) * np.float32(sign)
    stats = {}
    ks, kc = N.kernel_sincos(car, stats)
    cs, cc, _, _ = N.cr_sincos(car)
    bad = car[(ks != cs) | (kc != cc)]
    ws, wc = no_tail(car)
    _, fs, fc = N.chain_muladd(car)
    sure = ~(N.near_half(car) | (N.midpoint_ulps(fs) <= N.BAND) | (N.midpoint_ulps(fc) <= N.BAND))
    tail = int(np.sum(sure & ((ws != ks) | (wc != kc))))
    doubt_vals = car[N.near_half(car) | (N.midpoint_ulps(fs) <= N.BAND) | (N.midpoint_ulps(fc) <= N.BAND)]
    return car.size, doubt_vals.tolist(), bad.tolist(), tail


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--procs", type=int, default=os.cpu_count())
    a = ap.parse_args()
    jobs = [(lo, s) for s in (1, -1) for lo in range(0, TOP + 1, STEP)]
    t0 = time.time()
    total, doubt, bad, tail = 0, [], [], 0
    with Pool(a.procs) as p:
        for n, d, b, t in p.imap_unordered(scan, jobs):
            total += n
            doubt += d
            bad += b
            tail += t
    print(f"floats scanned in [-8, 8] (+0 and -0 both): {total}")
    print(f"doubtful (chain within {N.BAND} binary64 ulps of a float midpoint), resolved with exact FMAs: {len(doubt)}")
    print("  " + " ".join(f"{x:.9g}" for x in sorted(doubt)))
    print(f"kernel float != correctly rounded float: {len(bad)}" + ("  " + " ".join(f"{x:.9g}" for x in bad) if bad else ""))
    print(f"floats changed by dropping c_trig[14] (outside the doubt set): {tail}")
    print(f"{time.time() - t0:.0f} s")


if __name__ == "__main__":
    main()
