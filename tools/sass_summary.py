#!/usr/bin/env python
"""SASS opcode histogram and the hot loop of the step's kernels (cuobjdump -sass on the built
objects; no GPU needed).  Usage: python tools/sass_summary.py > profiles/r02_sass.txt"""
import collections
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "java-sdr_b200", "csrc", "build")
KERNELS = [
    ("fft_n4096.o", r"fft_kernelINS0_4PlanILi4096.*Li1ELi0E", "fft_kernel<Plan<4096,64,1,64,64>, IN_S16, OUT_PSD>"),
    ("bpsk.o", r"k_mixdecim_streamILi1ELi0ELi64ELi20ELi16E", "k_mixdecim_stream<S16, F64, 64 taps, D=20, 16 warps>"),
    ("bpsk.o", r"k_tuner_scoutEPK", "k_tuner_scout"),
    ("fec.o", r"k_fec_decode", "k_fec_decode"),
]
INS = re.compile(r"^\s+/\*([0-9a-f]{4,})\*/\s+(.*?);")


def function_sass(obj, pat):
    out = subprocess.run(["cuobjdump", "-sass", os.path.join(BUILD, obj)], capture_output=True, text=True).stdout
    cur, keep = None, []
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            continue
        if cur and re.search(pat, cur):
            mi = INS.match(line)
            if mi:
                keep.append((int(mi.group(1), 16), mi.group(2).strip()))
    return keep


def opcode(text):
    t = re.sub(r"^@!?U?P\d+\s+", "", text)
    return t.split()[0].split(".")[0]


def main():
    for obj, pat, title in KERNELS:
        ins = function_sass(obj, pat)
        print(f"==== {title}   ({obj}, {len(ins)} instructions)")
        hist = collections.Counter(opcode(t) for _, t in ins)
        print("  " + "  ".join(f"{k}:{v}" for k, v in hist.most_common(28)))
        blk = [t for _, t in ins if re.match(r"(@!?U?P\d+\s+)?(UBLK|UTMA|SYNCS|LDGSTS|REDUX|SHFL|VOTE|MATCH)", t)]
        if blk:
            print("  bulk-copy / warp-collective instructions: " + "; ".join(sorted(set(re.sub(r"\s+", " ", re.sub(r"^@!?U?P\d+\s+", "", b)).split(",")[0][:40] for b in blk))[:16]))
        # the hot loop: the backward branch that spans the most floating-point instructions
        best = None
        for i, (addr, t) in enumerate(ins):
            m = re.search(r"BRA(?:\.U)?\s+(?:!?U?P\d+,\s*)?0x([0-9a-f]+)", t)
            if not m:
                continue
            tgt = int(m.group(1), 16)
            if tgt >= addr:
                continue
            body = [x for a, x in ins if tgt <= a <= addr]
            fp = sum(1 for x in body if re.match(r"(@!?U?P\d+\s+)?(F(ADD|MUL|FMA)2?|D(ADD|MUL|FMA)|DSETP)", x))
            if best is None or fp > best[0]:
                best = (fp, tgt, addr, body)
        if best:
            fp, tgt, addr, body = best
            h2 = collections.Counter(opcode(t) for t in body)
            print(f"  hot loop 0x{tgt:x}..0x{addr:x}: {len(body)} instructions, {fp} floating-point; mix: " +
                  "  ".join(f"{k}:{v}" for k, v in h2.most_common(14)))
            print("  first 24 instructions of the loop:")
            for t in body[:24]:
                print("      " + re.sub(r"\s+", " ", t))
        print()


if __name__ == "__main__":
    main()
