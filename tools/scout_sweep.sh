#!/bin/bash
# Sweep of the phase scout's shape on the pump step of BASELINE config 5 (4096 channels x
# 2^19 samples): CTA size (= warps per SM) and the shared-memory reservation that keeps two
# scout CTAs off one SM.  Prints the step time and the per-kernel event times (scout, FFT,
# tuner + decimator).  Output is committed as profiles/r02_scout_sweep.txt, which also has the
# rows for 2-4 chains per thread, a kernel form removed after commit 3563be3.
out=${1:-gpurun_out/scout_sweep.txt}
: > $out
run() {  # threads smem_kb
  sms=$(( (4096 + $1 - 1) / $1 ))
  echo -n "threads=$1 smem_kb=$2 SMs_held=$sms  " >> $out
  JSDR_SCOUT_THREADS=$1 JSDR_SCOUT_SMEM_KB=$2 python tools/kbench.py pump 2>&1 | tail -1 >> $out
}
for t in 64 128 160 192 224 256 320; do run $t 116; done
for t in 128 192 256; do run $t 88; done
for t in 128 256; do run $t 24; done
cat $out
