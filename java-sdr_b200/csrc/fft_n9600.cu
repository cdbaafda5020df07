// generated per-length instantiation (see fft_plans.h)
#include "fft_inst.cuh"
JSDR_FFT_DEFINE(9600, 320, 1, 32, 20, 15, 1)
