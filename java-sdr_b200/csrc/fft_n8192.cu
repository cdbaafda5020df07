// generated per-length instantiation (see fft_plans.h)
#include "fft_inst.cuh"
JSDR_FFT_DEFINE(8192, 256, 1, 32, 16, 16, 1)
