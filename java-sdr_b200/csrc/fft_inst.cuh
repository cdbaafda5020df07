// fft_inst.cuh — one translation unit per FFT length includes this with
// JSDR_FFT_N etc. defined, so the plans compile in parallel.
#pragma once
#include <algorithm>

#include "fft_kernels.cuh"

namespace jsdr {
namespace fft {

template <class P, int IN, int OUT, int SPLIT, bool WIN>
static int launch_one(jsdr_ctx *ctx, const Args &a, cudaStream_t st)
{
    static PerDeviceFlag attr_done;
    auto kern = fft_kernel<P, IN, OUT, SPLIT, WIN>;
    constexpr size_t smem = (P::PERSIST && IN == IN_S16 && SPLIT == 1) ? P::SMEM_PERSIST
                          : (P::TW_SMEM_NP && SPLIT == 1) ? P::SMEM_TW : P::SMEM;   // + twiddle tables
    JSDR_TRY(attr_done.once(ctx->device, [&]() -> int {
        JSDR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        return JSDR_OK;
    }));
    int grid = (a.nblocks + P::G - 1) / P::G;
    if (grid <= 0) return JSDR_OK;
    static int per_sm = 0;                        // a property of the kernel and sm_100a, not of the device index
    if (!per_sm) {
        JSDR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, P::T, smem));
        per_sm = std::max(1, per_sm);
    }
    Args b = a;
    if constexpr (P::PERSIST && IN == IN_S16 && SPLIT == 1) grid = std::min(grid, per_sm * ctx->sm_count);   // resident CTAs loop over the blocks
    else b.pf_dist = ctx->l2_prefetch * per_sm * ctx->sm_count;                // L2 look-ahead distance in CTAs
    ProfScope prof(ctx, JSDR_K_FFT, st);
    kern<<<grid, P::T, smem, st>>>(b);
    return launched(ctx, "fft_kernel");
}

template <class P, int SPLIT, bool WIN>
static int launch_fmt(jsdr_ctx *ctx, const Args &a, int in_fmt, int out_mode, cudaStream_t st)
{
    if (out_mode == OUT_SPECTRUM) {
        if (in_fmt != IN_F32) { set_error("spectrum output needs float input"); return JSDR_EINVAL; }
        return launch_one<P, IN_F32, OUT_SPECTRUM, SPLIT, WIN>(ctx, a, st);
    }
    if (in_fmt == IN_F32) return launch_one<P, IN_F32, OUT_PSD, SPLIT, WIN>(ctx, a, st);
    return launch_one<P, IN_S16, OUT_PSD, SPLIT, WIN>(ctx, a, st);
}

// a handle with a window (a.win set) runs the windowed instantiations of the same plan
template <class P, int SPLIT = 1>
static int launch_plan(jsdr_ctx *ctx, const Args &a, int in_fmt, int out_mode, cudaStream_t st)
{
    return a.win ? launch_fmt<P, SPLIT, true>(ctx, a, in_fmt, out_mode, st)
                 : launch_fmt<P, SPLIT, false>(ctx, a, in_fmt, out_mode, st);
}

}  // namespace fft
}  // namespace jsdr

#define JSDR_FFT_DEFINE(N, T, G, R0, R1, R2, R3)                                               \
    namespace jsdr { namespace fft {                                                           \
    int launch_n##N(jsdr_ctx *ctx, const Args &a, int in_fmt, int out_mode, cudaStream_t st)   \
    {                                                                                          \
        return launch_plan<Plan<N, T, G, R0, R1, R2, R3>>(ctx, a, in_fmt, out_mode, st);       \
    }                                                                                          \
    size_t smem_n##N() { return Plan<N, T, G, R0, R1, R2, R3>::SMEM; }                         \
    } }

// the same plan as a split plan: blocks of 2N samples, two CTAs per block (fft_kernel, SPLIT = 2)
#define JSDR_FFT_DEFINE_SPLIT(N, T, G, R0, R1, R2, R3)                                                \
    namespace jsdr { namespace fft {                                                                  \
    int launch_split_n##N(jsdr_ctx *ctx, const Args &a, int in_fmt, int out_mode, cudaStream_t st)    \
    {                                                                                                 \
        return launch_plan<Plan<N, T, G, R0, R1, R2, R3>, 2>(ctx, a, in_fmt, out_mode, st);           \
    }                                                                                                 \
    } }
