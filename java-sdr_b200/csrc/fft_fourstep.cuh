// fft_fourstep.cuh — FFT + PSD for block lengths that do not fit one CTA's shared
// memory (32768 = 128 x 256, 65536 = 256 x 256), the top of BASELINE config 3's sweep.
//
// N = N1*N2, n = n1*N2 + n2, k = k1 + N1*k2 (the "four-step" factorisation):
//   k_fs_cols   for every n2: N1-point transform over n1 (stride N2), times w_N^(n2*k1),
//               stored transposed as Z[k1][n2];
//   k_fs_rows   for every k1: N2-point transform over n2 (a contiguous row of Z), then the
//               fft.java:199-211 epilogue on bins k1 + N1*k2.
// Both kernels give a CTA 16 neighbouring sub-transforms (16 x 256 or 16 x 128 points, two
// register passes through shared memory, the same radix-16 butterflies as fft_kernels.cuh),
// and every global access of a warp is 16 neighbouring n2 (or k1): 64..128 contiguous bytes.
// The host runs the pair over chunks of blocks small enough for Z to stay in L2, so HBM
// still sees the input once and the PSD once.
#pragma once

#include "fft_kernels.cuh"

namespace jsdr {
namespace fft {

struct FsArgs {
    const void *in;        // [nblocks][N] float2 or s16x2 (first block of this chunk)
    float2 *z;             // [nblocks][N1][N2] intermediate
    float *out;            // [nblocks][N+2] PSD or [nblocks][N] float2 spectrum (first block of this chunk)
    unsigned long long *best;   // [nblocks] packed (ordered dB key << 32 | ~bin), reset to 0 before the chunk
    const float2 *tw;      // exp(-2*pi*i*t/N), t in [0, N)
    int nblocks;
    float cf, db_off;
    int ic, qc;
    const float *win;      // [N] window of jsdr_fft_set_window, read by k_fs_cols<..., true> only
};

constexpr int kFsPitch = 18;                     // float2 per 16-element row (16 + 2 pad)
constexpr int kFsGroup = 16 * kFsPitch + 2;      // float2 per sub-transform (16 rows + 2 pad)

template <int IN>
__device__ __forceinline__ float2 fs_load(const FsArgs &a, long idx)
{
    if constexpr (IN == IN_F32) {
        return ldg_stream_f2(reinterpret_cast<const float2 *>(a.in) + idx);
    } else {
        uint32_t w = ldg_stream_u32(reinterpret_cast<const uint32_t *>(a.in) + idx);
        if (a.ic | a.qc)
            w = (((w & 0xffffu) + (unsigned)a.ic) & 0xffffu) | ((((w >> 16) + (unsigned)a.qc) & 0xffffu) << 16);
        w ^= 0x80008000u;
        const float fi = __uint_as_float(__byte_perm(w, 0x4b000000u, 0x7410)) - 8421376.0f;
        const float fq = __uint_as_float(__byte_perm(w, 0x4b000000u, 0x7432)) - 8421376.0f;
        return make_float2(fi, fq);
    }
}

// grid = nblocks * N2/16 CTAs of 256 threads; thread = (g = n2 within the CTA's 16, c)
// WIN: each sample times a.win[t] as it is loaded (apply_win, fft_kernels.cuh).  Left alone, ptxas
// holds the 16 window values beside the 16 samples and the CTAs per SM drop by one (N1 = 256: 48
// -> 50..54 registers, four CTAs instead of five); the bound keeps the CTAs per SM of the
// unwindowed kernel: five, six for N1 = 128 with float input (40 registers there).
template <int N1, int IN>
constexpr int fs_cols_win_ctas() { return (N1 == 128 && IN == IN_F32) ? 6 : 5; }
template <int N1, int N2, int IN, bool WIN = false>
__global__ void __launch_bounds__(256, WIN ? fs_cols_win_ctas<N1, IN>() : 0) k_fs_cols(const FsArgs a)
{
    constexpr int N = N1 * N2, R1 = N1 / 16;
    __shared__ __align__(16) float2 sm[16 * kFsGroup];
    const int tid = threadIdx.x, g = tid & 15, c = tid >> 4;
    const long vb = (long)blockIdx.x * 16;
    const long blk = vb / N2;
    const int n2 = (int)(vb - blk * N2) + g;
    const long base = blk * (long)N;
    if (c < R1) {                                  // pass 0: x[(c + m*R1)*N2 + n2], m < 16
        float2 v[16];
#pragma unroll
        for (int m = 0; m < 16; m++) v[m] = fs_load<IN>(a, base + (long)(c + m * R1) * N2 + n2);
        if constexpr (WIN) {
#pragma unroll
            for (int m = 0; m < 16; m++) v[m] = apply_win(v[m], a.win, (c + m * R1) * N2 + n2);
        }
        Dft<16>::run(v);
        float4 *dst = reinterpret_cast<float4 *>(sm + g * kFsGroup + c * kFsPitch);
#pragma unroll
        for (int m = 0; m < 8; m++) dst[m] = make_float4(v[2 * m].x, v[2 * m].y, v[2 * m + 1].x, v[2 * m + 1].y);
    }
    __syncthreads();
    {                                              // last pass: j = c, outputs k1 = j + 16q
        const int j = c;
        float2 v[R1];
        const float2 *p = sm + g * kFsGroup + j;
#pragma unroll
        for (int r = 0; r < R1; r++) v[r] = p[r * kFsPitch];
        twiddle_powers<R1>(v, __ldg(a.tw + j * (N / N1)));
        Dft<R1>::run(v);
        // times w_N^(n2*k1) = w_N^(n2*j) * (w_N^(16*n2))^q
        float2 w = __ldg(a.tw + n2 * j);
        const float2 step = __ldg(a.tw + 16 * n2);
        float2 *z = a.z + (blk * (long)N1 + j) * N2 + n2;
#pragma unroll
        for (int q = 0; q < R1; q++) {
            z[(long)q * 16 * N2] = cmul(v[q], w);
            w = cmul(w, step);
        }
    }
}

// grid = nblocks * N1/16 CTAs of 256 threads; pass 0 with n2 fastest (contiguous rows of Z),
// last pass with k1 fastest (contiguous bins)
template <int N1, int N2, int OUT>
__global__ void __launch_bounds__(256) k_fs_rows(const FsArgs a)
{
    static_assert(N2 == 256, "rows are 16 x 16");
    constexpr int N = N1 * N2;
    __shared__ __align__(16) float2 sm[16 * kFsGroup];
    __shared__ unsigned long long s_best;
    const int tid = threadIdx.x;
    const long vb = (long)blockIdx.x * 16;
    const long blk = vb / N1;
    const int k1_0 = (int)(vb - blk * N1);
    if (tid == 0) s_best = 0ull;
    {
        const int g = tid >> 4, c = tid & 15;
        const float2 *row = a.z + (blk * (long)N1 + k1_0 + g) * N2;
        float2 v[16];
#pragma unroll
        for (int m = 0; m < 16; m++) v[m] = row[c + 16 * m];
        Dft<16>::run(v);
        float4 *dst = reinterpret_cast<float4 *>(sm + g * kFsGroup + c * kFsPitch);
#pragma unroll
        for (int m = 0; m < 8; m++) dst[m] = make_float4(v[2 * m].x, v[2 * m].y, v[2 * m + 1].x, v[2 * m + 1].y);
    }
    __syncthreads();
    const int g = tid & 15, j = tid >> 4;
    const int k1 = k1_0 + g;
    float2 v[16];
    const float2 *p = sm + g * kFsGroup + j;
#pragma unroll
    for (int r = 0; r < 16; r++) v[r] = p[r * kFsPitch];
    twiddle_powers<16>(v, __ldg(a.tw + j * (N / N2)));
    Dft<16>::run(v);
    if constexpr (OUT == OUT_SPECTRUM) {
        float2 *spec = reinterpret_cast<float2 *>(a.out) + blk * (long)N;
#pragma unroll
        for (int q = 0; q < 16; q++) stg_stream_f2(spec + k1 + (long)N1 * (j + 16 * q), v[q]);
    } else {
        float *psd = a.out + blk * (long)(N + 2);
        float best = -3.4028234663852886e38f;
        int best_k = 0x7fffffff;
#pragma unroll
        for (int q = 0; q < 16; q++) {
            const float pw = fmaf(v[q].x, v[q].x, v[q].y * v[q].y);
            const float db = fmaf(3.0102999566398120f, lg2_approx(pw), a.db_off);
            const int k = k1 + N1 * (j + 16 * q);
            stg_stream_f32(psd + k, db);
            if (best < db) {                       // k increases with q: the first maximum wins
                best = db;
                best_k = k;
            }
        }
        // first strict maximum over the block (fft.java:208-211): highest dB, lowest bin among equals
        unsigned long long key = (best_k == 0x7fffffff) ? 0ull
                               : (((unsigned long long)ordered_key(best) << 32) | (unsigned)(0x7fffffff - best_k));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
            key = other > key ? other : key;
        }
        if ((tid & 31) == 0 && key != 0ull) atomicMax(&s_best, key);
        __syncthreads();
        if (tid == 0 && s_best != 0ull) atomicMax(a.best + blk, s_best);
    }
}

// psd[N], psd[N+1], peak_bin from the packed maximum (fft.java:214-224)
__global__ void __launch_bounds__(128) k_fs_finish(const unsigned long long *__restrict__ best, float *__restrict__ out,
                                                   int32_t *__restrict__ peak_bin, int N, int rate, int nblocks)
{
    const int blk = blockIdx.x * blockDim.x + threadIdx.x;
    if (blk >= nblocks) return;
    const unsigned long long key = best[blk];
    float *psd = out + (long)blk * (N + 2);
    int bin = -1;
    float m = -3.4028234663852886e38f;
    if (key != 0ull) {
        bin = 0x7fffffff - (int)(unsigned)(key & 0xffffffffu);
        const unsigned k = (unsigned)(key >> 32);
        m = __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
    }
    int p = (bin < 0) ? -1 : 2 * bin;              // int32 wrap, truncating division
    const int datlen = 2 * N;
    if (p >= datlen / 2) p -= datlen;
    p = (int)((unsigned)p * (unsigned)rate) / datlen;
    psd[N] = (float)p;
    psd[N + 1] = m;
    if (peak_bin) peak_bin[blk] = bin;
}

}  // namespace fft
}  // namespace jsdr
