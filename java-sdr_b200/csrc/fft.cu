// fft.cu — host side of the fft.java replacement (jsdr_fft_* in jsdrcuda.h).
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <memory>
#include <vector>

#include "fft_fourstep.cuh"
#include "fft_generic.cuh"
#include "fft_kernels.cuh"
#include "fft_plans.h"
#include "handles.h"

namespace jsdr {
namespace fft {

#define DECL(N, T, G, R0, R1, R2, R3)                                                         \
    int launch_n##N(jsdr_ctx *ctx, const Args &a, int in_fmt, int out_mode, cudaStream_t st); \
    size_t smem_n##N();
JSDR_FFT_PLANS(DECL)
#undef DECL

int launch_split_n16384(jsdr_ctx *ctx, const Args &a, int in_fmt, int out_mode, cudaStream_t st);

typedef int (*launch_fn)(jsdr_ctx *, const Args &, int, int, cudaStream_t);
struct PlanEntry { int n; launch_fn fn; };
static const PlanEntry kPlans[] = {
#define ROW(N, T, G, R0, R1, R2, R3) {N, launch_n##N},
    JSDR_FFT_PLANS(ROW)
#undef ROW
};

static const PlanEntry *find_plan(int n)
{
    for (const PlanEntry &p : kPlans)
        if (p.n == n) return &p;
    return nullptr;
}


// Lengths that run as a split plan: two CTAs per block, each an n/2-point plan behind one
// radix-2 decimation-in-frequency step folded into its loads (fft_kernel, SPLIT = 2).
// Measured (profiles/r02_fft_split.txt): 32768 as 2 x 16384 beats the four-step pair (0.278 / 0.424
// against 0.256 / 0.355 of peak for s16 / float input); 16384 as 2 x 8192 and 19200 as 2 x 9600 do
// not beat their whole-block plans (the second read and conversion of every sample and the
// strided stores cost what the second CTA per SM gains).
static launch_fn split_plan(int n) { return n == 32768 ? launch_split_n16384 : nullptr; }

// ---- lengths without a single-CTA plan: fft_generic.cuh stages + a PSD pass -------------
// WIN: sample i times win[i mod n] (apply_win, fft_kernels.cuh)
template <bool WIN>
__global__ void __launch_bounds__(256) k_generic_load(const void *__restrict__ in, float2 *__restrict__ out, long long total,
                                                     int in_fmt, int ic, int qc, const float *__restrict__ win, int n)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    if (in_fmt == IN_F32) {
        out[i] = reinterpret_cast<const float2 *>(in)[i];
    } else {
        const uint32_t w = reinterpret_cast<const uint32_t *>(in)[i];
        // JavaAudio.java:281-288: s += (short)ic with 16-bit wrap; the 1/32767 is folded into cf
        const short si = (short)((int)(w & 0xffffu) + ic), sq = (short)((int)(w >> 16) + qc);
        out[i] = make_float2((float)si, (float)sq);
    }
    if constexpr (WIN) out[i] = apply_win(out[i], win, (int)(i % n));
}

// fft.java:199-224 on a finished spectrum: one CTA per block
__global__ void __launch_bounds__(256) k_generic_psd(const float2 *__restrict__ spec, float *__restrict__ out,
                                                    int32_t *__restrict__ peak_bin, int N, int rate, float db_off)
{
    __shared__ unsigned s_max;
    __shared__ int s_idx;
    const long blk = blockIdx.x;
    const float2 *x = spec + blk * (long)N;
    float *psd = out + blk * (long)(N + 2);
    if (threadIdx.x == 0) {
        s_max = 0u;
        s_idx = 0x7fffffff;
    }
    __syncthreads();
    float best = -3.4028234663852886e38f;
    int best_idx = 0x7fffffff;
    for (int k = threadIdx.x; k < N; k += blockDim.x) {
        const float2 v = x[k];
        const float pw = fmaf(v.x, v.x, v.y * v.y);
        const float db = fmaf(3.0102999566398120f, lg2_approx(pw), db_off);
        psd[k] = db;
        if (best < db) {           // k increases per thread: the first maximum wins
            best = db;
            best_idx = k;
        }
    }
    const unsigned key = (best_idx == 0x7fffffff) ? 0u : ordered_key(best);
    if (key != 0u) atomicMax(&s_max, key);
    __syncthreads();
    if (key != 0u && key == s_max) atomicMin(&s_idx, best_idx);
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned k = s_max;
        const int bin = (k != 0u) ? s_idx : -1;
        float m = -3.4028234663852886e38f;
        if (k != 0u) m = __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
        int p = (bin < 0) ? -1 : 2 * bin;              // fft.java:214-221, int32 wrap, truncating division
        const int datlen = 2 * N;
        if (p >= datlen / 2) p -= datlen;
        p = (int)((unsigned)p * (unsigned)rate) / datlen;
        psd[N] = (float)p;
        psd[N + 1] = m;
        if (peak_bin) peak_bin[blk] = bin;
    }
}


// ---- 32768 / 65536: the four-step pair (fft_fourstep.cuh), chunked so that Z stays in L2 ----
template <int N1, int IN, int OUT, bool WIN>
static int launch_fourstep_chunk(jsdr_ctx *ctx, const FsArgs &fa, cudaStream_t st)
{
    constexpr int N2 = 256;
    {
        ProfScope prof(ctx, JSDR_K_FFT, st);
        k_fs_cols<N1, N2, IN, WIN><<<(unsigned)((long)fa.nblocks * (N2 / 16)), 256, 0, st>>>(fa);
        JSDR_TRY(launched(ctx, "k_fs_cols"));
    }
    ProfScope prof(ctx, JSDR_K_FFT, st);
    k_fs_rows<N1, N2, OUT><<<(unsigned)((long)fa.nblocks * (N1 / 16)), 256, 0, st>>>(fa);
    return launched(ctx, "k_fs_rows");
}

template <int N1, bool WIN>
static int launch_fourstep_fmt(jsdr_ctx *ctx, const FsArgs &fa, int in_fmt, int out_mode, cudaStream_t st)
{
    if (out_mode == OUT_SPECTRUM) return launch_fourstep_chunk<N1, IN_F32, OUT_SPECTRUM, WIN>(ctx, fa, st);
    if (in_fmt == IN_F32) return launch_fourstep_chunk<N1, IN_F32, OUT_PSD, WIN>(ctx, fa, st);
    return launch_fourstep_chunk<N1, IN_S16, OUT_PSD, WIN>(ctx, fa, st);
}

static int launch_fourstep(jsdr_fft *f, const Args &a, int in_fmt, int out_mode, cudaStream_t st)
{
    jsdr_ctx *ctx = f->ctx;
    const int N = f->n, N1 = f->fs_n1;
    static int chunk_mb = 0;
    if (!chunk_mb) {
        const char *e = getenv("JSDR_FS_CHUNK_MB");             // (tuning aid) size of Z per chunk
        // 32 MB: two chunks of Z plus their input and PSD stay inside the 126 MB L2 (measured on
        // N = 65536: 8 MB 0.17, 16 MB 0.25, 24 MB 0.30, 32 MB 0.32, 48 MB 0.28 of peak)
        chunk_mb = e ? std::max(1, atoi(e)) : 32;
    }
    const int chunk = std::max(1, std::min(f->max_batch, (int)(((long)chunk_mb << 20) / ((long)N * 8))));
    if (!f->work.best) {
        jsdr_fft::Work w;
        JSDR_TRY(w.z[0].alloc((size_t)chunk * N * sizeof(float2), "fft workspace"));
        JSDR_TRY(w.z[1].alloc((size_t)chunk * N * sizeof(float2), "fft workspace"));
        JSDR_TRY(w.best.alloc(sizeof(unsigned long long) * (size_t)f->max_batch, "fft workspace"));
        f->work = std::move(w);
    }
    unsigned long long *best = f->work.best.get();
    if (out_mode == OUT_PSD)
        JSDR_CUDA(cudaMemsetAsync(best, 0, sizeof(unsigned long long) * (size_t)a.nblocks, st));
    // Chunks alternate between two streams (and two Z buffers): while one chunk's row kernel
    // drains, the next chunk's column kernel already fills the SMs.
    const bool two = a.nblocks > chunk && st != ctx->aux;
    if (two) {
        JSDR_CUDA(cudaEventRecord(ctx->ev_aux_fork, st));
        JSDR_CUDA(cudaStreamWaitEvent(ctx->aux, ctx->ev_aux_fork, 0));
    }
    const size_t in_el = (in_fmt == IN_S16) ? 4 : 8;
    int ci = 0;
    for (int b0 = 0; b0 < a.nblocks; b0 += chunk, ci++) {
        cudaStream_t cs = (two && (ci & 1)) ? ctx->aux : st;
        FsArgs fa;
        fa.nblocks = std::min(chunk, a.nblocks - b0);
        fa.in = reinterpret_cast<const char *>(a.in) + (size_t)b0 * N * in_el;
        fa.z = f->work.z[ci & 1].get();
        fa.out = (out_mode == OUT_PSD) ? a.out + (size_t)b0 * (N + 2) : a.out + (size_t)b0 * N * 2;
        fa.best = best + b0;
        fa.tw = a.tw;
        fa.cf = a.cf;
        fa.db_off = a.db_off;
        fa.ic = a.ic;
        fa.qc = a.qc;
        fa.win = a.win;
        int rc;
        if (fa.win) {
            rc = (N1 == 128) ? launch_fourstep_fmt<128, true>(ctx, fa, in_fmt, out_mode, cs)
                             : launch_fourstep_fmt<256, true>(ctx, fa, in_fmt, out_mode, cs);
        } else {
            rc = (N1 == 128) ? launch_fourstep_fmt<128, false>(ctx, fa, in_fmt, out_mode, cs)
                             : launch_fourstep_fmt<256, false>(ctx, fa, in_fmt, out_mode, cs);
        }
        JSDR_TRY(rc);
    }
    if (two) {
        JSDR_CUDA(cudaEventRecord(ctx->ev_aux_join, ctx->aux));
        JSDR_CUDA(cudaStreamWaitEvent(st, ctx->ev_aux_join, 0));
    }
    if (out_mode == OUT_PSD) {
        k_fs_finish<<<(a.nblocks + 127) / 128, 128, 0, st>>>(best, a.out, a.peak_bin, N, a.rate, a.nblocks);
        JSDR_TRY(launched(ctx, "k_fs_finish"));
    }
    return JSDR_OK;
}

static int launch_generic(jsdr_fft *f, const Args &a, int in_fmt, int out_mode, cudaStream_t st)
{
    jsdr_ctx *ctx = f->ctx;
    const size_t need = (size_t)f->max_batch * (size_t)f->n * sizeof(float2);
    if (!f->work.z[0]) {
        jsdr_fft::Work w;
        JSDR_TRY(w.z[0].alloc(need, "fft workspace"));
        JSDR_TRY(w.z[1].alloc(need, "fft workspace"));
        f->work = std::move(w);
    }
    float2 *z0 = f->work.z[0].get(), *z1 = f->work.z[1].get();
    const long long total = (long long)a.nblocks * f->n;
    const unsigned grid = (unsigned)((total + 255) / 256);
    if (a.win) k_generic_load<true><<<grid, 256, 0, st>>>(a.in, z0, total, in_fmt, a.ic, a.qc, a.win, f->n);
    else k_generic_load<false><<<grid, 256, 0, st>>>(a.in, z0, total, in_fmt, a.ic, a.qc, nullptr, f->n);
    JSDR_TRY(launched(ctx, "k_generic_load"));
    int rc = JSDR_OK;
    float2 *res = fftg::run<float>(ctx, st, z0, z1, f->n, a.nblocks, -1, &rc);
    if (rc != JSDR_OK) return rc;
    if (out_mode == OUT_SPECTRUM) {
        JSDR_CUDA(cudaMemcpyAsync(a.out, res, (size_t)total * sizeof(float2), cudaMemcpyDeviceToDevice, st));
        return JSDR_OK;
    }
    k_generic_psd<<<a.nblocks, 256, 0, st>>>(res, a.out, a.peak_bin, f->n, a.rate, a.db_off);
    return launched(ctx, "k_generic_psd");
}

int launch(jsdr_fft *f, const void *d_in, int in_fmt, int batch, float *d_out, int32_t *d_peak,
           int out_mode, int ic, int qc, cudaStream_t st)
{
    Args a;
    a.in = d_in;
    a.out = d_out;
    a.peak_bin = d_peak;
    a.tw = f->d_tw.get();
    a.nblocks = batch;
    a.rate = f->rate;
    // fft.java:199-200  cf = 2f/(float)N; cf = cf*cf  (float arithmetic)
    float cf = 2.0f / (float)f->n;
    cf = cf * cf;
    if (in_fmt == IN_S16) {
        // JavaAudio.java:283 divides each sample by 32767f before the transform;
        // the transform is linear, so the scale moves into cf.
        cf = (float)((double)cf / (32767.0 * 32767.0));
    }
    a.cf = cf;
    a.db_off = (float)(10.0 * log10((double)cf));
    a.ic = ic;
    a.qc = qc;
    a.pf_dist = 0;
    a.tw2 = nullptr;
    a.best = nullptr;
    a.cnt = nullptr;
    a.win = f->win_on ? f->d_win.get() : nullptr;
    if (out_mode == OUT_SPECTRUM && in_fmt != IN_F32) {
        set_error("spectrum output needs float input");
        return JSDR_EINVAL;
    }
    if (f->split) {
        a.nblocks = 2 * batch;                    // half blocks
        a.tw2 = f->d_tw2.get();
        a.best = f->d_best.get();
        a.cnt = f->d_cnt.get();
        return reinterpret_cast<launch_fn>(f->launch)(f->ctx, a, in_fmt, out_mode, st);
    }
    if (f->fs_n1) return launch_fourstep(f, a, in_fmt, out_mode, st);
    if (!f->launch) return launch_generic(f, a, in_fmt, out_mode, st);
    return reinterpret_cast<launch_fn>(f->launch)(f->ctx, a, in_fmt, out_mode, st);
}

}  // namespace fft
}  // namespace jsdr

using namespace jsdr;

extern "C" int jsdr_fft_supported(int n)
try {
    if (fft::find_plan(n) || fft::split_plan(n)) return 1; // single-CTA plan (whole or split)
    if (n == 32768 || n == 65536) return 3;                // four-step pair
    return n >= 2 && fftg::make_plan(n).nstages > 0 ? 2 : 0;   // staged path (slower)
} JSDR_CATCH_ALL

extern "C" int jsdr_fft_create(jsdr_ctx *ctx, int n, int rate, int max_batch, jsdr_fft **out)
try {
    JSDR_REQUIRE(ctx && out, JSDR_EINVAL, "null argument");
    JSDR_REQUIRE(max_batch > 0 && rate > 0, JSDR_EINVAL, "max_batch and rate must be positive");
    const fft::PlanEntry *p = fft::find_plan(n);
    if (!p && !(n >= 2 && fftg::make_plan(n).nstages > 0)) {
        set_error("jsdr_fft_create: no FFT plan for n=%d (needs n = 2^a 3^b 5^c 7^d)", n);
        return JSDR_EUNSUPPORTED;
    }
    JSDR_TRY(ctx->bind());
    const char *what = "jsdr_fft_create";
    std::unique_ptr<jsdr_fft> f(new jsdr_fft(ctx));
    f->n = n;
    f->rate = rate;
    f->max_batch = max_batch;
    f->launch = p ? reinterpret_cast<void *>(p->fn) : nullptr;   // null: four-step or the staged path
    if (fft::launch_fn sp = fft::split_plan(n)) {
        f->launch = reinterpret_cast<void *>(sp);
        f->split = 2;
    }
    f->fs_n1 = (!f->launch && n == 32768) ? 128 : (!f->launch && n == 65536) ? 256 : 0;
    // twiddle table exp(-2*pi*i*t/m) of the transform the plan runs (m = n, or n/2 for a split
    // plan), computed in double, rounded once
    const int m = f->split ? n / f->split : n;
    std::vector<float2> tw(m);
    for (int t = 0; t < m; t++) {
        double ang = 2.0 * M_PI * (double)t / (double)m;
        tw[t] = make_float2((float)cos(ang), (float)-sin(ang));
    }
    JSDR_TRY(f->d_tw.alloc(sizeof(float2) * m, what));
    JSDR_CUDA(cudaMemcpyAsync(f->d_tw.get(), tw.data(), sizeof(float2) * m, cudaMemcpyHostToDevice, ctx->stream));
    if (f->split) {                                              // the radix-2 step's twiddles and the halves' meeting point
        for (int t = 0; t < m; t++) {
            double ang = 2.0 * M_PI * (double)t / (double)n;
            tw[t] = make_float2((float)cos(ang), (float)-sin(ang));
        }
        JSDR_TRY(f->d_tw2.alloc(sizeof(float2) * m, what));
        JSDR_CUDA(cudaMemcpyAsync(f->d_tw2.get(), tw.data(), sizeof(float2) * m, cudaMemcpyHostToDevice, ctx->stream));
        JSDR_TRY(f->d_best.alloc_zeroed(sizeof(unsigned long long) * (size_t)max_batch, ctx->stream, what));
        JSDR_TRY(f->d_cnt.alloc_zeroed(sizeof(unsigned) * (size_t)max_batch, ctx->stream, what));
    }
    JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
    *out = f.release();
    return JSDR_OK;
} JSDR_CATCH_ALL

// The window is checked whole before anything is enqueued.  The first window is uploaded into a
// buffer of its own that is installed only once the copy is enqueued; later ones are copied over
// it on the context's stream, so that every call enqueued before this one keeps the window it was
// enqueued with and every call after it sees the new one.  Removing the window keeps the buffer.
extern "C" int jsdr_fft_set_window(jsdr_fft *f, const float *win)
try {
    JSDR_REQUIRE(f, JSDR_EINVAL, "null handle");
    if (!win) {
        f->win_on = false;
        return JSDR_OK;
    }
    for (int t = 0; t < f->n; t++) {
        if (!isfinite(win[t])) {
            set_error("jsdr_fft_set_window: win[%d] = %g is not finite", t, (double)win[t]);
            return JSDR_EINVAL;
        }
    }
    jsdr_ctx *ctx = f->ctx;
    JSDR_TRY(ctx->bind());
    const size_t bytes = sizeof(float) * (size_t)f->n;
    if (f->d_win) {
        JSDR_CUDA(cudaMemcpyAsync(f->d_win.get(), win, bytes, cudaMemcpyHostToDevice, ctx->stream));
    } else {
        DevBuf<float> w;
        JSDR_TRY(w.alloc(bytes, "fft window"));
        JSDR_CUDA(cudaMemcpyAsync(w.get(), win, bytes, cudaMemcpyHostToDevice, ctx->stream));
        f->d_win = std::move(w);
    }
    f->win_on = true;
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_fft_destroy(jsdr_fft *f)
try {
    delete f;
    return JSDR_OK;
} JSDR_CATCH_ALL

int jsdr::fft::ensure_staging(jsdr_fft *f, size_t in_bytes, size_t out_bytes)
{
    JSDR_TRY(f->d_in.grow(in_bytes, "fft staging"));
    JSDR_TRY(f->d_out.grow(out_bytes, "fft staging"));
    return f->d_peak.grow(sizeof(int32_t) * (size_t)f->max_batch, "fft staging");
    return JSDR_OK;
}

namespace {

// shared body of the three receive flavours
int fft_run(jsdr_fft *f, const void *in, int in_fmt, int batch, int ic, int qc, float *out,
            int32_t *peak_bin, int out_mode, int mem)
{
    JSDR_REQUIRE(f && in && out, JSDR_EINVAL, "null argument");
    JSDR_REQUIRE(batch >= 0 && batch <= f->max_batch, JSDR_EINVAL, "batch exceeds max_batch");
    JSDR_REQUIRE(mem == JSDR_MEM_HOST || mem == JSDR_MEM_DEVICE, JSDR_EINVAL, "bad mem");
    if (batch == 0) return JSDR_OK;   // empty input: nothing to publish
    jsdr_ctx *ctx = f->ctx;
    JSDR_TRY(ctx->bind());
    const size_t n = (size_t)f->n;
    const size_t in_bytes = (size_t)batch * n * (in_fmt == fft::IN_S16 ? 4 : 8);
    const size_t out_elems = (size_t)batch * (out_mode == fft::OUT_PSD ? n + 2 : 2 * n);
    if (mem == JSDR_MEM_DEVICE) {
        return fft::launch(f, in, in_fmt, batch, out, peak_bin, out_mode, ic, qc, ctx->stream);
    }
    JSDR_TRY(fft::ensure_staging(f, in_bytes, out_elems * sizeof(float)));
    JSDR_CUDA(cudaMemcpyAsync(f->d_in.get(), in, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    JSDR_TRY(fft::launch(f, f->d_in.get(), in_fmt, batch, f->d_out.get(), f->d_peak.get(), out_mode, ic, qc, ctx->stream));
    JSDR_CUDA(cudaMemcpyAsync(out, f->d_out.get(), out_elems * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (peak_bin && out_mode == fft::OUT_PSD)
        JSDR_CUDA(cudaMemcpyAsync(peak_bin, f->d_peak.get(), sizeof(int32_t) * (size_t)batch,
                                  cudaMemcpyDeviceToHost, ctx->stream));
    JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
    return JSDR_OK;
}

}  // namespace

extern "C" int jsdr_fft_receive_f32(jsdr_fft *f, const float *iq, int batch, float *psd,
                                    int32_t *peak_bin, int mem)
try {
    return fft_run(f, iq, fft::IN_F32, batch, 0, 0, psd, peak_bin, fft::OUT_PSD, mem);
} JSDR_CATCH_ALL

extern "C" int jsdr_fft_receive_s16(jsdr_fft *f, const int16_t *raw, int batch, int ic, int qc,
                                    float *psd, int32_t *peak_bin, int mem)
try {
    return fft_run(f, raw, fft::IN_S16, batch, ic, qc, psd, peak_bin, fft::OUT_PSD, mem);
} JSDR_CATCH_ALL

extern "C" int jsdr_fft_forward_f32(jsdr_fft *f, const float *iq, int batch, float *spec, int mem)
try {
    return fft_run(f, iq, fft::IN_F32, batch, 0, 0, spec, nullptr, fft::OUT_SPECTRUM, mem);
} JSDR_CATCH_ALL
