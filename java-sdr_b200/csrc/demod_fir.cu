// demod_fir.cu — the FIR + NCO parts of demod.java (:341-434) and the four
// arithmetic methods of fir.java (:169-228), batched over channels.
//
// demod.java works in binary32 with a multiply and an add rounded separately
// per tap (filter(), :385-389) and a float phase accumulator (:424-429);
// __fmul_rn/__fadd_rn keep that order and never contract.  fir.java multiplies int
// samples by double taps and truncates the double sum to int (:202-210).
#include <limits.h>
#include <math.h>
#include <string.h>

#include <type_traits>
#include <vector>

#include "handles.h"

namespace jsdr {
namespace dsp {

constexpr int kChunk = 32;          // samples between NCO phase checkpoints
constexpr int kTile = 1024;         // samples per CTA
constexpr int kDemodOut = 4;        // consecutive outputs per thread of k_demod (kTile = kDemodOut * kThreads)
constexpr int kThreads = 256;
constexpr int kTaps = 21, kHist = 20;

// ------------------------------------------------------------------ demod.java
// car is a sequential float accumulator (:427-429), data independent: replay it
// once per channel and leave the value seen by every kChunk-th sample.
__global__ void k_car_scout(const float *__restrict__ phi_, float *__restrict__ car_,
                            float *__restrict__ chunk_car, int nchan, int S)
{
    int ch = blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= nchan) return;
    float car = car_[ch];
    const float phi = phi_[ch];
    const float twopi = (float)(2 * M_PI);
    int nchunks = (S + kChunk - 1) / kChunk;
    for (int c = 0; c < nchunks; c++) {
        chunk_car[(size_t)c * nchan + ch] = car;
        int steps = min(kChunk, S - c * kChunk);
        for (int s = 0; s < steps; s++) {
            car = __fsub_rn(car, phi);
            if (car < 0.0f) car = __fadd_rn(car, twopi);
        }
    }
    car_[ch] = car;
}

// Per-half multiply of an (I, Q) pair (one FMUL2), each half rounded exactly as the scalar
// __fmul_rn.  The additions that follow stay scalar __fadd_rn on purpose: ptxas contracts a
// mul.rn.f32x2 feeding an add.rn.f32x2 into one FFMA2 -- with -fmad=false as well, and even when both
// are written as explicit fma.rn.f32x2 (a*b + -0, then p*1 + c); seen in the SASS -- which would
// round once where filter() (:385-389) rounds twice.  It leaves FMUL2 + FADD alone
// (tests/test_abi.py looks for FFMA2 in the built k_demod).
__device__ __forceinline__ float2 mul2(float2 a, float2 b)
{
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(*reinterpret_cast<unsigned long long *>(&a)), "l"(*reinterpret_cast<unsigned long long *>(&b)));
    return *reinterpret_cast<float2 *>(&r);
}

// (float)Math.sin(car), (float)Math.cos(car) for the NCO (:425-426).  For 0 <= phi < 2 pi car stays
// in [0, 2 pi] (:427-429), where the binary64 sine and cosine need no large-argument path: one
// Cody-Waite step by k*(pi/2) (|k| <= 5, the product is exact inside the fma), the two minimax
// kernels of the classic binary64 libm on [-pi/4, pi/4], quadrant by selects on the rounded floats.
// Over every float in [-8, 8] the float results equal the correctly rounded sin and cos
// (tools/nco_scan.py; tests/test_nco_model.py, tests/test_gpu_nco.py).  Coefficients sit in
// constant memory and enter the DFMAs as operands; the library's sincos() spent as many
// instructions moving its constants into uniform registers and testing for its slow path as on
// arithmetic.  Arguments beyond |x| <= 8 and NaN go to the library, out of line: car reaches them
// for flo < 0 (phi < 0: car grows until car - phi rounds back to car, near 2^24 |phi|) and for
// flo > rate (phi > 2 pi: car runs negative), as in the reference.
__constant__ double c_trig[15] = {
    -1.66666666666666324348e-01, 8.33333333332248946124e-03, -1.98412698298579493134e-04,
    2.75573137070700676789e-06, -2.50507602534068634195e-08, 1.58969099521155010221e-10,
    4.16666666666666019037e-02, -1.38888888888741095749e-03, 2.48015872894767294178e-05,
    -2.75573143513906633035e-07, 2.08757232129817482790e-09, -1.13596475577881948265e-11,
    0.6366197723675814, 1.5707963267948966, 6.123233995736766e-17};

__device__ __noinline__ void nco_sincos_any(float car, float *sn_out, float *cs_out)
{
    double ds, dc;
    sincos((double)car, &ds, &dc);
    *sn_out = (float)ds;
    *cs_out = (float)dc;
}

__device__ __forceinline__ void nco_sincos(float car, float *sn_out, float *cs_out)
{
    const double x = (double)car;
    if (!(fabsf(car) <= 8.0f)) {
        nco_sincos_any(car, sn_out, cs_out);
        return;
    }
    const double magic = 6755399441055744.0;                       // 1.5 * 2^52: nearest integer in the low word
    const double t = __fma_rn(x, c_trig[12], magic);
    const int k = __double2loint(t);
    const double kd = __dsub_rn(t, magic);
    double r = __fma_rn(-kd, c_trig[13], x);
    r = __fma_rn(-kd, c_trig[14], r);
    const double z = __dmul_rn(r, r);
    double ps = __fma_rn(z, c_trig[5], c_trig[4]);
    ps = __fma_rn(z, ps, c_trig[3]);
    ps = __fma_rn(z, ps, c_trig[2]);
    ps = __fma_rn(z, ps, c_trig[1]);
    ps = __fma_rn(z, ps, c_trig[0]);
    const float fs = (float)__fma_rn(__dmul_rn(z, r), ps, r);
    double pc = __fma_rn(z, c_trig[11], c_trig[10]);
    pc = __fma_rn(z, pc, c_trig[9]);
    pc = __fma_rn(z, pc, c_trig[8]);
    pc = __fma_rn(z, pc, c_trig[7]);
    pc = __fma_rn(z, pc, c_trig[6]);
    const float fc = (float)__fma_rn(__dmul_rn(z, z), pc, __fma_rn(z, -0.5, 1.0));
    const float a = (k & 1) ? fc : fs, b = (k & 1) ? fs : fc;     // sin, cos of r + k*pi/2
    *sn_out = (k & 2) ? -a : a;
    *cs_out = ((k + 1) & 2) ? -b : b;
}

struct DemodParams {
    const void *in;            // float2 IQ, or s16 (I, Q) words for k_demod_s16
    long long chan_stride;
    int S, nchan;
    const float *w;            // [nchan][21]
    const float *phi;
    const float *chunk_car;
    const float2 *hist_in;     // [nchan][20], entry k is local sample k-20 (converted floats)
    float2 *hist_out;
    float2 *out;               // [nchan][S]
    int dofir, dodwn;
    int ic, qc;                // s16 input: JavaAudio's I/Q corrections (JavaAudio.java:281-288)
};

// Input sample n >= 0 of channel row `src` as the float IQ demod.receive sees: the f32 row
// itself, or the s16 word converted as JavaAudio does before it calls its handlers.
template <bool S16>
__device__ __forceinline__ float2 demod_input(const DemodParams &p, const void *src, int n)
{
    if constexpr (S16) return s16_iq_to_float2(static_cast<const uint32_t *>(src)[n], p.ic, p.qc);
    else return static_cast<const float2 *>(src)[n];
}

template <bool S16>
__device__ __forceinline__ const void *demod_row(const DemodParams &p, int ch)
{
    using T = typename std::conditional<S16, uint32_t, float2>::type;
    return static_cast<const T *>(p.in) + (long long)ch * p.chan_stride;
}

// k_demod and k_demod_s16: the input form only changes how a sample is staged into sX (each
// sample is converted once there, not once per tap); the FIR and the NCO see floats either way.
template <bool S16>
__device__ __forceinline__ void demod_tile(const DemodParams &p)
{
    __shared__ __align__(16) float2 sX[kTile + kHist + 4];   // (+4: the last thread's 128-bit reads stay inside)
    __shared__ float sCar[kTile + kTile / kChunk];
    __shared__ float sW[kTaps];
    const int tid = threadIdx.x, ch = blockIdx.y;
    const int t0 = blockIdx.x * kTile;
    const int cnt = min(kTile, p.S - t0);
    const void *src = demod_row<S16>(p, ch);
    if (tid < kTaps) sW[tid] = p.w[ch * kTaps + tid];
    for (int i = tid; i < cnt + kHist; i += kThreads) {
        int n = t0 - kHist + i;
        sX[i] = (n < 0) ? p.hist_in[(size_t)ch * kHist + kHist + n] : demod_input<S16>(p, src, n);
    }
    if (p.dodwn) {
        // one thread per checkpoint chunk replays car (:427-429); padded so lanes
        // (32 samples apart) do not share a bank
        const float phi = p.phi[ch];
        const float twopi = (float)(2 * M_PI);
        const int nch = (cnt + kChunk - 1) / kChunk;
        if (tid < nch) {
            float car = p.chunk_car[(size_t)(t0 / kChunk + tid) * p.nchan + ch];
            int steps = min(kChunk, cnt - tid * kChunk);
            for (int s = 0; s < steps; s++) {
                sCar[tid * (kChunk + 1) + s] = car;        // value used by this sample (:425-426)
                car = __fsub_rn(car, phi);
                if (car < 0.0f) car = __fadd_rn(car, twopi);
            }
        }
    }
    __syncthreads();
    float2 *dst = p.out + (size_t)ch * p.S + t0;
    // One thread = kDemodOut consecutive outputs (second session of round 2; one output per thread
    // and 21 shared-memory loads each before): the window of kDemodOut + 20 samples is read once,
    // 128 bits at a time, and the accumulations run side by side, each in the reference's tap order.
    constexpr int R = kDemodOut;
    static_assert(kTile == R * kThreads, "one round per tile");
    const int i0 = tid * R;
    if (i0 >= cnt) return;
    float si[R], sq[R];
    if (p.dofir) {
        // filter() :385-389 — newest sample first, w[0..20]; the two products of a tap as one packed multiply
        float2 x[R + kHist];
        const float4 *s4 = reinterpret_cast<const float4 *>(sX + i0);     // (sX is 16-byte aligned, i0 a multiple of 4)
#pragma unroll
        for (int i = 0; i < (R + kHist) / 2; i++) {
            const float4 v = s4[i];
            x[2 * i] = make_float2(v.x, v.y);
            x[2 * i + 1] = make_float2(v.z, v.w);
        }
#pragma unroll
        for (int r = 0; r < R; r++) si[r] = sq[r] = 0.0f;
#pragma unroll
        for (int k = 0; k < kTaps; k++) {
            const float w = sW[k];
            const float2 w2 = make_float2(w, w);
#pragma unroll
            for (int r = 0; r < R; r++) {
                const float2 pr = mul2(x[r + kHist - k], w2);
                si[r] = __fadd_rn(si[r], pr.x);
                sq[r] = __fadd_rn(sq[r], pr.y);
            }
        }
    } else {
#pragma unroll
        for (int r = 0; r < R; r++) {
            si[r] = sX[i0 + r + kHist].x;
            sq[r] = sX[i0 + r + kHist].y;
        }
    }
#pragma unroll
    for (int r = 0; r < R; r++) {
        const int i = i0 + r;
        if (i >= cnt) break;
        if (p.dodwn) {
            float car = sCar[(i / kChunk) * (kChunk + 1) + (i % kChunk)];
            float ci, cq;                                  // :425-426 (float)Math.cos(car), (float)Math.sin(car):
            nco_sincos(car, &cq, &ci);                     // one argument reduction for both
            float a = si[r], b = sq[r];
            si[r] = __fsub_rn(__fmul_rn(a, ci), __fmul_rn(b, cq));   // :432
            sq[r] = __fadd_rn(__fmul_rn(a, cq), __fmul_rn(b, ci));   // :433
        }
        dst[i] = make_float2(si[r], sq[r]);
    }
}

__global__ void __launch_bounds__(kThreads) k_demod(const DemodParams p) { demod_tile<false>(p); }
__global__ void __launch_bounds__(kThreads) k_demod_s16(const DemodParams p) { demod_tile<true>(p); }

// The delay line holds converted floats whatever the input form, so that s16 and f32 blocks
// may alternate on one handle.
template <bool S16>
__global__ void k_demod_tail(const DemodParams p)
{
    const int ch = blockIdx.x, k = threadIdx.x;
    if (k >= kHist) return;
    const void *src = demod_row<S16>(p, ch);
    int n = p.S - kHist + k;
    p.hist_out[(size_t)ch * kHist + k] = (n < 0) ? p.hist_in[(size_t)ch * kHist + k + p.S] : demod_input<S16>(p, src, n);
}

// ------------------------------------------------------------------ fir.java
struct FirParams {
    const int32_t *in;
    long long chan_stride;
    int S;
    const double *w;           // [nchan][21]
    const int32_t *hist_in;    // [nchan][20]
    int32_t *hist_out;
    int32_t *out;              // [nchan][S]
};

// One thread = kFirOut consecutive outputs: it reads its window of kFirOut + 20 samples once
// (128-bit loads where the row allows it; neighbouring windows overlap in L1), converts each sample
// to binary64 once, and runs the kFirOut accumulations side by side, each in the reference's order
// k = 0 .. 20 (:202-206).  (The first form gave every output its own 21 shared-memory loads and 21
// int -> double conversions: 0.92 ms per 2^27 samples, bound by the LSU and the conversion pipe,
// not by the 42 binary64 operations per output.)
constexpr int kFirOut = 8;
__global__ void __launch_bounds__(kThreads) k_fir_i32(const FirParams p)
{
    __shared__ double sW[kTaps];
    const int tid = threadIdx.x, ch = blockIdx.y;
    const int o0 = (blockIdx.x * kThreads + tid) * kFirOut;      // first output of this thread
    if (tid < kTaps) sW[tid] = p.w[ch * kTaps + tid];
    __syncthreads();
    if (o0 >= p.S) return;
    const int32_t *src = p.in + (long long)ch * p.chan_stride;
    constexpr int WIN = kFirOut + kHist;                           // samples o0-20 .. o0+kFirOut-1
    double x[WIN];
    const int n0 = o0 - kHist;
    const bool fast = n0 >= 0 && o0 + kFirOut <= p.S && ((reinterpret_cast<size_t>(src + n0) & 15) == 0);
    if (fast) {
        static_assert(WIN % 4 == 0, "window in 128-bit pieces");
        const int4 *s4 = reinterpret_cast<const int4 *>(src + n0);
#pragma unroll
        for (int i = 0; i < WIN / 4; i++) {
            const int4 v = __ldg(s4 + i);
            x[4 * i + 0] = (double)v.x;
            x[4 * i + 1] = (double)v.y;
            x[4 * i + 2] = (double)v.z;
            x[4 * i + 3] = (double)v.w;
        }
    } else {
#pragma unroll
        for (int i = 0; i < WIN; i++) {
            const int n = n0 + i;
            int32_t v = 0;
            if (n < 0) v = p.hist_in[(size_t)ch * kHist + kHist + n];
            else if (n < p.S) v = src[n];
            x[i] = (double)v;
        }
    }
    double o[kFirOut];
#pragma unroll
    for (int r = 0; r < kFirOut; r++) o[r] = 0.0;
#pragma unroll
    for (int k = 0; k < kTaps; k++) {
        const double w = sW[k];
#pragma unroll
        for (int r = 0; r < kFirOut; r++) o[r] = __dadd_rn(o[r], __dmul_rn(x[r + kHist - k], w));   // :202-206
    }
    // :210 (int)o — truncation toward zero, saturating, NaN -> 0 (cvt.rzi.s32.f64 does exactly that)
    int32_t *dst = p.out + (size_t)ch * p.S + o0;
    if (o0 + kFirOut <= p.S && ((reinterpret_cast<size_t>(dst) & 15) == 0)) {
        int4 *d4 = reinterpret_cast<int4 *>(dst);
        d4[0] = make_int4(__double2int_rz(o[0]), __double2int_rz(o[1]), __double2int_rz(o[2]), __double2int_rz(o[3]));
        d4[1] = make_int4(__double2int_rz(o[4]), __double2int_rz(o[5]), __double2int_rz(o[6]), __double2int_rz(o[7]));
    } else {
#pragma unroll
        for (int r = 0; r < kFirOut; r++)
            if (o0 + r < p.S) dst[r] = __double2int_rz(o[r]);
    }
}

__global__ void k_fir_tail(const FirParams p)
{
    const int ch = blockIdx.x, k = threadIdx.x;
    if (k >= kHist) return;
    const int32_t *src = p.in + (long long)ch * p.chan_stride;
    int n = p.S - kHist + k;
    p.hist_out[(size_t)ch * kHist + k] = (n < 0) ? p.hist_in[(size_t)ch * kHist + k + p.S] : src[n];
}

// complex_mod :214-218, int32 wrapping
__global__ void k_complex_mod(const int2 *__restrict__ a, const int2 *__restrict__ b,
                              int2 *__restrict__ out, long long n)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        int2 x = a[i], y = b[i];
        unsigned re = (unsigned)x.x * (unsigned)y.x - (unsigned)x.y * (unsigned)y.y;
        unsigned im = (unsigned)x.x * (unsigned)y.y + (unsigned)x.y * (unsigned)y.x;
        out[i] = make_int2((int)re, (int)im);
    }
}

// Java (int)double
static int java_d2i(double d)
{
    if (d != d) return 0;
    if (d >= 2147483647.0) return INT_MAX;
    if (d <= -2147483648.0) return INT_MIN;
    return (int)d;
}

}  // namespace dsp
}  // namespace jsdr

using namespace jsdr;
using namespace jsdr::dsp;

// =========================================================================== demod
extern "C" int jsdr_demod_create(jsdr_ctx *ctx, int rate, int nchan, int max_block_samples, jsdr_demod **out)
try {
    JSDR_REQUIRE(ctx && out, JSDR_EINVAL, "null argument");
    JSDR_REQUIRE(rate > 0 && nchan > 0 && max_block_samples > 0, JSDR_EINVAL, "sizes must be positive");
    JSDR_REQUIRE(nchan <= 65535, JSDR_EINVAL, "at most 65535 channels per handle (the channel is the grid's y index)");
    JSDR_TRY(ctx->bind());
    std::unique_ptr<jsdr_demod> d(new jsdr_demod(ctx));
    d->rate = rate;
    d->nchan = nchan;
    d->max_block = max_block_samples;
    d->max_chunks = (int)((max_block_samples + kChunk - 1LL) / kChunk + 1);
    d->h_w.assign((size_t)nchan * kTaps, 0.0f);       // taps are zero until weights() runs (SURVEY Q5)
    d->h_phi.assign(nchan, 0.0f);
    const size_t nc = (size_t)nchan;
    const char *what = "jsdr_demod_create";
    cudaStream_t st = ctx->stream;
    JSDR_TRY(d->d_w.alloc_zeroed(sizeof(float) * kTaps * nc, st, what));
    JSDR_TRY(d->d_phi.alloc_zeroed(sizeof(float) * nc, st, what));
    JSDR_TRY(d->d_car.alloc_zeroed(sizeof(float) * nc, st, what));
    JSDR_TRY(d->d_chunk_car.alloc(sizeof(float) * nc * d->max_chunks, what));
    for (int i = 0; i < 2; i++) JSDR_TRY(d->d_hist[i].alloc_zeroed(sizeof(float2) * kHist * nc, st, what));
    JSDR_TRY(d->d_lilq.alloc_zeroed(sizeof(float2) * 2 * nc, st, what));
    JSDR_TRY(d->ev_car_ready.create(what));
    JSDR_TRY(d->ev_audio_ready.create(what));
    JSDR_CUDA(cudaStreamSynchronize(st));
    *out = d.release();
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_demod_destroy(jsdr_demod *d)
try {
    delete d;
    return JSDR_OK;
} JSDR_CATCH_ALL

// demod.weights(), demod.java:341-375
extern "C" int jsdr_demod_weights(jsdr_demod *d, int chan, int flo, int fhi)
try {
    JSDR_REQUIRE(d && chan >= 0 && chan < d->nchan, JSDR_EINVAL, "bad channel");
    jsdr_ctx *ctx = d->ctx;
    JSDR_TRY(ctx->bind());
    float *w = &d->h_w[(size_t)chan * kTaps];
    if (flo == INT_MIN) {                               // :343 all-pass; phi and car keep their values
        for (int i = 0; i < kTaps; i++) w[i] = 0.0f;
        w[(kTaps - 1) / 2] = 1.0f;
    } else {
        float rate = (float)d->rate;
        float nlo = (float)flo / rate;
        float nhi = (float)fhi / rate;
        int ord = kTaps - 1;
        for (int n = 0; n < kTaps; n++) {
            if (n == ord / 2) {
                w[n] = 2.0f * (nhi - nlo);
            } else {
                double dn = (double)(n - ord / 2);
                w[n] = (float)((sin(2 * M_PI * nhi * dn) / (M_PI * dn)) - (sin(2 * M_PI * nlo * dn) / (M_PI * dn)));
            }
            w[n] *= (float)(0.54 - 0.46 * cos(2 * M_PI * (double)n / (double)ord));
        }
        d->h_phi[chan] = (float)(2 * M_PI * nlo);       // :368
        const float zero = 0.0f;
        JSDR_TRY(upload(ctx, d->d_phi.get() + chan, &d->h_phi[chan], sizeof(float)));
        JSDR_TRY(upload(ctx, d->d_car.get() + chan, &zero, sizeof(float)));   // :369
    }
    JSDR_TRY(upload(ctx, d->d_w.get() + (size_t)chan * kTaps, w, sizeof(float) * kTaps));
    // :372-374 clear the delay line
    for (int i = 0; i < 2; i++)
        JSDR_CUDA(cudaMemsetAsync(d->d_hist[i].get() + (size_t)chan * kHist, 0, sizeof(float2) * kHist, ctx->stream));
    JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_demod_get_weights(jsdr_demod *d, int chan, float w[21])
try {
    JSDR_REQUIRE(d && w && chan >= 0 && chan < d->nchan, JSDR_EINVAL, "bad channel");
    memcpy(w, &d->h_w[(size_t)chan * kTaps], sizeof(float) * kTaps);
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_demod_set_flags(jsdr_demod *d, int dofir, int dodwn)
try {
    JSDR_REQUIRE(d, JSDR_EINVAL, "null argument");
    d->dofir = dofir != 0;
    d->dodwn = dodwn != 0;
    return JSDR_OK;
} JSDR_CATCH_ALL

namespace {

// The car replay of S samples (k_car_scout) on `side`, forked from the main stream (so it follows
// the previous k_demod of this handle, which read the checkpoints it overwrites) and joined back
// through `join`, which the main stream waits on before k_demod.
int demod_car_fork(jsdr_demod *d, int S, cudaEvent_t fork, cudaStream_t side, cudaEvent_t join)
{
    jsdr_ctx *ctx = d->ctx;
    JSDR_CUDA(cudaEventRecord(fork, ctx->stream));
    JSDR_CUDA(cudaStreamWaitEvent(side, fork, 0));
    k_car_scout<<<(d->nchan + 127) / 128, 128, 0, side>>>(d->d_phi.get(), d->d_car.get(), d->d_chunk_car.get(), d->nchan, S);
    JSDR_TRY(launched(ctx, "k_car_scout"));
    JSDR_CUDA(cudaEventRecord(join, side));
    return JSDR_OK;
}

// k_demod (or k_demod_s16) and the delay-line update over S samples per channel of device input
// d_in into d_out, on the main stream behind `car_ready` (the car replay of these S samples).
int demod_launch(jsdr_demod *d, const void *d_in, bool s16, int S, int64_t chan_stride, int ic, int qc,
                 float2 *d_out, cudaEvent_t car_ready)
{
    jsdr_ctx *ctx = d->ctx;
    const int nchan = d->nchan;
    if (d->dodwn) JSDR_CUDA(cudaStreamWaitEvent(ctx->stream, car_ready, 0));
    DemodParams p;
    p.in = d_in;
    p.chan_stride = chan_stride;
    p.S = S;
    p.nchan = nchan;
    p.w = d->d_w.get();
    p.phi = d->d_phi.get();
    p.chunk_car = d->d_chunk_car.get();
    p.hist_in = d->d_hist[d->hist_cur].get();
    p.hist_out = d->d_hist[d->hist_cur ^ 1].get();
    p.out = d_out;
    p.dofir = d->dofir;
    p.dodwn = d->dodwn;
    p.ic = ic;
    p.qc = qc;
    dim3 grid((S + kTile - 1) / kTile, nchan);
    {
        ProfScope prof(ctx, JSDR_K_DEMOD, ctx->stream);
        if (s16) k_demod_s16<<<grid, kThreads, 0, ctx->stream>>>(p);
        else k_demod<<<grid, kThreads, 0, ctx->stream>>>(p);
    }
    JSDR_TRY(launched(ctx, s16 ? "k_demod_s16" : "k_demod"));
    if (d->dofir) {   // the delay line only moves when filter() runs (:415-419)
        if (s16) k_demod_tail<true><<<nchan, 32, 0, ctx->stream>>>(p);
        else k_demod_tail<false><<<nchan, 32, 0, ctx->stream>>>(p);
        JSDR_TRY(launched(ctx, "k_demod_tail"));
        d->hist_cur ^= 1;
    }
    return JSDR_OK;
}

// FIR + NCO of one block for every channel; the result stays on the device in *d_result
// ([nchan][S] float2: `out` itself for device calls, the staging buffer for host calls).
// `in` is float IQ, or s16 IQ with its I/Q corrections when s16 is set.
int demod_run(jsdr_demod *d, const void *in, bool s16, int S, int64_t chan_stride, int ic, int qc, float *out,
              int mem, float2 **d_result)
{
    jsdr_ctx *ctx = d->ctx;
    const int nchan = d->nchan;
    if (d->dodwn) JSDR_TRY(demod_car_fork(d, S, ctx->ev_fork, ctx->side, ctx->ev_join));
    const void *d_in = in;
    float2 *d_out = reinterpret_cast<float2 *>(out);
    const size_t out_bytes = sizeof(float2) * (size_t)nchan * S;
    if (mem == JSDR_MEM_HOST) {
        const size_t esz = s16 ? 4 : 8;
        const size_t total = (chan_stride == 0) ? (size_t)S : (size_t)chan_stride * (nchan - 1) + S;
        JSDR_TRY(d->d_in.grow(total * esz, "demod staging"));
        JSDR_CUDA(cudaMemcpyAsync(d->d_in.get(), in, total * esz, cudaMemcpyHostToDevice, ctx->stream));
        d_in = d->d_in.get();
    }
    if (mem == JSDR_MEM_HOST || !out) {
        JSDR_TRY(d->d_out.grow(out_bytes, "demod staging"));
        d_out = d->d_out.get();
    }
    JSDR_TRY(demod_launch(d, d_in, s16, S, chan_stride, ic, qc, d_out, ctx->ev_join));
    *d_result = d_out;
    return JSDR_OK;
}

int demod_check(jsdr_demod *d, const void *iq, const void *out, int S, int64_t chan_stride, int mem)
{
    JSDR_REQUIRE(d && iq && out, JSDR_EINVAL, "null argument");
    JSDR_REQUIRE(S >= 0 && S <= d->max_block, JSDR_EINVAL, "nsamples exceeds max_block_samples");
    JSDR_REQUIRE(chan_stride == 0 || chan_stride >= S, JSDR_EINVAL, "chan_stride smaller than nsamples");
    JSDR_REQUIRE(mem == JSDR_MEM_HOST || mem == JSDR_MEM_DEVICE, JSDR_EINVAL, "bad mem");
    return JSDR_OK;
}

int demod_receive(jsdr_demod *d, const void *in, bool s16, int S, int64_t chan_stride, int ic, int qc,
                  float *out, int mem)
{
    JSDR_TRY(demod_check(d, in, out, S, chan_stride, mem));
    if (S == 0) return JSDR_OK;
    jsdr_ctx *ctx = d->ctx;
    JSDR_TRY(ctx->bind());
    float2 *res = nullptr;
    JSDR_TRY(demod_run(d, in, s16, S, chan_stride, ic, qc, out, mem, &res));
    if (mem == JSDR_MEM_HOST) {
        JSDR_CUDA(cudaMemcpyAsync(out, res, sizeof(float2) * (size_t)d->nchan * S, cudaMemcpyDeviceToHost, ctx->stream));
        JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return JSDR_OK;
}

}  // namespace

extern "C" int jsdr_demod_receive_f32(jsdr_demod *d, const float *iq, int S, int64_t chan_stride,
                                      float *out, int mem)
try {
    return demod_receive(d, iq, false, S, chan_stride, 0, 0, out, mem);
} JSDR_CATCH_ALL

extern "C" int jsdr_demod_receive_s16(jsdr_demod *d, const int16_t *raw, int S, int64_t chan_stride,
                                      int ic, int qc, float *out, int mem)
try {
    return demod_receive(d, raw, true, S, chan_stride, ic, qc, out, mem);
} JSDR_CATCH_ALL

// ------------------------------------------------------------------ detectors, AGC, s16 (:405-481)
namespace jsdr {
namespace dsp {

enum { MODE_OFF = 0, MODE_RAW = 1, MODE_AM = 2, MODE_NFM = 3, MODE_WFM = 4 };   // demod.java:39-43

__device__ __forceinline__ int java_f2i(float x)
{   // Java (int)float: NaN -> 0, saturating
    if (x != x) return 0;
    if (x >= 2147483648.0f) return 2147483647;
    if (x <= -2147483648.0f) return (int)0x80000000;
    return (int)x;
}

// demod.java:451 for the `cnt` samples of a tile (operands in .z) from sample index k0 with the
// IEEE division itself: the blocks k_detect's running mean does not take through its reciprocal
// pairs (out of line, so that the common path stays small)
__device__ __noinline__ float running_mean_div(float avg, const float4 *op, int k0, int cnt)
{
    for (int i = 0; i < cnt; i++)
        avg = __fdiv_rn(__fadd_rn(__fmul_rn((float)(k0 + i), avg), op[i].z), (float)(k0 + i + 1));
    return avg;
}

// One CTA per (channel, block): a row of Srow samples per channel is cut into blocks of L
// samples (the last may be shorter), each one demod.receive call -- so the maximum, the AM running
// mean (avg restarts at k = 0) and the AGC gain are per block, while li/lq run across blocks.
// Pass 1: the detector output of every sample (sample parallel; the FM discriminator's previous
// sample is the neighbour: for the first sample of block j > 0 the last of block j - 1, for the
// first of the row the carried lilq_in) and the block maximum of |.| (:448-463).  Pass 2 (AM): the
// running mean avg = ((k)*avg + x)/(k+1) is a sequential float recurrence (:451), replayed by one
// thread over tiles staged in shared memory.  Pass 3: AM subtracts the mean, AGC scales by
// 1.0f/max, narrow to s16 as Java's (short) does (:469-473).  The last block of a row leaves its
// last sample in lilq_out (FM modes); lilq_out may be lilq_in when a row is one block (the CTA
// reads before it writes).  `det` is scratch [nchan][Srow]; max_avg is [nchan][nblocks][2].
__global__ void __launch_bounds__(256, 8) k_detect(const float2 *__restrict__ mixed, int Srow, int L, int mode, float fmgain,
                                                int doagc, const float2 *lilq_in, float2 *lilq_out, float *__restrict__ det,
                                                int16_t *__restrict__ audio, float *__restrict__ max_avg)
{
    __shared__ unsigned s_max;
    __shared__ int s_nan;
    __shared__ float s_avg;
    __shared__ int s_slow;
    __shared__ __align__(16) float4 s_op[2][512];    // per sample of a tile: (y_hi, y_lo, x, x*y_lo), 1/n = y_hi + y_lo; two tiles
    const int nblk = (Srow + L - 1) / L;
    const int ch = blockIdx.x / nblk, blk = blockIdx.x - ch * nblk, tid = threadIdx.x;
    const size_t base = (size_t)ch * Srow + (size_t)blk * L;
    const int S = min(L, Srow - blk * L);                        // this block's samples
    const float2 *x = mixed + base;
    float *dv = det + base;
    if (tid == 0) {
        s_max = 0u;
        s_nan = 0;
        s_slow = 0;
        s_avg = 0.0f;
    }
    __syncthreads();
    const float2 prev0 = (blk == 0) ? lilq_in[ch] : x[-1];
    unsigned mymax = 0u;
    int mynan = 0;
    for (int k = tid; k < S; k += blockDim.x) {
        const float2 v = x[k];
        float o;
        if (mode == MODE_OFF) o = 0.0f;
        else if (mode == MODE_RAW) o = v.x;
        else if (mode == MODE_AM) {
            // (float)Math.sqrt(sam[s]*sam[s]+sam[s+1]*sam[s+1]): float sum of squares, double sqrt
            const float ss = __fadd_rn(__fmul_rn(v.x, v.x), __fmul_rn(v.y, v.y));
            o = (float)__dsqrt_rn((double)ss);
        } else {
            const float2 l = (k == 0) ? prev0 : x[k - 1];          // li, lq (:456-458)
            o = __fmul_rn(__fsub_rn(__fmul_rn(l.x, v.y), __fmul_rn(l.y, v.x)), fmgain);
        }
        dv[k] = o;
        const float a = fabsf(o);
        if (a != a) mynan = 1;
        else mymax = max(mymax, __float_as_uint(a));               // non-negative floats order like their bits
    }
    atomicMax(&s_max, mymax);
    if (mynan) s_nan = 1;
    __syncthreads();
    if ((mode == MODE_NFM || mode == MODE_WFM) && tid == 0 && S > 0 && blk == nblk - 1) lilq_out[ch] = x[S - 1];
    if (mode == MODE_AM) {
        // avg = ((float)k*avg + x) / (float)(k+1) (:451) is a sequential float recurrence with a
        // division on the chain, walked by one thread.  What does not depend on the chain is filled
        // in per tile by the other threads: 1/n as a float pair y_hi + y_lo (relative error < 2^-47) and
        // x*y_lo.  With t = RN(k*avg) and a = RN(t + x) (the reference's two roundings) the quotient
        // is q = fma(a, y_hi, p), p = fma(t, y_lo, RN(x*y_lo)): p is a*y_lo to within 3*2^-24 (t and
        // x are both >= 0 here: amplitudes and their mean), so the value in front of q's rounding is
        // a/n to within 2^-46 (relative), while a quotient of a 24-bit significand by an integer
        // n < 2^19 is a float or at least 2^-44 away from every rounding boundary of the float
        // format (it cannot sit on one: n times a 25-bit midpoint does not fit 24 bits) -- so q is
        // the IEEE quotient, with FMUL, FADD, FFMA on the chain (13.5 cycles) instead of the division
        // subroutine (about 110) or a binary64 detour (FMUL, FADD, F2F, DMUL, F2F: about 55).
        // Range: with every x so far in {0} or [2^-38, 2^64] (the largest finite amplitude is below
        // 2^64) every sum a is 0 or in [2^-39, 2^85] (three roundings per step over < 2^19 steps
        // lose less than 12 %), so no product above leaves the normal range by more than a rounding
        // of y_lo's term, 2^-150 against a/n >= 2^-58.  A block takes the division itself from the
        // first tile that holds anything else (tiny, infinite, NaN) or reaches n = 2^19.
        // tests/test_detect_quotient.py checks the arithmetic in exact rationals.
        // Tiles of 512 samples, two buffers: while thread 0 walks tile t, warps 1..7 fill tile t + 1
        // (its global loads and binary64 reciprocals stay off the walker's time).  s_slow set by the
        // fill of tile t + 1 may already be seen by the walk of tile t: both paths give the same bits.
        constexpr int kT = 512;
        auto fill = [&](int t0, float4 *buf, int first, int stride) {
            const int cnt = min(kT, S - t0);
            bool odd = false;
            for (int i = first; i < cnt; i += stride) {
                const float xv = dv[t0 + i];
                const double r = __drcp_rn((double)(t0 + i + 1));
                const float yh = __double2float_rn(r);
                const float yl = __double2float_rn(__dsub_rn(r, (double)yh));
                buf[i] = make_float4(yh, yl, xv, __fmul_rn(xv, yl));
                odd |= !(xv == 0.0f || (xv >= 3.637978807091713e-12f && xv <= 1.8446744073709552e19f));
            }
            if (odd || t0 + cnt >= (1 << 19)) s_slow = 1;
        };
        if (S > 0) fill(0, s_op[0], tid, blockDim.x);
        __syncthreads();
        for (int t0 = 0, t = 0; t0 < S; t0 += kT, t++) {
            const int cnt = min(kT, S - t0);
            const float4 *cur = s_op[t & 1];
            if (tid >= 32) {
                if (t0 + kT < S) fill(t0 + kT, s_op[(t + 1) & 1], tid - 32, blockDim.x - 32);
            } else if (tid == 0) {
                float avg = s_avg;
                if (!s_slow) {
                    float kf = (float)t0;
                    auto step = [&](const float4 op) {
                        const float tk = __fmul_rn(kf, avg);
                        const float a = __fadd_rn(tk, op.z);
                        avg = __fmaf_rn(a, op.x, __fmaf_rn(tk, op.y, op.w));
                        kf = __fadd_rn(kf, 1.0f);
                    };
                    // two samples per round, the next round's operands fetched ahead of the chain
                    float4 n0 = cur[0], n1 = cur[1];
                    int i = 0;
#pragma unroll 2
                    for (; i + 2 <= cnt; i += 2) {
                        const float4 c0 = n0, c1 = n1;
                        const int nx = min(i + 2, kT - 2);
                        n0 = cur[nx];
                        n1 = cur[nx + 1];
                        step(c0);
                        step(c1);
                    }
                    if (i < cnt) step(cur[i]);
                } else {
                    avg = running_mean_div(avg, cur, t0, cnt);
                }
                s_avg = avg;
            }
            __syncthreads();
        }
    }
    float mx = s_nan ? __uint_as_float(0x7fc00000u) : __uint_as_float(s_max);      // Math.max keeps NaN
    const float avg = s_avg;
    if (mode == MODE_AM) mx = __fsub_rn(mx, avg);                                  // :466-468
    const float gain = doagc ? __fdiv_rn(1.0f, mx) : 1.0f;
    for (int k = tid; k < S; k += blockDim.x) {
        float o = dv[k];
        if (mode == MODE_AM) o = __fsub_rn(o, avg);
        o = __fmul_rn(o, gain);
        audio[base + k] = (int16_t)(java_f2i(__fmul_rn(o, 32767.0f)) & 0xffff);   // (short)(float)
    }
    if (tid == 0 && max_avg) {
        max_avg[2 * (size_t)blockIdx.x] = mx;
        max_avg[2 * (size_t)blockIdx.x + 1] = avg;
    }
}

}  // namespace dsp
}  // namespace jsdr

extern "C" int jsdr_demod_set_mode(jsdr_demod *d, int mode, int doagc)
try {
    JSDR_REQUIRE(d && mode >= dsp::MODE_OFF && mode <= dsp::MODE_WFM, JSDR_EINVAL, "mode must be 0..4 (demod.java:39-43)");
    d->mode = mode;
    d->doagc = doagc != 0;
    return JSDR_OK;
} JSDR_CATCH_ALL

namespace {

// k_detect over rows of Srow samples per channel of the FIR + NCO output `res`, cut into blocks
// of L samples: audio [nchan][Srow], max_avg (nullable) [nchan][ceil(Srow/L)][2].
int detect_launch(jsdr_demod *d, const float2 *res, int Srow, int L, int16_t *audio, float *max_avg)
{
    jsdr_ctx *ctx = d->ctx;
    const int nchan = d->nchan, nblk = (Srow + L - 1) / L;
    JSDR_TRY(d->d_det.grow((size_t)nchan * Srow * sizeof(float), "demod detector"));
    // :409 fmgain = ad.rate / (MODE_NFM==mode ? 5000f : 75000f), int / float in float
    const float fmgain = (float)d->rate / (d->mode == dsp::MODE_NFM ? 5000.0f : 75000.0f);
    // One block per row: the CTA reads li/lq before it writes them.  Several: block 0 of a row may
    // still read the carried li/lq while the last block writes its own, so that one goes to the
    // second half of d_lilq and is copied back behind the kernel.
    float2 *lilq = d->d_lilq.get(), *lilq_out = nblk > 1 ? lilq + nchan : lilq;
    {
        ProfScope prof(ctx, JSDR_K_DETECT, ctx->stream);
        dsp::k_detect<<<(unsigned)nchan * nblk, 256, 0, ctx->stream>>>(res, Srow, L, d->mode, fmgain, d->doagc, lilq,
                                                                        lilq_out, d->d_det.get(), audio, max_avg);
    }
    JSDR_TRY(launched(ctx, "k_detect"));
    if (nblk > 1 && (d->mode == dsp::MODE_NFM || d->mode == dsp::MODE_WFM))
        JSDR_CUDA(cudaMemcpyAsync(lilq, lilq_out, sizeof(float2) * nchan, cudaMemcpyDeviceToDevice, ctx->stream));
    return JSDR_OK;
}

// staging of a host call's audio and max/avg pairs (npairs of them) in d->d_audio
int audio_staging(jsdr_demod *d, size_t nsamp, size_t npairs, int16_t **d_audio, float **d_ma)
{
    const size_t ma_off = (nsamp * sizeof(int16_t) + 15) & ~(size_t)15;
    JSDR_TRY(d->d_audio.grow(ma_off + sizeof(float) * 2 * npairs, "demod staging"));
    *d_audio = d->d_audio.get();
    *d_ma = reinterpret_cast<float *>(reinterpret_cast<char *>(d->d_audio.get()) + ma_off);
    return JSDR_OK;
}

int demod_receive_audio(jsdr_demod *d, const void *in, bool s16, int S, int64_t chan_stride, int ic, int qc,
                        int16_t *audio, float *max_avg, int mem)
{
    JSDR_TRY(demod_check(d, in, audio, S, chan_stride, mem));
    if (S == 0) return JSDR_OK;
    jsdr_ctx *ctx = d->ctx;
    JSDR_TRY(ctx->bind());
    const size_t n = (size_t)d->nchan * S;
    float2 *res = nullptr;
    JSDR_TRY(demod_run(d, in, s16, S, chan_stride, ic, qc, nullptr, mem, &res));
    int16_t *d_audio = audio;
    float *d_ma = max_avg;
    if (mem == JSDR_MEM_HOST) JSDR_TRY(audio_staging(d, n, d->nchan, &d_audio, &d_ma));
    JSDR_TRY(detect_launch(d, res, S, S, d_audio, d_ma));
    if (mem == JSDR_MEM_HOST) {
        JSDR_CUDA(cudaMemcpyAsync(audio, d_audio, n * sizeof(int16_t), cudaMemcpyDeviceToHost, ctx->stream));
        if (max_avg)
            JSDR_CUDA(cudaMemcpyAsync(max_avg, d_ma, sizeof(float) * 2 * d->nchan, cudaMemcpyDeviceToHost, ctx->stream));
        JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return JSDR_OK;
}

}  // namespace

extern "C" int jsdr_demod_receive_audio_f32(jsdr_demod *d, const float *iq, int S, int64_t chan_stride,
                                            int16_t *audio, float *max_avg, int mem)
try {
    return demod_receive_audio(d, iq, false, S, chan_stride, 0, 0, audio, max_avg, mem);
} JSDR_CATCH_ALL

extern "C" int jsdr_demod_receive_audio_s16(jsdr_demod *d, const int16_t *raw, int S, int64_t chan_stride,
                                            int ic, int qc, int16_t *audio, float *max_avg, int mem)
try {
    return demod_receive_audio(d, raw, true, S, chan_stride, ic, qc, audio, max_avg, mem);
} JSDR_CATCH_ALL

// ------------------------------------------------------------------ the pump's demod handler
// jsdr_pump_demod_s16 (pump.cu) runs demod over the pump's resident rows of S samples per channel
// (chan_stride S) as nblocks successive demod.receive calls of L samples: one FIR + NCO launch over
// the whole row (the delay line and car carry from call to call anyway), then k_detect per block.

// The car replay of the S samples, on side2 behind whatever the main stream holds now: side2
// carries only the bank's short VCO / bit-phase replay, while the side stream may still be busy
// with the bank's tuner-phase replay for this very call (enqueued at the end of the previous one).
// d->ev_car_ready marks its end; jsdr_pump_demod_run waits on it.
int jsdr_pump_demod_fork(jsdr_demod *d, int S)
{
    if (!d->dodwn) return JSDR_OK;
    return demod_car_fork(d, S, d->ctx->ev_fork, d->ctx->side2, d->ev_car_ready);
}

// Staging of the host pump's audio [nchan][S] and max/avg pairs [nchan][nblocks][2].
int jsdr_pump_demod_staging(jsdr_demod *d, int S, int nblocks, int16_t **d_audio, float **d_max_avg)
{
    return audio_staging(d, (size_t)d->nchan * S, (size_t)d->nchan * nblocks, d_audio, d_max_avg);
}

// FIR + NCO of the s16 rows d_raw [nchan][S] and the detectors per block of L samples, on the main
// stream: audio [nchan][S] and max_avg (nullable) [nchan][S/L][2] are device pointers.
int jsdr_pump_demod_run(jsdr_demod *d, const int16_t *d_raw, int S, int L, int ic, int qc, int16_t *audio,
                        float *max_avg)
{
    JSDR_TRY(d->d_out.grow(sizeof(float2) * (size_t)d->nchan * S, "demod staging"));
    float2 *mixed = d->d_out.get();
    JSDR_TRY(demod_launch(d, d_raw, true, S, S, ic, qc, mixed, d->ev_car_ready));
    return detect_launch(d, mixed, S, L, audio, max_avg);
}

// =========================================================================== fir.java
// fir.weights(), fir.java:169-195 (host, one-off)
extern "C" int jsdr_fir_design(int f1, int f2, float rate, double w[21])
try {
    JSDR_REQUIRE(w && rate > 0, JSDR_EINVAL, "bad argument");
    if (f1 == INT_MIN && f2 == INT_MIN) {
        for (int i = 0; i < kTaps; i++) w[i] = 0;
        w[(kTaps - 1) / 2] = 1;
        return JSDR_OK;
    }
    double df1 = (double)f1 / rate;
    double df2 = (double)f2 / rate;
    int ord = kTaps - 1;
    for (int n = 0; n < kTaps; n++) {
        if (n == ord / 2) {
            w[n] = 2 * (df2 - df1);
        } else {
            int dn = n - ord / 2;
            w[n] = (sin(2 * M_PI * df2 * dn) / (M_PI * dn)) - (sin(2 * M_PI * df1 * dn) / (M_PI * dn));
        }
        w[n] = w[n] * (0.54 - 0.46 * cos(2 * M_PI * n / ord));
    }
    return JSDR_OK;
} JSDR_CATCH_ALL

// one period of complex_gen, fir.java:221-228 (the counter wraps at (int)rate)
extern "C" int jsdr_fir_nco_table(int freq, float rate, int32_t *sig)
try {
    JSDR_REQUIRE(sig && rate >= 1.0f, JSDR_EINVAL, "bad argument");
    const int period = (int)rate;
    for (int n = 0; n < period; n++) {
        double w = (((2 * M_PI) * freq) * n) / rate;
        sig[2 * n] = java_d2i(cos(w) * 4096);
        sig[2 * n + 1] = java_d2i(sin(w) * 4096);
    }
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_fir_create(jsdr_ctx *ctx, int nchan, int max_block_samples, jsdr_fir **out)
try {
    JSDR_REQUIRE(ctx && out, JSDR_EINVAL, "null argument");
    JSDR_REQUIRE(nchan > 0 && max_block_samples > 0, JSDR_EINVAL, "sizes must be positive");
    JSDR_REQUIRE(nchan <= 65535, JSDR_EINVAL, "at most 65535 channels per handle (the channel is the grid's y index)");
    JSDR_TRY(ctx->bind());
    std::unique_ptr<jsdr_fir> f(new jsdr_fir(ctx));
    f->nchan = nchan;
    f->max_block = max_block_samples;
    const size_t nc = (size_t)nchan;
    JSDR_TRY(f->d_w.alloc_zeroed(sizeof(double) * kTaps * nc, ctx->stream, "jsdr_fir_create"));
    for (int i = 0; i < 2; i++) JSDR_TRY(f->d_hist[i].alloc_zeroed(sizeof(int32_t) * kHist * nc, ctx->stream, "jsdr_fir_create"));
    JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
    *out = f.release();
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_fir_destroy(jsdr_fir *f)
try {
    delete f;
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_fir_set_weights(jsdr_fir *f, int chan, const double w[21])
try {
    JSDR_REQUIRE(f && w && chan >= 0 && chan < f->nchan, JSDR_EINVAL, "bad channel");
    jsdr_ctx *ctx = f->ctx;
    JSDR_TRY(ctx->bind());
    JSDR_TRY(upload(ctx, f->d_w.get() + (size_t)chan * kTaps, w, sizeof(double) * kTaps));
    for (int i = 0; i < 2; i++)                          // :192-193 clear previous samples
        JSDR_CUDA(cudaMemsetAsync(f->d_hist[i].get() + (size_t)chan * kHist, 0, sizeof(int32_t) * kHist, ctx->stream));
    JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_fir_filter_i32(jsdr_fir *f, const int32_t *in, int S, int64_t chan_stride,
                                   int32_t *out, int mem)
try {
    JSDR_REQUIRE(f && in && out, JSDR_EINVAL, "null argument");
    JSDR_REQUIRE(S >= 0 && S <= f->max_block, JSDR_EINVAL, "nsamples exceeds max_block_samples");
    JSDR_REQUIRE(chan_stride == 0 || chan_stride >= S, JSDR_EINVAL, "chan_stride smaller than nsamples");
    JSDR_REQUIRE(mem == JSDR_MEM_HOST || mem == JSDR_MEM_DEVICE, JSDR_EINVAL, "bad mem");
    if (S == 0) return JSDR_OK;
    jsdr_ctx *ctx = f->ctx;
    JSDR_TRY(ctx->bind());
    const int nchan = f->nchan;
    const int32_t *d_in = in;
    int32_t *d_out = out;
    const size_t out_bytes = sizeof(int32_t) * (size_t)nchan * S;
    if (mem == JSDR_MEM_HOST) {
        const size_t total = (chan_stride == 0) ? (size_t)S : (size_t)chan_stride * (nchan - 1) + S;
        JSDR_TRY(f->d_in.grow(total * sizeof(int32_t), "fir staging"));
        JSDR_TRY(f->d_out.grow(out_bytes, "fir staging"));
        JSDR_CUDA(cudaMemcpyAsync(f->d_in.get(), in, total * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
        d_in = f->d_in.get();
        d_out = f->d_out.get();
    }
    FirParams p;
    p.in = d_in;
    p.chan_stride = chan_stride;
    p.S = S;
    p.w = f->d_w.get();
    p.hist_in = f->d_hist[f->hist_cur].get();
    p.hist_out = f->d_hist[f->hist_cur ^ 1].get();
    p.out = d_out;
    dim3 grid((S + kThreads * kFirOut - 1) / (kThreads * kFirOut), nchan);
    {
        ProfScope prof(ctx, JSDR_K_FIR, ctx->stream);
        k_fir_i32<<<grid, kThreads, 0, ctx->stream>>>(p);
    }
    JSDR_TRY(launched(ctx, "k_fir_i32"));
    k_fir_tail<<<nchan, 32, 0, ctx->stream>>>(p);
    JSDR_TRY(launched(ctx, "k_fir_tail"));
    f->hist_cur ^= 1;
    if (mem == JSDR_MEM_HOST) {
        JSDR_CUDA(cudaMemcpyAsync(out, f->d_out.get(), out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_fir_complex_mod_i32(jsdr_ctx *ctx, const int32_t *a, const int32_t *b, int32_t *out,
                                        int64_t npairs, int mem)
try {
    JSDR_REQUIRE(ctx && a && b && out && npairs >= 0, JSDR_EINVAL, "bad argument");
    JSDR_REQUIRE(mem == JSDR_MEM_HOST || mem == JSDR_MEM_DEVICE, JSDR_EINVAL, "bad mem");
    if (npairs == 0) return JSDR_OK;
    JSDR_TRY(ctx->bind());
    const size_t bytes = sizeof(int2) * (size_t)npairs;
    const int2 *da = reinterpret_cast<const int2 *>(a), *db = reinterpret_cast<const int2 *>(b);
    int2 *dout = reinterpret_cast<int2 *>(out);
    DevBuf<int2> tmp;
    if (mem == JSDR_MEM_HOST) {
        JSDR_TRY(tmp.alloc(3 * bytes, "jsdr_fir_complex_mod_i32"));
        int2 *t = tmp.get();
        JSDR_CUDA(cudaMemcpyAsync(t, a, bytes, cudaMemcpyHostToDevice, ctx->stream));
        JSDR_CUDA(cudaMemcpyAsync(t + npairs, b, bytes, cudaMemcpyHostToDevice, ctx->stream));
        da = t;
        db = t + npairs;
        dout = t + 2 * npairs;
    }
    long long blocks = (npairs + 255) / 256;
    int grid = (int)(blocks < 148 * 16 ? blocks : 148 * 16);
    k_complex_mod<<<grid, 256, 0, ctx->stream>>>(da, db, dout, npairs);
    JSDR_TRY(launched(ctx, "k_complex_mod"));
    if (mem == JSDR_MEM_HOST) {
        JSDR_CUDA(cudaMemcpyAsync(out, dout, bytes, cudaMemcpyDeviceToHost, ctx->stream));
        JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return JSDR_OK;
} JSDR_CATCH_ALL

// =========================================================================== waterfall.java
// paintLine (waterfall.java:90-107): max-decimate one published "fft-psd" row to the pixel
// width, map -100 dBFS..0 to 0..255, tint with the peak colour, rotate by half the width
// (the row is in FFT order) and pack as ColorModel.getRGBdefault() ARGB.
namespace jsdr {
namespace dsp {
__global__ void __launch_bounds__(256) k_waterfall(const float *__restrict__ psd, int n, int width, unsigned peak_rgb,
                                                   int32_t *__restrict__ pix)
{
    const int row = blockIdx.x;                                    // rows in x: a batch has more than 65535 of them
    const int p = blockIdx.y * blockDim.x + threadIdx.x;
    if (p >= width) return;
    const float *a = psd + (size_t)row * (n + 2);
    const float step = __fdiv_rn((float)n, (float)width);          // :61 (float)(length-2)/(float)getWidth()
    const int o = java_f2i(__fmul_rn((float)p, step)), l = java_f2i(step);
    float r = a[min(max(o, 0), n + 1)];                            // getMax (:109-116)
    for (int i = o + 1; i < o + l && i < n + 2; i++)
        if (a[i] > r) r = a[i];
    int f = 255 - java_f2i(__fmul_rn(r, -2.55f));                  // :95
    f = f < 0 ? 0 : f;
    f = f > 255 ? 255 : f;
    const int pr = (peak_rgb >> 16) & 255, pg = (peak_rgb >> 8) & 255, pb = peak_rgb & 255;
    const unsigned c = 0xff000000u | ((unsigned)(pr * f / 256) << 16) | ((unsigned)(pg * f / 256) << 8) | (unsigned)(pb * f / 256);
    pix[(size_t)row * width + (p + width / 2) % width] = (int32_t)c;   // :104 off = getWidth()/2
}
}  // namespace dsp
}  // namespace jsdr

// paintLine for `rows` device-resident PSD rows on a given stream (jsdr_waterfall_rows and the
// pump's pixel path, bpsk.cu)
int jsdr_launch_waterfall(jsdr_ctx *ctx, const float *d_psd, int n, int rows, int width, uint32_t peak_rgb,
                          int32_t *d_pix, cudaStream_t st)
{
    if (rows <= 0) return JSDR_OK;
    dim3 grid(rows, (width + 255) / 256);
    ProfScope prof(ctx, JSDR_K_WATERFALL, st);
    jsdr::dsp::k_waterfall<<<grid, 256, 0, st>>>(d_psd, n, width, peak_rgb, d_pix);
    return launched(ctx, "k_waterfall");
}

extern "C" int jsdr_waterfall_rows(jsdr_ctx *ctx, const float *psd, int n, int rows, int width, uint32_t peak_rgb,
                                   int32_t *pixels, int mem)
try {
    JSDR_REQUIRE(ctx && psd && pixels, JSDR_EINVAL, "null argument");
    JSDR_REQUIRE(n > 0 && rows >= 0 && width > 0 && width <= n, JSDR_EINVAL, "need 0 < width <= n");
    JSDR_REQUIRE(mem == JSDR_MEM_HOST || mem == JSDR_MEM_DEVICE, JSDR_EINVAL, "bad mem");
    if (rows == 0) return JSDR_OK;
    JSDR_TRY(ctx->bind());
    const float *d_psd = psd;
    int32_t *d_pix = pixels;
    DevBuf<float> tmp_in;
    DevBuf<int32_t> tmp_out;
    const size_t in_bytes = sizeof(float) * (size_t)rows * (n + 2), out_bytes = sizeof(int32_t) * (size_t)rows * width;
    if (mem == JSDR_MEM_HOST) {
        JSDR_TRY(tmp_in.alloc(in_bytes, "jsdr_waterfall_rows"));
        JSDR_TRY(tmp_out.alloc(out_bytes, "jsdr_waterfall_rows"));
        JSDR_CUDA(cudaMemcpyAsync(tmp_in.get(), psd, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
        d_psd = tmp_in.get();
        d_pix = tmp_out.get();
    }
    JSDR_TRY(jsdr_launch_waterfall(ctx, d_psd, n, rows, width, peak_rgb, d_pix, ctx->stream));
    if (mem == JSDR_MEM_HOST) {
        JSDR_CUDA(cudaMemcpyAsync(pixels, d_pix, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return JSDR_OK;
} JSDR_CATCH_ALL
