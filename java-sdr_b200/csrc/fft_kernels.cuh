// fft_kernels.cuh — batched complex FFT + power spectrum for sm_100a.
//
// Replaces the arithmetic behind fft.receive (reference fft.java:190-228): an
// unnormalised forward complex DFT (JTransforms FloatFFT_1D.complexForward,
// fft.java:194-195) followed by psd = 10*log10((re^2+im^2)*(2/N)^2)
// (fft.java:199-207), the first strict maximum (:208-211) and its frequency in
// wrapping int32 arithmetic (:214-221).
//
// Structure: one CTA transforms G whole blocks in shared memory.
//   pass 0     reads x[c + m*N/R0] straight from HBM (each warp request is a
//              contiguous run), does an R0-point DFT in registers and scatters the
//              R0 results as one contiguous chunk to the digit-reversed row,
//              so every later pass is in place;
//   middle     in-place radix-Rp butterflies, twiddle before the butterfly (DIT);
//   last pass  radix-RL butterfly whose outputs are bins j + q*N/RL, i.e. natural
//              order with consecutive lanes on consecutive bins: the PSD epilogue
//              (|X|^2*cf -> dB, arg-max) is fused here and the spectrum is never
//              written back to shared memory.
// Rows (one per last-pass input) are padded so that the chunk scatter of pass 0
// does not bank-conflict.  The index plan is emulated in tools/fft_plan_emulate.py.
#pragma once

#include <type_traits>

#include "handles.h"

namespace jsdr {
namespace fft {

// ------------------------------------------------------------------ constants
__host__ __device__ constexpr double cx_pi() { return 3.14159265358979323846264338327950288; }

__host__ __device__ constexpr double cx_sin_small(double x)
{   // |x| <= pi/4, Taylor to ~1e-19
    double x2 = x * x, term = x, sum = x;
    for (int i = 1; i < 14; i++) {
        term *= -x2 / (double)((2 * i) * (2 * i + 1));
        sum += term;
    }
    return sum;
}
__host__ __device__ constexpr double cx_cos_small(double x)
{
    double x2 = x * x, term = 1.0, sum = 1.0;
    for (int i = 1; i < 14; i++) {
        term *= -x2 / (double)((2 * i - 1) * (2 * i));
        sum += term;
    }
    return sum;
}
// cos / sin of 2*pi*k/r with the octant reduced on the integers
__host__ __device__ constexpr double cx_cos2pi(int k, int r)
{
    k %= r;
    if (k < 0) k += r;
    // work in eighths of a turn: a / (8r) turns
    long a = 8L * k, q = r;            // angle = 2*pi*a/(8q)
    if (a > 4 * q) a = 8 * q - a;      // cos(2pi - t) = cos t
    bool neg = false;
    if (a > 2 * q) { a = 4 * q - a; neg = true; }     // cos(pi - t) = -cos t
    double v = 0;
    if (a > q) v = cx_sin_small(2.0 * cx_pi() * (double)(2 * q - a) / (double)(8 * q));  // cos t = sin(pi/2 - t)
    else v = cx_cos_small(2.0 * cx_pi() * (double)a / (double)(8 * q));
    return neg ? -v : v;
}
__host__ __device__ constexpr double cx_sin2pi(int k, int r)
{
    // sin t = cos(t - pi/2) = cos(2*pi*(k/r - 1/4)) = cos(2*pi*(4k - r)/(4r))
    return cx_cos2pi(4 * k - r, 4 * r);
}

template <int I, int N, class F>
__device__ __forceinline__ void static_for(F &&f)
{
    if constexpr (I < N) {
        f(std::integral_constant<int, I>{});
        static_for<I + 1, N>(f);
    }
}

// ---- packed complex arithmetic ---------------------------------------------
// sm_100a has two-wide FP32 instructions (PTX add/mul/fma .f32x2 -> SASS FADD2 /
// FMUL2 / FFMA2) whose operands take a half-swap, per-half negation or a scalar
// broadcast for free.  A complex value is one 64-bit register pair, so a complex
// add is ONE instruction, a multiply by -i or +i folds into the consumer, and a
// complex multiply is two.  The FFT is issue-bound, so this is the main lever.
__device__ __forceinline__ unsigned long long as_u64(float2 a)
{
    return *reinterpret_cast<unsigned long long *>(&a);
}
__device__ __forceinline__ float2 as_f2(unsigned long long a)
{
    return *reinterpret_cast<float2 *>(&a);
}
__device__ __forceinline__ float2 cadd(float2 a, float2 b)
{
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(as_u64(a)), "l"(as_u64(b)));
    return as_f2(r);
}
__device__ __forceinline__ float2 csub(float2 a, float2 b)
{
    unsigned long long r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(as_u64(a)), "l"(as_u64(b)));
    return as_f2(r);
}
__device__ __forceinline__ float2 pmul(float2 a, float2 b)          // per-half product
{
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(as_u64(a)), "l"(as_u64(b)));
    return as_f2(r);
}
__device__ __forceinline__ float2 pfma(float2 a, float2 b, float2 c)  // per-half a*b+c
{
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(as_u64(a)), "l"(as_u64(b)), "l"(as_u64(c)));
    return as_f2(r);
}
__device__ __forceinline__ float2 bcast(float x) { return make_float2(x, x); }
__device__ __forceinline__ float2 mul_mi(float2 a) { return make_float2(a.y, -a.x); }   // a * (-i)
__device__ __forceinline__ float2 mul_pi(float2 a) { return make_float2(-a.y, a.x); }   // a * (+i)

__device__ __forceinline__ float2 cmul(float2 a, float2 b)
{   // a*b = a.x*b + i*(a.y*b): the half-swap and the sign ride on the FFMA2 addend, so this
    // is two instructions and no rotated copy of either operand is ever materialised
    return pfma(bcast(a.x), b, mul_pi(pmul(bcast(a.y), b)));
}

// a * exp(-2*pi*i*K/R), K and R compile-time
template <int K, int R>
__device__ __forceinline__ float2 cmul_w(float2 a)
{
    constexpr int k = ((K % R) + R) % R;
    if constexpr (k == 0) return a;
    else if constexpr (4 * k == R) return mul_mi(a);
    else if constexpr (2 * k == R) return make_float2(-a.x, -a.y);
    else if constexpr (4 * k == 3 * R) return mul_pi(a);
    else if constexpr (8 * k == R) {              // (1-i)/sqrt2
        constexpr float h = 0.70710678118654752440f;
        return pmul(bcast(h), cadd(a, mul_mi(a)));
    } else if constexpr (8 * k == 3 * R) {        // (-1-i)/sqrt2
        constexpr float h = 0.70710678118654752440f;
        return pmul(bcast(-h), csub(a, mul_mi(a)));
    } else if constexpr (8 * k == 5 * R) {        // (-1+i)/sqrt2
        constexpr float h = 0.70710678118654752440f;
        return pmul(bcast(-h), cadd(a, mul_mi(a)));
    } else if constexpr (8 * k == 7 * R) {        // (1+i)/sqrt2
        constexpr float h = 0.70710678118654752440f;
        return pmul(bcast(h), csub(a, mul_mi(a)));
    } else {
        constexpr float c = (float)cx_cos2pi(k, R);
        constexpr float sn = (float)(-cx_sin2pi(k, R));   // w = (c, sn)
        return pfma(a, bcast(c), mul_pi(pmul(a, bcast(sn))));   // scalar immediates, no constant pairs
    }
}

// ------------------------------------------------------------------ register DFTs
// Constant twiddles are never multiplied out.  Every register DFT exists in the form
// run_tw<K, RR>: the DFT of v[n] * w^n with w = exp(-2*pi*i*K/RR) (run = run_tw<0, R>).  A
// composite length hands its internal twiddles W_R^(n2*k1) down as the K of its sub-transforms
// (they are geometric in n2), so they all arrive at radix-2 / radix-4 butterflies of the form
// a +- w*b, which cost THREE packed instructions instead of four (cmul + add + sub):
//   w = c*(1 + i*t):  u = b + t*(i*b);  a + c*u;  a - c*u        (|c| >= |s|, t = s/c)
//   w = s*(i + t'):   u = i*b + t'*b;   a + s*u;  a - s*u        (otherwise,  t' = c/s)
// (the multiply-add form of Linzer & Feig / Goedecker).  A 64-point DFT is 482 packed
// instructions this way against 546 with the twiddles multiplied out.

constexpr int pick_factor(int r)
{
    if (r % 4 == 0) return 4;
    if (r % 2 == 0) return 2;
    for (int p = 3; p * p <= r; p += 2)
        if (r % p == 0) return p;
    return r;
}
constexpr bool is_base(int r) { return r == 1 || r == 2 || r == 4 || (r % 2 == 1 && pick_factor(r) == r); }
__host__ __device__ constexpr int mod_pos(int k, int r) { return ((k % r) + r) % r; }
__host__ __device__ constexpr double cx_abs(double x) { return x < 0 ? -x : x; }

// plus = a + w*b, minus = a - w*b, w = exp(-2*pi*i*K/RR)
template <int K, int RR>
__device__ __forceinline__ void bfly_tw(float2 a, float2 b, float2 &plus, float2 &minus)
{
    constexpr int k = mod_pos(K, RR);
    if constexpr (k == 0) {
        plus = cadd(a, b);
        minus = csub(a, b);
    } else if constexpr (4 * k == RR) {            // w = -i
        plus = cadd(a, mul_mi(b));
        minus = csub(a, mul_mi(b));
    } else if constexpr (2 * k == RR) {            // w = -1
        plus = csub(a, b);
        minus = cadd(a, b);
    } else if constexpr (4 * k == 3 * RR) {        // w = +i
        plus = cadd(a, mul_pi(b));
        minus = csub(a, mul_pi(b));
    } else {
        constexpr double c = cx_cos2pi(k, RR), s = -cx_sin2pi(k, RR);     // w = c + i*s
        if constexpr (cx_abs(c) >= cx_abs(s)) {
            constexpr float t = (float)(s / c), cf = (float)c;
            const float2 u = pfma(mul_pi(b), bcast(t), b);                 // b + t*(i*b)
            plus = pfma(u, bcast(cf), a);
            minus = pfma(u, bcast(-cf), a);
        } else {
            constexpr float t = (float)(c / s), sf = (float)s;
            const float2 u = pfma(b, bcast(t), mul_pi(b));                 // i*b + t*b
            plus = pfma(u, bcast(sf), a);
            minus = pfma(u, bcast(-sf), a);
        }
    }
}

template <int R, bool BASE = is_base(R)>
struct Dft;

template <>
struct Dft<1, true> {
    template <int K, int RR>
    static __device__ __forceinline__ void run_tw(float2 *) {}
    static __device__ __forceinline__ void run(float2 *) {}
};

template <>
struct Dft<2, true> {
    template <int K, int RR>
    static __device__ __forceinline__ void run_tw(float2 *v)
    {
        float2 a = v[0], b = v[1];
        bfly_tw<K, RR>(a, b, v[0], v[1]);
    }
    static __device__ __forceinline__ void run(float2 *v) { run_tw<0, 2>(v); }
};

template <>
struct Dft<4, true> {
    // inputs u0, w*u1, w^2*u2, w^3*u3:  a0,a1 = u0 +- w^2*u2;  s,d = u1 +- w^2*u3;
    // X0,X2 = a0 +- w*s;  X1,X3 = a1 +- (-i*w)*d
    template <int K, int RR>
    static __device__ __forceinline__ void run_tw(float2 *v)
    {
        static_assert(RR % 4 == 0, "radix 4 inside a length that 4 does not divide");
        float2 a0, a1, s, d;
        bfly_tw<2 * K, RR>(v[0], v[2], a0, a1);
        bfly_tw<2 * K, RR>(v[1], v[3], s, d);
        bfly_tw<K, RR>(a0, s, v[0], v[2]);
        bfly_tw<K + RR / 4, RR>(a1, d, v[1], v[3]);
    }
    static __device__ __forceinline__ void run(float2 *v) { run_tw<0, 4>(v); }
};

// odd prime P: pair x[n] with x[P-n]
template <int P>
struct Dft<P, true> {
    template <int K, int RR>
    static __device__ __forceinline__ void run_tw(float2 *v)
    {
        if constexpr (mod_pos(K, RR) != 0) {
            static_for<1, P>([&](auto nn) {
                constexpr int n = decltype(nn)::value;
                v[n] = cmul_w<K * n, RR>(v[n]);
            });
        }
        run(v);
    }
    static __device__ __forceinline__ void run(float2 *v)
    {
        constexpr int H = (P - 1) / 2;
        float2 s[H + 1], d[H + 1];
#pragma unroll
        for (int n = 1; n <= H; n++) {
            s[n] = cadd(v[n], v[P - n]);
            d[n] = csub(v[n], v[P - n]);
        }
        float2 x0 = v[0];
        float2 acc = x0;
#pragma unroll
        for (int n = 1; n <= H; n++) acc = cadd(acc, s[n]);
        v[0] = acc;
        static_for<1, H + 1>([&](auto kk) {
            constexpr int k = decltype(kk)::value;
            float2 re = x0, im = make_float2(0.f, 0.f);
            static_for<1, H + 1>([&](auto nn) {
                constexpr int n = decltype(nn)::value;
                constexpr float c = (float)cx_cos2pi(n * k, P);
                constexpr float sn = (float)cx_sin2pi(n * k, P);
                re = pfma(s[n], bcast(c), re);
                if constexpr (n == 1) im = pmul(d[n], bcast(sn));
                else im = pfma(d[n], bcast(sn), im);
            });
            // X[k] = re - i*im ; X[P-k] = re + i*im
            v[k] = cadd(re, mul_mi(im));
            v[P - k] = csub(re, mul_mi(im));
        });
    }
};

// composite R = A*B: n = B*n1 + n2, k = k1 + A*k2
template <int R>
struct Dft<R, false> {
    static constexpr int A = pick_factor(R);
    static constexpr int B = R / A;
    // DFT of v[n] * w^n, w = exp(-2*pi*i*K/RR): w^n = (w^B)^n1 * w^n2; the first factor is the
    // twiddle progression of the length-A transforms, the second joins the internal twiddle
    // W_R^(n2*k1) = exp(-2*pi*i*n2*k1*(RR/R)/RR) as the progression of the length-B ones
    template <int K, int RR>
    static __device__ __forceinline__ void run_tw(float2 *v)
    {
        static_assert(RR % R == 0, "sub-transform length divides the outer one");
        float2 t[R];
        static_for<0, B>([&](auto nn2) {
            constexpr int n2 = decltype(nn2)::value;
            float2 a[A];
#pragma unroll
            for (int n1 = 0; n1 < A; n1++) a[n1] = v[B * n1 + n2];
            Dft<A>::template run_tw<mod_pos(K * B, RR), RR>(a);
#pragma unroll
            for (int k1 = 0; k1 < A; k1++) t[k1 * B + n2] = a[k1];
        });
        static_for<0, A>([&](auto kk1) {
            constexpr int k1 = decltype(kk1)::value;
            float2 b[B];
#pragma unroll
            for (int n2 = 0; n2 < B; n2++) b[n2] = t[k1 * B + n2];
            Dft<B>::template run_tw<mod_pos(K + k1 * (RR / R), RR), RR>(b);
#pragma unroll
            for (int k2 = 0; k2 < B; k2++) v[k1 + A * k2] = b[k2];
        });
    }
    static __device__ __forceinline__ void run(float2 *v) { run_tw<0, R>(v); }
};

// v[r] *= w1^r for r = 1..R-1, powers by a balanced product tree (depth log2 R)
template <int R>
__device__ __forceinline__ void twiddle_powers(float2 *v, float2 w1)
{
    if constexpr (R >= 64 && R % 8 == 0) {
        // large radix: r = 8a + b, w1^r = (w1^8)^a * w1^b.  The same number of complex products
        // as the tree below, but only 7 + R/8 powers are ever live instead of R/2.
        constexpr int A = R / 8;
        float2 wb[8], wa[A];
        wb[1] = w1;
#pragma unroll
        for (int b = 2; b < 8; b++) wb[b] = cmul(wb[b / 2], wb[b - b / 2]);
        wa[1] = cmul(wb[4], wb[4]);
#pragma unroll
        for (int q = 2; q < A; q++) wa[q] = cmul(wa[q / 2], wa[q - q / 2]);
#pragma unroll
        for (int r = 1; r < R; r++) {
            if (r % 8) v[r] = cmul(v[r], wb[r % 8]);
            if (r / 8) v[r] = cmul(v[r], wa[r / 8]);
        }
        return;
    }
    float2 w[R];
    w[0] = make_float2(1.f, 0.f);
    if (R > 1) w[1] = w1;
#pragma unroll
    for (int r = 2; r < R; r++) w[r] = cmul(w[r / 2], w[r - r / 2]);
#pragma unroll
    for (int r = 1; r < R; r++) v[r] = cmul(v[r], w[r]);
}

// ------------------------------------------------------------------ plan
template <int N_, int T_, int G_, int R0_, int R1_, int R2_ = 1, int R3_ = 1>
struct Plan {
    static constexpr int N = N_, T = T_, G = G_;
    static constexpr int R0 = R0_, R1 = R1_, R2 = R2_, R3 = R3_;
    static constexpr int K = (R3_ > 1) ? 4 : (R2_ > 1) ? 3 : 2;
    static constexpr int RL = (K == 4) ? R3_ : (K == 3) ? R2_ : R1_;
    static constexpr int ML = N_ / RL;                       // row length
    static constexpr int PAD = (ML % 4 == 0) ? 2 : 4;        // keeps (ML+PAD)/2 odd
    static constexpr int PITCH = ML + PAD;
    static constexpr int FFT_ELEMS = RL * PITCH;             // float2 per block in smem
    static constexpr size_t SMEM = (size_t)G_ * FFT_ELEMS * sizeof(float2);
    static_assert(R0_ * R1_ * R2_ * R3_ == N_, "radices must multiply to N");
    static_assert(R0_ % 2 == 0 && ML % 2 == 0, "chunk scatter uses 16-byte stores");
    static_assert(G_ == 1 || T_ == G_ * ML, "multi-block CTAs need one last-pass round");
    // Blocks that fill most of an SM's shared memory leave one to three CTAs per SM, too few to
    // hide the load phase behind other CTAs' butterflies.  Those plans run persistent CTAs that
    // fetch the next block's pass-0 samples into registers before the last pass of the current
    // one (s16 input: one register per sample).
    static constexpr bool PERSIST = (G_ == 1) && (N_ >= 9600) && (SMEM > 113 * 1024);   // one CTA per SM (at two, N = 9600 is faster as ordinary CTAs)
    // CTAs per SM the kernel is compiled for: what shared memory allows, at the register budget
    // the largest register DFT needs.  Radix <= 16 fits 48 registers (4096 = 16^3 then keeps five
    // CTAs per SM instead of slipping to four); radix 32 fits 80, and a 256-thread CTA at 81..88
    // registers drops from three per SM to two (measured on N = 512: 0.46 against 0.60 of peak).
    // Odd radices and the persistent plans are left to the compiler (0 = unspecified).
    static constexpr int RMAX = (R0_ > R1_ ? R0_ : R1_) > (R2_ > R3_ ? R2_ : R3_) ? (R0_ > R1_ ? R0_ : R1_) : (R2_ > R3_ ? R2_ : R3_);
    static constexpr int REG_BUDGET = (RMAX <= 16) ? 48 : 80;
    static constexpr int MINB_SMEM = (int)((227 * 1024) / (SMEM + 1024));
    static constexpr int MINB_REGS = 65536 / (T_ * REG_BUDGET);
    static constexpr int MINB_FIT = (MINB_SMEM < MINB_REGS ? MINB_SMEM : MINB_REGS) < 1 ? 1 : (MINB_SMEM < MINB_REGS ? MINB_SMEM : MINB_REGS);
    static constexpr int MINB = (PERSIST || RMAX > 32 || (RMAX & (RMAX - 1)) != 0) ? 0 : MINB_FIT;
    // Persistent plans keep the twiddle bases of every pass in shared memory behind the block (the
    // block leaves room: one CTA per SM): R0 values for the first middle pass, R0*R1 for the
    // second, ML for the last -- a shared-memory load where every butterfly waited for L2.
    static constexpr int TW1 = (K >= 3) ? R0_ : 0;
    static constexpr int TW2 = (K >= 4) ? R0_ * R1_ : 0;
    static constexpr int TW_ELEMS = TW1 + TW2 + ML;
    static constexpr bool TW_SMEM = PERSIST && (SMEM + TW_ELEMS * sizeof(float2) + 2048 <= 227 * 1024);
    static constexpr size_t SMEM_PERSIST = SMEM + (TW_SMEM ? TW_ELEMS * sizeof(float2) : 0);
    // The same tables for the ordinary (one CTA per block) three- and four-pass plans, where they
    // cost no CTA per SM: each thread fetches its share into registers before pass 0 and stores
    // it to shared memory behind pass 0, so the fetch hides behind the pass-0 loads.
    static constexpr int TW_PER_THREAD = (TW_ELEMS + T_ - 1) / T_;
    // (N >= 8192 only: measured +5.7 % at 8192 and +4.3 % at 9600 for s16 input; at 4800 the extra
    // registers cost a CTA per SM, -8 %, and 2048 / 4410 do not move)
    static constexpr bool TW_SMEM_NP = !PERSIST && G_ == 1 && K >= 3 && N_ >= 8192 && TW_PER_THREAD <= 4 &&
                                       (int)((227 * 1024) / (SMEM + TW_ELEMS * sizeof(float2) + 1024)) == (int)((227 * 1024) / (SMEM + 1024));
    static constexpr size_t SMEM_TW = SMEM + TW_ELEMS * sizeof(float2);
    static constexpr bool GROUP_IN = true;
    static constexpr int NB0 = N_ / R0_;
    static constexpr int PRE_IT = (NB0 + T_ - 1) / T_;        // pass-0 butterflies per thread
};

struct Args {
    const void *in;       // float2[nblocks][N] or int16x2[nblocks][N]
    float *out;           // float[nblocks][N+2] (PSD) or float2[nblocks][N] (spectrum)
    int32_t *peak_bin;    // nullable
    const float2 *tw;     // exp(-2*pi*i*t/N), t in [0,N)
    int nblocks;
    int rate;
    float cf;             // (2/N)^2, times 1/32767^2 for s16 input
    float db_off;         // 10*log10(cf): psd = 10*log10(re^2+im^2) + db_off, one FFMA behind the logarithm
    int ic, qc;           // I/Q DC correction added with 16-bit wrap (s16 input)
    int pf_dist;          // CTAs resident on the device (0: no L2 prefetch), see fft_kernel
    // split plans (SPLIT = 2, see fft_kernel): nblocks counts HALF blocks
    const float2 *tw2;          // exp(-2*pi*i*c/(2N)), c in [0, N)
    unsigned long long *best;   // [real blocks] packed (dB key, ~bin) of the halves seen so far; zero between launches
    unsigned *cnt;              // [real blocks] halves that have reported; zero between launches
    const float *win;           // [N * SPLIT] window of jsdr_fft_set_window, read by the WIN instantiations only
};

__device__ __forceinline__ unsigned ordered_key(float v)
{   // monotone float -> uint (never 0 for a finite or +inf v); -0.0 counts as +0.0
    unsigned u = __float_as_uint(v + 0.0f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// MUFU.LG2 without the denormal pre-scaling of __log2f: power below 1.2e-38
// (-379 dB) reads as -inf, exactly as an all-zero bin does (SURVEY Q4).
__device__ __forceinline__ float lg2_approx(float x)
{
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// exact s16 pair -> float pair: sign-extend on the ALU (PRMT with sign replication, arithmetic
// shift) and I2FP.F32.S32, four instructions per pair and nothing on the FMA pipe, the one this
// kernel saturates.  It is 0.5-2 % faster than biasing to unsigned, splicing into the mantissa of
// 2^23 and subtracting 2^23 + 32768 with one FADD2; I2F.S16 straight from the halves is two
// instructions, but on the XU pipe next to MUFU.LG2, and 2-3 % slower than the splice.
// (prmt in PTX: selector bit 3 replicates the chosen byte's sign; __byte_perm masks it off.)
// The 1/32767 of JavaAudio.java:283 is folded into cf (the transform is linear).
__device__ __forceinline__ float2 s16_bits_to_float(uint32_t w)
{
    float a, b;
    int lo;
    asm("prmt.b32 %0, %1, 0, 0x9910;" : "=r"(lo) : "r"(w));
    asm("cvt.rn.f32.s32 %0, %1;" : "=f"(a) : "r"(lo));
    asm("cvt.rn.f32.s32 %0, %1;" : "=f"(b) : "r"((int)w >> 16));
    return make_float2(a, b);
}

template <class P, int IN>
__device__ __forceinline__ float2 load_sample(const Args &a, long blk, int n)
{
    if constexpr (IN == IN_F32) {
        return ldg_stream_f2(reinterpret_cast<const float2 *>(a.in) + blk * P::N + n);
    } else {
        uint32_t w = ldg_stream_u32(reinterpret_cast<const uint32_t *>(a.in) + blk * P::N + n);
        // JavaAudio.java:281-288: s += (short)ic with 16-bit wrap, then (float)s.
        // The 1/32767 scale is folded into cf (the transform is linear).
        if (a.ic | a.qc) {   // uniform branch: the correction is normally zero
            w = (((w & 0xffffu) + (unsigned)a.ic) & 0xffffu) | ((((w >> 16) + (unsigned)a.qc) & 0xffffu) << 16);
        }
        return s16_bits_to_float(w);
    }
}

// jsdr_fft_set_window: sample t of the block times win[t], one binary32 rounding per component.
// __fmul_rn and not '*': under nvcc's default -fmad=true ptxas may fuse a plain product into the
// first butterfly's add, which would round once where the contract (jsdrcuda.h) rounds twice.
// The table is the same for every block, so the loads hit in L1.
__device__ __forceinline__ float2 apply_win(float2 v, const float *win, int t)
{
    const float w = __ldg(win + t);
    return make_float2(__fmul_rn(v.x, w), __fmul_rn(v.y, w));
}

template <int R, int M>
__device__ __forceinline__ void load_strided(float2 *v, const float2 *p)
{
#pragma unroll
    for (int r = 0; r < R; r++) v[r] = p[r * M];
}

// middle pass p: sub-transform length L = M*R, butterfly stride M
template <class P, int R, int M, bool TWS = false>
__device__ __forceinline__ void middle_pass(float2 *sm, const float2 *__restrict__ tw, int tid)
{
    constexpr int L = M * R;
    constexpr int NB = P::N / R;
    for (int U = tid; U < P::G * NB; U += P::T) {
        int g = U / NB, u = U - g * NB;
        int j = u % M, blk = u / M;
        int lin = blk * L + j;
        float2 *p = sm + g * P::FFT_ELEMS + lin + (lin / P::ML) * P::PAD;
        float2 v[R];
        load_strided<R, M>(v, p);
        float2 w1;
        if constexpr (TWS) w1 = tw[j];            // shared-memory copy of tw[j * N/L], j < M
        else w1 = __ldg(tw + j * (P::N / L));
        twiddle_powers<R>(v, w1);
        Dft<R>::run(v);
#pragma unroll
        for (int r = 0; r < R; r++) p[r * M] = v[r];
    }
}

// SPLIT = 2 ("split plan"): a block of 2N samples is transformed as two independent N-point
// transforms, one CTA each, by one radix-2 decimation-in-frequency step folded into the loads of
// pass 0: CTA h = 0 transforms x[n] + x[n+N] and owns the even bins, CTA h = 1 transforms
// (x[n] - x[n+N]) * w_2N^n and owns the odd bins.  Lengths whose whole block fills an SM's shared
// memory (one CTA per SM, every warp in step between barriers) then run two (or more) CTAs per
// SM that drift apart.  The block maximum is combined through one 64-bit atomicMax per half
// (dB key in the high word, complemented bin in the low one: first strict maximum as at
// fft.java:208-211) and the half that reports last publishes peak Hz / dB (:214-224).
// WIN: every converted sample of pass 0 times a.win[t] (apply_win) before the first butterfly; a
// handle without a window runs the WIN = false instantiations, which carry no code for it.
template <class P, int IN, int OUT, int SPLIT = 1, bool WIN = false>
__global__ void __launch_bounds__(P::T, P::MINB) fft_kernel(const Args a)
{
    static_assert(SPLIT == 1 || (SPLIT == 2 && P::G == 1), "split plans take one half block per CTA");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2 *sm = reinterpret_cast<float2 *>(smem_raw);
    __shared__ unsigned s_max[P::G];
    __shared__ int s_idx[P::G];

    const int tid = threadIdx.x;
    constexpr int N = P::N;
    constexpr int NR = N * SPLIT;                 // length of the block in memory
    // persistent only where the register prefetch exists (s16 input: one register per sample);
    // float input keeps one CTA per block and the L2 prefetch (measured: 0.50 -> 0.61 at 16384)
    constexpr bool PERSIST = P::PERSIST && IN == IN_S16 && SPLIT == 1;
    // Register prefetch only where one round of pass 0 covers the block (PRE_IT = 1: 16384).  With
    // two rounds (19200: 2 x 16 values beside the butterflies at a 96-register budget) the compiler
    // keeps pre[] in LOCAL memory, and the store that spills a value waits for its load: the
    // "prefetch" stalled every warp in front of the last pass (ncu source page: STL, long scoreboard,
    // 8 % of all stall samples).  Those plans ask for the next block with one bulk L2 prefetch
    // instead, as the non-persistent plans do, and load pass 0 from L2.
    constexpr bool PREFETCH = PERSIST && P::PRE_IT == 1;
    constexpr bool L2_NEXT = PERSIST && !PREFETCH;
    // ... and fetch BOTH rounds of their own pass 0 before the first butterfly (the shared-memory
    // stores of round one would otherwise hold back the loads of round two): pre[] then lives
    // only inside pass 0 and stays in registers.
    constexpr bool EARLY = IN == IN_S16 && SPLIT == 1 && P::G == 1 && !PREFETCH &&
                           P::PRE_IT >= 2 && P::PRE_IT * P::R0 <= 40;       // (19200: 2 x 16; 4410: 2 x 10)
    constexpr bool PRE = PREFETCH || EARLY;

    // pass-0 samples of the next block (persistent plans, s16 input)
    uint32_t pre[PRE ? P::PRE_IT : 1][PRE ? P::R0 : 1];
    auto prefetch = [&](long blk) {
        if constexpr (PRE) {
            const uint32_t *src = reinterpret_cast<const uint32_t *>(a.in) + blk * N;
#pragma unroll
            for (int it = 0; it < P::PRE_IT; it++) {
                const int c = tid + it * P::T;
                if (c < P::NB0) {
#pragma unroll
                    for (int m = 0; m < P::R0; m++) pre[it][m] = ldg_stream_u32(src + c + m * P::NB0);
                }
            }
        }
    };
    if constexpr (PREFETCH) {
        if ((long)blockIdx.x < a.nblocks) prefetch(blockIdx.x);
    }

    constexpr bool TWN = P::TW_SMEM_NP && SPLIT == 1;            // ordinary plans: through registers, see Plan
    constexpr bool TWP = P::TW_SMEM && PERSIST;
    constexpr bool TWS = TWP || TWN;
    float2 *tw_s1 = sm + P::G * P::FFT_ELEMS;      // [TW1]  tw[j * N/(R0*R1)]
    float2 *tw_s2 = tw_s1 + P::TW1;                // [TW2]  tw[j * N/(R0*R1*R2)]
    float2 *tw_sl = tw_s2 + P::TW2;                // [ML]   tw[j]
    float2 twr[TWN ? P::TW_PER_THREAD : 1];
    if constexpr (TWN) {
#pragma unroll
        for (int k = 0; k < P::TW_PER_THREAD; k++) {
            const int i = tid + k * P::T;
            if (i < P::TW_ELEMS) {
                const int src = (i < P::TW1) ? i * (N / (P::R0 * P::R1))
                              : (i < P::TW1 + P::TW2) ? (i - P::TW1) * (N / (P::R0 * P::R1 * (P::K >= 4 ? P::R2 : 1)))
                              : i - P::TW1 - P::TW2;
                twr[k] = __ldg(a.tw + src);
            }
        }
    }
    if constexpr (TWP) {
        for (int i = tid; i < P::TW1; i += P::T) tw_s1[i] = __ldg(a.tw + i * (N / (P::R0 * P::R1)));
        if constexpr (P::K >= 4)
            for (int i = tid; i < P::TW2; i += P::T) tw_s2[i] = __ldg(a.tw + i * (N / (P::R0 * P::R1 * P::R2)));
        for (int i = tid; i < P::ML; i += P::T) tw_sl[i] = __ldg(a.tw + i);
        // (visible to every thread after the barrier that follows pass 0)
    }

    // one pass for ordinary plans (a CTA owns blocks blk0 .. blk0+G-1); persistent plans loop
    long blk0 = (long)blockIdx.x * P::G;
    const long blk_step = gridDim.x;

    // Ordinary plans: CTAs start in blockIdx order, so the CTA that takes this one's place is
    // about pf_dist further on.  One bulk prefetch pulls its input into L2 now; its pass-0 loads
    // then wait for L2 instead of HBM (the few resident CTAs of the large-radix plans cannot hide
    // an HBM round trip behind each other).  Only the 16-byte-aligned interior of the range is
    // touched, and only whole groups inside the batch.
    if constexpr (!PERSIST) {
        if (tid == 0 && a.pf_dist > 0) {
            const long nb = blk0 + (long)a.pf_dist * P::G;
            if (nb + P::G <= a.nblocks) {
                constexpr size_t EL = (IN == IN_S16) ? 4 : 8;
                // (split plans: half block nb is N contiguous samples too — the two CTAs of a block
                // bring in one half each, and each of them then reads both)
                const size_t lo = (reinterpret_cast<size_t>(a.in) + (size_t)nb * N * EL + 15) & ~(size_t)15;
                const size_t hi = (reinterpret_cast<size_t>(a.in) + (size_t)(nb + P::G) * N * EL) & ~(size_t)15;
                if (hi > lo)
                    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(lo), "r"((unsigned)(hi - lo)) : "memory");
            }
        }
    }
    do {
    if constexpr (L2_NEXT) {
        if (tid == 0 && blk0 + blk_step < a.nblocks) {
            const size_t lo = (reinterpret_cast<size_t>(a.in) + (size_t)(blk0 + blk_step) * N * 4 + 15) & ~(size_t)15;
            const size_t hi = (reinterpret_cast<size_t>(a.in) + (size_t)(blk0 + blk_step + 1) * N * 4) & ~(size_t)15;
            if (hi > lo) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(lo), "r"((unsigned)(hi - lo)) : "memory");
        }
    }

    // Plans whose blocks keep the same warp in every pass (two passes, NB0 == ML == 32: N = 1024)
    // never exchange data between warps: warp convergence replaces the CTA barrier at every pass
    // boundary (measured 0.69 -> 0.74 of peak).  The same with a named barrier per two-warp
    // block made N = 4096 slower (0.66 -> 0.61), so that plan keeps the CTA-wide barrier.
    constexpr bool GROUP_SYNC = (P::G > 1) && (P::K == 2) && (P::NB0 == P::ML) && (P::ML == 32) && (P::T == P::G * P::ML);
    auto block_sync = [&]() {
        if constexpr (!GROUP_SYNC) __syncthreads();
        else if constexpr (P::ML == 32) __syncwarp();
        else asm volatile("bar.sync %0, %1;" ::"r"(1 + tid / P::ML), "n"(P::ML) : "memory");
    };
    if constexpr (GROUP_SYNC) {
        if (OUT == OUT_PSD && tid % P::ML == 0) {
            s_max[tid / P::ML] = 0u;
            s_idx[tid / P::ML] = 0x7fffffff;
        }
    } else if (OUT == OUT_PSD && tid < P::G) {
        s_max[tid] = 0u;
        s_idx[tid] = 0x7fffffff;
    }

    // ---------------- pass 0: HBM -> registers -> DFT_R0 -> digit-reversed chunk
    {
        constexpr int R0 = P::R0;
        constexpr int NB0 = N / R0;
        if constexpr (EARLY) prefetch(blk0);
#pragma unroll
        for (int it = 0; it < (PRE ? P::PRE_IT : 1); it++) {
        for (int U = PRE ? tid + it * P::T : tid; U < P::G * NB0; U += PRE ? P::G * NB0 : P::T) {
            int g = U / NB0, c = U - g * NB0;
            long blk = blk0 + g;
            if (blk >= a.nblocks) continue;
            float2 v[R0];
            if constexpr (SPLIT == 2) {
                // one radix-2 decimation-in-frequency step on the way in (see above), eight inputs of
                // the butterfly at a time so that only 2 x 8 raw values are ever live beside v[]
                const long rblk = blk >> 1;
                const int h = (int)(blk & 1);
                constexpr int CHK = (R0 % 8 == 0) ? 8 : (R0 % 5 == 0) ? 5 : (R0 % 4 == 0) ? 4 : 2;
                // w_2N^(c + m*NB0) = w_2N^c * exp(-2*pi*i*m/(2*R0)): one table value, constant rotations
                const float2 wc = h ? __ldg(a.tw2 + c) : make_float2(1.f, 0.f);
                static_for<0, R0 / CHK>([&](auto kk) {
                    constexpr int m0 = decltype(kk)::value * CHK;
                    float2 va[CHK], vb[CHK];
                    if constexpr (IN == IN_S16) {
                        const uint32_t *src = reinterpret_cast<const uint32_t *>(a.in) + rblk * NR + c;
                        uint32_t wa[CHK], wb[CHK];
#pragma unroll
                        for (int i = 0; i < CHK; i++) {
                            wa[i] = ldg_stream_u32(src + (m0 + i) * NB0);
                            wb[i] = ldg_stream_u32(src + N + (m0 + i) * NB0);
                        }
                        if (a.ic | a.qc) {
#pragma unroll
                            for (int i = 0; i < CHK; i++) {
                                wa[i] = (((wa[i] & 0xffffu) + (unsigned)a.ic) & 0xffffu) | ((((wa[i] >> 16) + (unsigned)a.qc) & 0xffffu) << 16);
                                wb[i] = (((wb[i] & 0xffffu) + (unsigned)a.ic) & 0xffffu) | ((((wb[i] >> 16) + (unsigned)a.qc) & 0xffffu) << 16);
                            }
                        }
#pragma unroll
                        for (int i = 0; i < CHK; i++) {
                            va[i] = s16_bits_to_float(wa[i]);
                            vb[i] = s16_bits_to_float(wb[i]);
                        }
                    } else {
                        const float2 *src = reinterpret_cast<const float2 *>(a.in) + rblk * NR + c;
#pragma unroll
                        for (int i = 0; i < CHK; i++) {
                            va[i] = ldg_stream_f2(src + (m0 + i) * NB0);
                            vb[i] = ldg_stream_f2(src + N + (m0 + i) * NB0);
                        }
                    }
                    if constexpr (WIN) {                // samples n and n + N of the whole block
#pragma unroll
                        for (int i = 0; i < CHK; i++) {
                            va[i] = apply_win(va[i], a.win, c + (m0 + i) * NB0);
                            vb[i] = apply_win(vb[i], a.win, N + c + (m0 + i) * NB0);
                        }
                    }
                    if (h == 0) {
#pragma unroll
                        for (int i = 0; i < CHK; i++) v[m0 + i] = cadd(va[i], vb[i]);
                    } else {
                        static_for<0, CHK>([&](auto ii) {
                            constexpr int i = decltype(ii)::value;
                            v[m0 + i] = cmul(cmul_w<m0 + i, 2 * R0>(csub(va[i], vb[i])), wc);
                        });
                    }
                });
            } else if constexpr (IN == IN_S16 && P::GROUP_IN) {
                uint32_t w[R0];
                if constexpr (PRE) {
#pragma unroll
                    for (int m = 0; m < R0; m++) w[m] = pre[it][m];
                } else {
                    const uint32_t *src = reinterpret_cast<const uint32_t *>(a.in) + blk * N + c;
#pragma unroll
                    for (int m = 0; m < R0; m++) w[m] = ldg_stream_u32(src + m * NB0);
                }
                // JavaAudio.java:281-288: s += (short)ic with 16-bit wrap.  A real (uniform) branch
                // around the whole group: the correction is normally zero and predicated-off
                // instructions would still take issue slots.
                if (a.ic | a.qc) {
#pragma unroll
                    for (int m = 0; m < R0; m++)
                        w[m] = (((w[m] & 0xffffu) + (unsigned)a.ic) & 0xffffu) | ((((w[m] >> 16) + (unsigned)a.qc) & 0xffffu) << 16);
                }
#pragma unroll
                for (int m = 0; m < R0; m++) v[m] = s16_bits_to_float(w[m]);
                if constexpr (WIN) {
#pragma unroll
                    for (int m = 0; m < R0; m++) v[m] = apply_win(v[m], a.win, c + m * NB0);
                }
            } else {
#pragma unroll
                for (int m = 0; m < R0; m++) v[m] = load_sample<P, IN>(a, blk, c + m * NB0);
                if constexpr (WIN) {
#pragma unroll
                    for (int m = 0; m < R0; m++) v[m] = apply_win(v[m], a.win, c + m * NB0);
                }
            }
            Dft<R0>::run(v);
            int pos;
            if constexpr (P::K == 2) {
                pos = c * P::PITCH;
            } else if constexpr (P::K == 3) {
                int r2 = c % P::R2, r1 = c / P::R2;
                pos = r2 * P::PITCH + r1 * R0;
            } else {
                int r3 = c % P::R3, t = c / P::R3;
                int r2 = t % P::R2, r1 = t / P::R2;
                pos = r3 * P::PITCH + r2 * (R0 * P::R1) + r1 * R0;
            }
            // 64-bit stores: pairing the outputs for 128-bit ones costs more register moves
            // than the stores it saves (the shared-memory wavefront count is the same)
            const unsigned dst = (unsigned)__cvta_generic_to_shared(sm + g * P::FFT_ELEMS + pos);
            static_for<0, R0>([&](auto mm) {
                constexpr int m = decltype(mm)::value;
                asm volatile("st.shared.v2.f32 [%0+%1], {%2,%3};" ::"r"(dst), "n"(m * 8), "f"(v[m].x), "f"(v[m].y) : "memory");
            });
        }
        }
    }
    if constexpr (TWN) {
#pragma unroll
        for (int k = 0; k < P::TW_PER_THREAD; k++) {
            const int i = tid + k * P::T;
            if (i < P::TW_ELEMS) tw_s1[i] = twr[k];
        }
    }
    block_sync();

    // ---------------- middle passes (in place)
    if constexpr (P::K >= 3) {
        if constexpr (TWS) middle_pass<P, P::R1, P::R0, true>(sm, tw_s1, tid);
        else middle_pass<P, P::R1, P::R0>(sm, a.tw, tid);
        __syncthreads();
    }
    if constexpr (P::K >= 4) {
        if constexpr (TWS) middle_pass<P, P::R2, P::R0 * P::R1, true>(sm, tw_s2, tid);
        else middle_pass<P, P::R2, P::R0 * P::R1>(sm, a.tw, tid);
        __syncthreads();
    }

    // ---------------- last pass + epilogue
    if constexpr (PREFETCH) {
        if (blk0 + blk_step < a.nblocks) prefetch(blk0 + blk_step);   // in flight behind the last pass
    }
    {
        constexpr int RL = P::RL, ML = P::ML;
        // running first-strict-maximum exactly as fft.java:201-211: m starts at
        // -Float.MAX_VALUE, a bin wins only if m < psd (NaN and -inf never do)
        float best = -3.4028234663852886e38f;
        int my_g = 0;
        // the dB values stay in registers (one per bin, replacing the two of the spectrum value)
        // until the block's maximum is known: only the thread that holds it looks for the bin
        constexpr int ITERS = (P::G * ML + P::T - 1) / P::T;
        float db[OUT == OUT_PSD ? ITERS : 1][OUT == OUT_PSD ? RL : 1];
#pragma unroll
        for (int it = 0; it < ITERS; it++) {
            const int U = tid + it * P::T;
            if (ITERS * P::T != P::G * ML && U >= P::G * ML) break;
            int g = U / ML, j = U - g * ML;
            long blk = blk0 + g;
            my_g = g;
            if (blk >= a.nblocks) {
                if constexpr (OUT == OUT_PSD) {
#pragma unroll
                    for (int q = 0; q < RL; q++) db[it][q] = -3.4028234663852886e38f;
                }
                continue;
            }
            float2 v[RL];
            const float2 *p = sm + g * P::FFT_ELEMS + j;
#pragma unroll
            for (int r = 0; r < RL; r++) v[r] = p[r * P::PITCH];
            float2 w1;
            if constexpr (TWS) w1 = tw_sl[j];
            else w1 = __ldg(a.tw + j);
            twiddle_powers<RL>(v, w1);
            Dft<RL>::run(v);
            // where this (half) block's bin k goes: bin SPLIT*k + h of block blk / SPLIT
            const long rblk = blk / SPLIT;
            const int h = (int)(blk % SPLIT);
            if constexpr (OUT == OUT_SPECTRUM) {
                float2 *spec = reinterpret_cast<float2 *>(a.out) + rblk * NR + h;
#pragma unroll
                for (int q = 0; q < RL; q++) stg_stream_f2(spec + SPLIT * (j + q * ML), v[q]);
            } else {
                float *psd = a.out + rblk * (long)(NR + 2) + h;
#pragma unroll
                for (int q = 0; q < RL; q++) {
                    // fft.java:207 (re*re + im*im) * cf -> dB.  The scale is applied behind the logarithm
                    // and the sum of squares is one multiply and one FMA: 1e-7 relative in power
                    // (4e-7 dB) from the reference's float sequence, far inside the 1e-4 tolerance.
                    float pw = fmaf(v[q].x, v[q].x, v[q].y * v[q].y);
                    // 10*log10(x) = 10*log10(2) * log2(x); MUFU.LG2 is accurate to ~1e-7 in log2
                    db[it][q] = fmaf(3.0102999566398120f, lg2_approx(pw), a.db_off);
                    stg_stream_f32(psd + SPLIT * (j + q * ML), db[it][q]);
                    // only the running maximum here (FMNMX; NaN never wins, and neither does
                    // anything <= -Float.MAX_VALUE)
                    best = fmaxf(best, db[it][q]);
                }
            }
        }
        const unsigned best_key = (best > -3.4028234663852886e38f) ? ordered_key(best) : 0u;
        if constexpr (OUT == OUT_PSD) {
            // first strict maximum (fft.java:208-211): max value, lowest bin among equals
            constexpr bool WARP_UNIFORM = (P::G == 1) || (ML % 32 == 0);
            unsigned k1 = best_key;
            if constexpr (WARP_UNIFORM) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) k1 = max(k1, __shfl_xor_sync(0xffffffffu, k1, o));
                if ((tid & 31) == 0 && k1 != 0u) atomicMax(&s_max[my_g], k1);
            } else {
                if (k1 != 0u) atomicMax(&s_max[my_g], k1);
            }
            block_sync();
            unsigned gmax = s_max[my_g];
            if (best_key != 0u && best_key == gmax) {
                // one thread per block as a rule: the lowest of its bins that equals the maximum
                // (what the strict '<' of :208 keeps), from the registers
                int best_idx = 0x7fffffff;
#pragma unroll
                for (int it = 0; it < ITERS; it++) {
                    const int U = tid + it * P::T;
                    const int j = U - (U / ML) * ML;
#pragma unroll
                    for (int q = 0; q < RL; q++)
                        if (db[it][q] == best) best_idx = min(best_idx, j + q * ML);
                }
                atomicMin(&s_idx[my_g], best_idx);
            }
            block_sync();
            // one writer per block: the block's first thread where blocks synchronise on their own
            const int wg = GROUP_SYNC ? tid / P::ML : tid;
            if ((GROUP_SYNC ? (tid % P::ML == 0) : (tid < P::G)) && blk0 + wg < a.nblocks) {
                long blk = blk0 + wg;
                unsigned key = s_max[wg];
                int bin = (key != 0u) ? s_idx[wg] : -1;
                bool publish = true;
                if constexpr (SPLIT == 2) {
                    // this half's maximum joins the block's; the half that reports last publishes
                    const long rblk = blk >> 1;
                    const int h = (int)(blk & 1);
                    const unsigned long long mine =
                        key ? ((unsigned long long)key << 32) | (0xffffffffu - (unsigned)(2 * bin + h)) : 0ull;
                    if (mine) atomicMax(&a.best[rblk], mine);
                    __threadfence();
                    publish = atomicAdd(&a.cnt[rblk], 1u) == 1u;
                    if (publish) {
                        __threadfence();
                        const unsigned long long both = atomicExch(&a.best[rblk], 0ull);   // (left zero for the next launch)
                        a.cnt[rblk] = 0u;
                        key = (unsigned)(both >> 32);
                        bin = key ? (int)(0xffffffffu - (unsigned)both) : -1;
                        blk = rblk;
                    }
                }
                if (publish) {
                    float *psd = a.out + blk * (long)(NR + 2);
                    float m = -3.4028234663852886e38f;
                    if (key != 0u) {
                        unsigned u = (key & 0x80000000u) ? (key & 0x7fffffffu) : ~key;
                        m = __uint_as_float(u);
                    }
                    // fft.java:214-221 with p = 2*bin, dat.length = 2N, int32 wrap, trunc division
                    int p = (bin < 0) ? -1 : 2 * bin;
                    const int datlen = 2 * NR;
                    if (p >= datlen / 2) p -= datlen;
                    p = (int)((unsigned)p * (unsigned)a.rate) / datlen;
                    psd[NR] = (float)p;
                    psd[NR + 1] = m;
                    if (a.peak_bin) a.peak_bin[blk] = bin;
                }
            }
        }
    }
    if constexpr (!PERSIST) break;
    __syncthreads();                             // shared memory and s_max/s_idx are reused by the next block
    blk0 += blk_step;
    } while (blk0 < a.nblocks);
}

}  // namespace fft
}  // namespace jsdr
