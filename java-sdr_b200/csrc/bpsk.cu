// bpsk.cu — FUNcubeBPSKDemod.java:366-595 for a bank of independent tuners.
//
// Every arithmetic step is binary64 with explicit round-to-nearest intrinsics
// (__dadd_rn / __dmul_rn never contract into FMA), in the reference's operation
// order, so results are bit-identical to the Java arithmetic:
//   RxMixTuner   :382-397   RxDownSample :467-492   RxDemodulate :505-595
//
// How the sequential reference becomes block-parallel:
//   * tuPhase, vcoPhase and dmBitPhase are data-independent accumulators
//     (:384-386, :511-513, :581-583).  A "scout" replays the adds exactly on a
//     side stream and leaves a phase checkpoint every kChunk input samples (per
//     channel) and the table index / roll-over flag per 9600 S/s sample (shared by
//     all channels).  The data kernels then start anywhere.
//   * the tuner + decimator and the matched filter are FIRs over staged,
//     already-mixed samples: one CTA per (channel, tile), shared memory padded so
//     the decimating reads do not bank-conflict.
//   * only the bit-timing tracker (:533-595) is data-dependent; it runs one
//     thread per channel over the 9600 S/s stream.
#include <math.h>

#include <algorithm>
#include <cmath>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "fft_generic.cuh"
#include "handles.h"

namespace jsdr {
namespace bpsk {

constexpr double kTwoPi = 2.0 * 3.141592653589793;       // Java 2.0*Math.PI
constexpr double kInvTwoPi = 1.0 / kTwoPi;
constexpr int kTileOut = 128;                            // decimator outputs per CTA
constexpr int kTileThreads = 128;                        // one thread per output in the FIR phase
constexpr int kPrefetch = 21;                            // raw samples held per thread (covers D <= 20, 128 taps)
// 256/(2*pi) for the double constant 2.0*Math.PI, split hi + lo (host long double)
constexpr double kIdxScaleHi = 40.74366543152521;
constexpr double kIdxScaleLo = -9.306125250357089e-16;
constexpr int kDmTile = 128;                             // matched-filter outputs per CTA

// FUNcubeBPSKDemod.java:27-55 — F-suffixed literals inside a double[]: each is
// rounded to float first, then widened.
static const float kDsFilterF[27] = {
    -6.103515625000e-004F, -1.220703125000e-004F, +2.380371093750e-003F, +6.164550781250e-003F,
    +7.324218750000e-003F, +7.629394531250e-004F, -1.464843750000e-002F, -3.112792968750e-002F,
    -3.225708007813e-002F, -1.617431640625e-003F, +6.463623046875e-002F, +1.502380371094e-001F,
    +2.231445312500e-001F, +2.518310546875e-001F, +2.231445312500e-001F, +1.502380371094e-001F,
    +6.463623046875e-002F, -1.617431640625e-003F, -3.225708007813e-002F, -3.112792968750e-002F,
    -1.464843750000e-002F, +7.629394531250e-004F, +7.324218750000e-003F, +6.164550781250e-003F,
    +2.380371093750e-003F, -1.220703125000e-004F, -6.103515625000e-004F};
// :58-67 — the reference stores this table twice back to back; one copy here,
// indexed modulo 65.
static const float kDmFilterF[65] = {
    -0.0101130691F, -0.0086975143F, -0.0038246093F, +0.0033563764F, +0.0107237026F, +0.0157790936F,
    +0.0164594107F, +0.0119213911F, +0.0030315224F, -0.0076488191F, -0.0164594107F, -0.0197184277F,
    -0.0150109226F, -0.0023082460F, +0.0154712381F, +0.0327423589F, +0.0424493086F, +0.0379940454F,
    +0.0154712381F, -0.0243701991F, -0.0750320094F, -0.1244834076F, -0.1568500423F, -0.1553748911F,
    -0.1061032953F, -0.0015013786F, +0.1568500423F, +0.3572048240F, +0.5786381191F, +0.7940228249F,
    +0.9744923010F, +1.0945250059F, +1.1366117829F, +1.0945250059F, +0.9744923010F, +0.7940228249F,
    +0.5786381191F, +0.3572048240F, +0.1568500423F, -0.0015013786F, -0.1061032953F, -0.1553748911F,
    -0.1568500423F, -0.1244834076F, -0.0750320094F, -0.0243701991F, +0.0154712381F, +0.0379940454F,
    +0.0424493086F, +0.0327423589F, +0.0154712381F, -0.0023082460F, -0.0150109226F, -0.0197184277F,
    -0.0164594107F, -0.0076488191F, +0.0030315224F, +0.0119213911F, +0.0164594107F, +0.0157790936F,
    +0.0107237026F, +0.0033563764F, -0.0038246093F, -0.0086975143F, -0.0101130691F};

// ------------------------------------------------------------------ device helpers
__device__ __forceinline__ double phase_step(double p, double inc)
{   // :384-386 / :511-513  p += inc; if (p > 2pi) p -= 2pi
    const double a = __dadd_rn(p, inc);
    const double w = __dadd_rn(a, -kTwoPi);      // speculative, off the compare's path
    return (a > kTwoPi) ? w : a;
}

// (int)(p*256.0/(2.0*Math.PI)) % 256 for p > 0 (:389).  The division is replaced
// by a multiply unless the quotient is within reach of an integer, where the
// IEEE division the reference performs decides.
__device__ __forceinline__ int table_index(double p)
{
    const double t = __dmul_rn(p, 256.0);
    // A phase beyond 4pi only happens for a tuning above the sample rate (inc > 2pi: the single
    // subtraction of :385 no longer keeps up and tuPhase grows without bound).  The reference then
    // takes Java's saturating (int) of the quotient, % 256 of a non-negative int: do exactly that.
    if (!(p < 16.0)) return __double2int_rz(__ddiv_rn(t, kTwoPi)) & 255;
    // a*2^20 + 1.5*2^52: the low word of the sum is round(a*2^20) (a < 2^9)
    const double y = __fma_rn(t, kInvTwoPi * 1048576.0, 6755399441055744.0);
    const int yi = __double2loint(y);
    const int frac = yi & 0xfffff;
    int k = yi >> 20;
    if (frac < 64 || frac > 1048576 - 64)       // within 6e-5 of an integer: decide exactly
        k = __double2int_rz(__ddiv_rn(t, kTwoPi));
    return k & 255;
}

template <int FMT>
struct RawT;
template <>
struct RawT<FMT_F32> { typedef float2 type; };
template <>
struct RawT<FMT_S16> { typedef uint32_t type; };

template <int FMT>
__device__ __forceinline__ void raw_to_iq(typename RawT<FMT>::type w, int ic, int qc, double &i, double &q)
{
    if constexpr (FMT == FMT_F32) {
        i = (double)w.x;            // :372-373 (double)buf[n*2]
        q = (double)w.y;
    } else {
        const float2 f = s16_iq_to_float2(w, ic, qc);   // common.cuh
        i = (double)f.x;
        q = (double)f.y;
    }
}

// ------------------------------------------------------------------ scouts
// The tuner phase is data independent but must be replayed add by add to stay bit-exact.
// That serial chain is all this kernel does: it steps every channel's phase through the
// block and leaves a checkpoint (the phase before the first sample) for every 32-sample
// chunk.  It runs on the side stream, one block ahead of the data (see bpsk_receive).
//
// Two reference steps in three dependent additions and NO comparison on the results.  With
// 0 < inc < pi a wrap cannot follow a wrap, so a pair of steps is one of (none, none),
// (wrap, none), (none, wrap), and the additions are the reference's own:
//   t1 = p + inc;  t2 = t1 + (-2pi | inc);  t3 = t2 + (inc | -2pi | 0).
// Which pattern applies is decided from the phase BEFORE the pair by two thresholds that are
// exact, not estimates: rounding is monotone, so {p : fl(p + inc) > 2pi} is an up-set of the
// doubles and has a largest non-member th1; likewise th2 for fl(fl(p + inc) + inc) > 2pi.  The
// host finds both by bisection over the bit patterns with the very same additions
// (scout_thresholds), so `p > th1` IS the reference's `tuPhase > 2pi` of the first step and
// `p > th2` that of the second — the result is the reference's sequence by construction.
// Round 1 predicted from approximate thresholds and re-evaluated both comparisons behind the
// chain (seven more instructions per pair, four of them on the FP64 pipe the chain itself
// needs): a sub-partition could host one such chain per thread and the bank's replay held 32
// SMs.  Without them a pair is 3 DADD + 2 DSETP + 6 SEL, so two warps of chains share a
// sub-partition and the same bank needs half the SMs (scout_threads).
struct ScoutChan {
    double inc, th1, th2, pad;
};

__device__ __forceinline__ double phase_step2(double p, double inc, double th1, double th2)
{
    const bool m1 = p > th1, m2 = p > th2;
    const double s2 = m1 ? -kTwoPi : inc;
    const double s3 = m1 ? inc : (m2 ? -kTwoPi : 0.0);
    const double t1 = __dadd_rn(p, inc);
    const double t2 = __dadd_rn(t1, s2);
    return __dadd_rn(t2, s3);
}

constexpr int kScoutThreads = 512;   // launch bound; the CTA size in use is scout_threads()
// Dynamic shared memory a scout CTA asks for (and never uses): more than half an SM's 227 KB, so
// that two scout CTAs can never share an SM (at 90 KB two did when an SM emptied -- a 1024-channel
// bank ran its replay in 7.4 ms instead of 6.0); what is left still takes three 33.8 KB CTAs of
// the N = 4096 FFT plan beside it.  JSDR_SCOUT_SMEM_KB overrides it (tuning aid).
constexpr int kScoutSmem = 116 * 1024;

static int env_int(const char *name, int lo, int hi, int dflt)
{
    const char *e = getenv(name);
    if (!e) return dflt;
    const int v = atoi(e);
    return (v < lo || v > hi) ? dflt : v;
}

// CTA size of the phase scout = how many SMs it takes (one CTA each; the streaming data kernel
// leaves them free when it runs beside it).  profiles/r02_scout_sweep.txt has the sweep behind
// the defaults.  JSDR_SCOUT_THREADS overrides (tuning aid).  `pump`: the receive is the tuner bank
// of a pump call (pump.cu).
static int scout_threads(const jsdr_bpsk *b, bool pump)
{
    static int forced = -1;
    if (forced < 0) {
        forced = env_int("JSDR_SCOUT_THREADS", 32, kScoutThreads, 0);
        if (forced & 31) forced = 0;
    }
    if (forced) return forced;
    // One warp per SM sub-partition (128 threads) is the fastest replay: 5.2 ms per 2^19-sample
    // block whatever the bank size, on nchan/128 SMs.  That is what a bank on its own wants (tuner
    // + decimator alone is bound by the replay, BASELINE config 4).  In the pump the data kernels
    // take 8 ms per block, so the replay may take 6.4 ms on half the SMs (two warps per
    // sub-partition): the FFT beside it gets 16 SMs back (4.63 -> 4.28 ms, step 8.29 -> 8.23 ms).
    return (pump && b->nchan >= 2048) ? 256 : 128;
}

// Thread t of the grid replays channel t (consecutive lanes hold consecutive channels, so the
// checkpoint stores coalesce).
__global__ void __launch_bounds__(kScoutThreads)
k_tuner_scout(const ScoutChan *__restrict__ par, const double *__restrict__ phase_in,
              double *__restrict__ phase_out, double *__restrict__ ckpt, int nchan, int S)
{
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    const int nfull = S >> 5;
    const bool live = ch < nchan;
    const ScoutChan c = par[live ? ch : 0];
    const double p = phase_in[live ? ch : 0];
    double inc = c.inc, th1 = c.th1, th2 = c.th2;
    // the pair form covers 0 < inc < 3.1 from a phase inside [0, 2pi]; anything else runs a dummy
    // chain in step with the warp and is then replayed step by step below
    const bool fast = live && inc > 0.0 && inc < 3.1 && p >= 0.0 && p <= kTwoPi;
    double q = fast ? p : 0.0;
    if (!fast) {
        inc = 1.0;
        th1 = 5.0;
        th2 = 4.0;
    }
    for (int w = 0; w < nfull; w++) {
        if (fast) ckpt[(size_t)w * nchan + ch] = q;
#pragma unroll
        for (int j = 0; j < 16; j++) q = phase_step2(q, inc, th1, th2);
    }
    if (!live) return;
    double ph;
    if (fast) {
        ph = q;
    } else {                                           // increments the pair form does not cover
        ph = p;
        const double ic = par[ch].inc;
        for (int w = 0; w < nfull; w++) {
            ckpt[(size_t)w * nchan + ch] = ph;
#pragma unroll 4
            for (int j = 0; j < 32; j++) ph = phase_step(ph, ic);
        }
    }
    if (S & 31) {
        const double ic = par[ch].inc;
        ckpt[(size_t)nfull * nchan + ch] = ph;
        for (int j = 0; j < (S & 31); j++) ph = phase_step(ph, ic);
    }
    phase_out[ch] = ph;
}

// vcoPhase (:511-516) and dmBitPhase (:581-584) are the same for every channel of
// a bank: warp 0 replays one, warp 1 the other.
__global__ void k_vco_scout(const double *__restrict__ state, double *__restrict__ state_out,
                            uint8_t *__restrict__ vco_ix, uint8_t *__restrict__ bit_roll, int NO, double vco_inc,
                            double bit_inc, double bit_time)
{
    if (threadIdx.x == 0) {
        double p = state[0];
        for (int m = 0; m < NO; m++) {
            p = phase_step(p, vco_inc);
            double q = __ddiv_rn(__dmul_rn(p, 256.0), kTwoPi);
            vco_ix[m] = (uint8_t)(__double2int_rz(q) & 255);
        }
        state_out[0] = p;
    } else if (threadIdx.x == 32) {
        double b = state[1];
        for (int m = 0; m < NO; m++) {
            b = __dadd_rn(b, bit_inc);
            uint8_t roll = 0;
            if (b >= bit_time) {
                b = __dadd_rn(b, -bit_time);
                roll = 1;
            }
            bit_roll[m] = roll;
        }
        state_out[1] = b;
    }
}

// ------------------------------------------------------------------ tuner + decimator
struct MixParams {
    const void *in;
    long long chan_stride;     // complex samples between channels (0: shared stream)
    int S;                     // samples in this block
    int ic, qc;
    const double *tu_inc;      // [nchan]
    const unsigned long long *tu_dx;   // [nchan] index step in 2^-48 units (0: use the exact path)
    const double *ckpt;        // [chunks][nchan] tuner phase before each 32-sample chunk
    int nchan;
    const double2 *hist_in;    // [nchan][kMaxDsTaps], entry k is local sample k-H
    double2 *hist_out;
    int ntaps;
    const double2 *cossin;     // [257] (cos, sin) pairs; entry 256 = (1, 1) for the bypass case
    int D, n0, NO;             // first output's local sample index, outputs this block
    unsigned magicD;           // 2^32/D + 1: i/D == __umulhi(i, magicD) for i, D < 65536
    int pad;                   // 1: one pad slot per D samples (even D), 0: none
    int ix_off;                // byte offset of the index array in dynamic shared memory
    double2 *ds_out;
    int max_ds;
    // in the parameter (constant) bank, read with uniform loads:
    double taps[kMaxDsTaps];
    int off[kMaxDsTaps];       // byte offset of tap k's sample from the thread's base slot
};

// table index of one tuner step, 256 = bypass (phase <= 0: RxDownSample(i, q), :395)
__device__ __forceinline__ int tuner_index(double ph) { return (ph > 0.0) ? table_index(ph) : 256; }

// One CTA = one channel x kTileOut outputs, four phases:
//   1  chunk threads replay the 32 phase steps of their chunk from the scout's
//      checkpoint and leave only the table index of each sample (:384-390);
//   2  every sample of the window is converted and mixed once, sample parallel with
//      coalesced loads (:389-390), into shared memory with one pad slot per D samples
//      so that lanes D apart fall in different banks;
//   3  the decimating FIR (:477-486), newest sample first, one thread per output,
//      one 16-byte load per tap.  With NTAPS/DD fixed at compile time the tap
//      offsets are immediates and the taps come straight from the constant bank.
template <int FMT, int NTAPS, int DD>
__global__ void __launch_bounds__(kTileThreads, 4) k_mixdecim(const MixParams p)
{
    typedef typename RawT<FMT>::type raw_t;
    extern __shared__ __align__(16) unsigned char smem[];
    double2 *sM = reinterpret_cast<double2 *>(smem);
    uint16_t *sIx = reinterpret_cast<uint16_t *>(smem + p.ix_off);   // window index i lives at i+32 (+ one pad per 32)
    __shared__ double2 sTab[257];

    const int tid = threadIdx.x;
    const int ch = blockIdx.y;
    const int m0 = blockIdx.x * kTileOut;
    const int cnt = min(kTileOut, p.NO - m0);
    const int D = DD ? DD : p.D;
    const int ntaps = NTAPS ? NTAPS : p.ntaps;
    const int H = ntaps - 1;
    const int pad = DD ? ((DD & 1) ? 0 : 1) : p.pad;
    const int n_lo = p.n0 + m0 * D - H;               // oldest sample needed (negative: history)
    const int span = (cnt - 1) * D + ntaps;           // window length
    const int i0 = max(-n_lo, 0);                     // first window index that is in this block

    for (int i = tid; i < 257; i += kTileThreads) sTab[i] = p.cossin[i];
    if (n_lo < 0) {                                   // window reaches into the previous block
        const double2 *hist = p.hist_in + (size_t)ch * kMaxDsTaps;
        for (int i = tid; i < i0; i += kTileThreads) {
            const int q = pad ? (int)__umulhi((unsigned)i, p.magicD) : 0;
            sM[i + q] = hist[n_lo + i + H];
        }
    }
    // raw samples of this thread's phase-2 work, fetched now so the loads are in
    // flight while phase 1 computes
    const raw_t *src = reinterpret_cast<const raw_t *>(p.in) + (long long)ch * p.chan_stride + n_lo;
    raw_t pre[kPrefetch];
#pragma unroll
    for (int r = 0; r < kPrefetch; r++) {
        const int i = i0 + tid + r * kTileThreads;
        if (i < span) pre[r] = src[i];
    }

    {   // phase 1: table indices, one thread per 32-sample chunk
        const double inc = p.tu_inc[ch];
        const unsigned long long dx = p.tu_dx[ch];
        const int c_lo = (n_lo + i0) >> 5, c_hi = (n_lo + span - 1) >> 5;
        for (int c = c_lo + tid; c <= c_hi; c += kTileThreads) {
            const double ph0 = p.ckpt[(size_t)c * p.nchan + ch];
            const int ibase = (c << 5) - n_lo;        // window index of the chunk's first sample
            const int steps = min(32, p.S - (c << 5));
            // (edge chunks hang over the window; the index array has a 32-entry margin at
            // both ends so they take the same unguarded path)
            bool exact = !(dx != 0ull && ph0 >= 0.0);
            if (!exact) {
                // Fast path.  x = phase*256/2pi as 8.48 fixed point, anchored at the exact
                // checkpoint and advanced by integer adds.  Over 32 steps the reference's
                // accumulated rounding moves the true value by < 2^-39, so the integer part
                // is the reference's index unless x is within 2^-16 of an integer; then the
                // chunk is redone with the reference's own arithmetic.
                const double hi = __dmul_rn(ph0, kIdxScaleHi);
                const double lo = __fma_rn(ph0, kIdxScaleLo, __fma_rn(ph0, kIdxScaleHi, -hi));
                unsigned long long x = (unsigned long long)(__double2ll_rn(hi * 281474976710656.0) +
                                                            __double2ll_rn(lo * 281474976710656.0));
                unsigned near = 0;
                const int ib = ibase + 32;
                uint16_t *dst = sIx + ib + (ib >> 5);
#pragma unroll
                for (int j = 0; j < 32; j++) {
                    x += dx;
                    const unsigned xh = (unsigned)(x >> 32);
                    near |= ((xh + 1u) & 0xffffu) <= 1u;
                    dst[j + ((((ib & 31) + j) >> 5))] = (uint16_t)((xh >> 16) & 255u);
                }
                exact = near != 0u;
            }
            if (exact) {                              // reference arithmetic, step by step
                double ph = ph0;
                for (int j = 0; j < steps; j++) {
                    ph = phase_step(ph, inc);
                    const int i = ibase + j;
                    if (i >= i0 && i < span) sIx[i + 32 + ((i + 32) >> 5)] = (uint16_t)tuner_index(ph);
                }
            }
        }
    }
    __syncthreads();

    {   // phase 2: convert + mix, sample parallel
#pragma unroll
        for (int r = 0; r < kPrefetch; r++) {
            const int i = i0 + tid + r * kTileThreads;
            if (i < span) {
                double xi, xq;
                raw_to_iq<FMT>(pre[r], p.ic, p.qc, xi, xq);
                const double2 cs = sTab[sIx[i + 32 + ((i + 32) >> 5)]];
                const int q = pad ? (int)__umulhi((unsigned)i, p.magicD) : 0;
                sM[i + q] = make_double2(__dmul_rn(xi, cs.x), __dmul_rn(xq, cs.y));   // i*cosTab[ix], q*sinTab[ix]
            }
        }
        for (int i = i0 + tid + kPrefetch * kTileThreads; i < span; i += kTileThreads) {   // very wide windows only
            double xi, xq;
            raw_to_iq<FMT>(src[i], p.ic, p.qc, xi, xq);
            const double2 cs = sTab[sIx[i + 32 + ((i + 32) >> 5)]];
            const int q = pad ? (int)__umulhi((unsigned)i, p.magicD) : 0;
            sM[i + q] = make_double2(__dmul_rn(xi, cs.x), __dmul_rn(xq, cs.y));
        }
    }
    __syncthreads();

    if (tid < cnt) {   // phase 3
        // window index of tap k is tid*D + H - k -> slot tid*(D+pad) + (H-k) + pad*((H-k)/D)
        const unsigned char *base = smem + (size_t)tid * (D + pad) * sizeof(double2);
        double ai = 0.0, aq = 0.0;
        if constexpr (NTAPS > 0 && DD > 0) {
#pragma unroll
            for (int k = 0; k < NTAPS; k++) {
                constexpr int PADC = (DD & 1) ? 0 : 1;
                const int d = NTAPS - 1 - k;
                const double2 x = *reinterpret_cast<const double2 *>(base + sizeof(double2) * (d + PADC * (d / DD)));
                const double h = p.taps[k];
                ai = __dadd_rn(ai, __dmul_rn(x.x, h));
                aq = __dadd_rn(aq, __dmul_rn(x.y, h));
            }
        } else {
#pragma unroll 4
            for (int k = 0; k < ntaps; k++) {
                const double2 x = *reinterpret_cast<const double2 *>(base + p.off[k]);
                const double h = p.taps[k];
                ai = __dadd_rn(ai, __dmul_rn(x.x, h));
                aq = __dadd_rn(aq, __dmul_rn(x.y, h));
            }
        }
        // :469,486  fi * HOWARD_FUDGE_FACTOR, 0.9*32768.0 folded by javac to one double
        p.ds_out[(size_t)ch * p.max_ds + m0 + tid] =
            make_double2(__dmul_rn(ai, 0.9 * 32768.0), __dmul_rn(aq, 0.9 * 32768.0));
    }
}

// New history = the last H mixed samples of the block (or old history shifted,
// for blocks shorter than H).  One CTA per channel.
template <int FMT>
__global__ void k_tuner_tail(const MixParams p)
{
    typedef typename RawT<FMT>::type raw_t;
    const int ch = blockIdx.x;
    const int H = p.ntaps - 1;
    const int k = threadIdx.x;
    if (k >= H) return;
    const int n = p.S - H + k;
    double2 v;
    if (n < 0) {
        v = p.hist_in[(size_t)ch * kMaxDsTaps + k + p.S];
    } else {
        const raw_t *src = reinterpret_cast<const raw_t *>(p.in) + (long long)ch * p.chan_stride;
        double ph = p.ckpt[(size_t)(n >> 5) * p.nchan + ch];
        const double inc = p.tu_inc[ch];
        for (int j = n & ~31; j <= n; j++) ph = phase_step(ph, inc);
        const double2 cs = p.cossin[tuner_index(ph)];
        double xi, xq;
        raw_to_iq<FMT>(src[n], p.ic, p.qc, xi, xq);
        v = make_double2(__dmul_rn(xi, cs.x), __dmul_rn(xq, cs.y));
    }
    p.hist_out[(size_t)ch * kMaxDsTaps + k] = v;
}

}  // namespace bpsk
}  // namespace jsdr
#include "bpsk_stream.cuh"
namespace jsdr {
namespace bpsk {


// ------------------------------------------------------------------ auto-tune (doBufferFFT, :406-464)
// :417-420 (double)buf[..] into the forward transform's input
template <int FMT>
__global__ void __launch_bounds__(256) k_at_load(const void *__restrict__ in, long long chan_stride, int S, int nchan,
                                                 int ic, int qc, double2 *__restrict__ out)
{
    typedef typename RawT<FMT>::type raw_t;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)nchan * S) return;
    const int ch = (int)(i / S), n = (int)(i - (long long)ch * S);
    double xi, xq;
    raw_to_iq<FMT>(reinterpret_cast<const raw_t *>(in)[(long long)ch * chan_stride + n], ic, qc, xi, xq);
    out[i] = make_double2(xi, xq);
}

// :425-458 for one channel per CTA: magnitude, 100-bin boxcar sums in the reference's summation
// order, first strict maximum, the smoothing / gate / clamp of the centre bin, and the copy of
// 204 bins to DC of the (pre-zeroed) inverse transform's input.
__global__ void __launch_bounds__(256) k_at_search(const double2 *__restrict__ fwd, double2 *__restrict__ rev, int N,
                                                   int doUp, AutoTuneState *__restrict__ state)
{
    extern __shared__ double s_psd[];                  // psd[lo .. hi)
    __shared__ unsigned long long s_max;
    __shared__ int s_idx;
    __shared__ int s_centre;
    const int ch = blockIdx.x, tid = threadIdx.x;
    const double2 *x = fwd + (size_t)ch * N;
    const int beg = doUp ? N / 4 : 0, end = doUp ? N / 2 : N / 4;
    const int lo = max(beg + 75 - 50, 0), hi = max(min(end - 75 + 50, N / 2), lo);   // psd[] range the sums touch
    for (int i = lo + tid; i < hi; i += blockDim.x) {
        const double2 v = x[i];
        s_psd[i - lo] = __dsqrt_rn(__dadd_rn(__dmul_rn(v.x, v.x), __dmul_rn(v.y, v.y)));   // :426
    }
    if (tid == 0) {
        s_max = 0ull;
        s_idx = 0x7fffffff;
    }
    __syncthreads();
    auto boxcar = [&](int i) {                         // :436-439, j ascending from a zero start
        double a = 0.0;
        for (int j = i - 50; j < i + 50; j++) a = __dadd_rn(a, s_psd[j - lo]);
        return a;
    };
    double best = 0.0;                                 // :429 maxBin starts at 0.0; strict '<' (:440)
    int best_i = 0x7fffffff;
    for (int i = beg + 75 + tid; i < end - 75; i += blockDim.x) {
        const double a = boxcar(i);
        if (best < a) {
            best = a;
            best_i = i;
        }
    }
    // sums are non-negative: their bit patterns order like the values
    if (best_i != 0x7fffffff) atomicMax(&s_max, (unsigned long long)__double_as_longlong(best));
    __syncthreads();
    if (best_i != 0x7fffffff && (unsigned long long)__double_as_longlong(best) == s_max) atomicMin(&s_idx, best_i);
    __syncthreads();
    if (tid == 0) {
        AutoTuneState st = state[ch];
        const double maxBin = (s_idx != 0x7fffffff) ? __longlong_as_double((long long)s_max) : 0.0;
        const int binPos = (s_idx != 0x7fffffff) ? s_idx : -1;
        if (st.centreBin < 0) st.centreBin = 0;                                        // :444-445
        if (st.centreBin > end - 1) st.centreBin = end - 1;
        // avePsd[] is zero outside the scanned range (SURVEY Q9)
        const double aveC = (st.centreBin >= beg + 75 && st.centreBin < end - 75) ? boxcar(st.centreBin) : 0.0;
        const double PSD_AVE = (double)(2.0f / (10 + 1)), PSD_INV = (double)(1.0f - (2.0f / (10 + 1)));   // :401-402
        const double CF_AVE = (double)(2.0f / (1 + 1)), CF_INV = (double)(1.0f - (2.0f / (1 + 1)));       // :399-400
        st.avePeakPower = __dadd_rn(__dmul_rn(PSD_AVE, aveC), __dmul_rn(PSD_INV, st.avePeakPower));       // :446
        if (maxBin > __dmul_rn(__ddiv_rn(st.avePeakPower, 4.0), 5.0) && binPos > 0) {                     // :447
            st.aveCentreBin = __dadd_rn(__dmul_rn(CF_AVE, (double)(float)binPos), __dmul_rn(CF_INV, st.aveCentreBin));
            const double c = __dadd_rn(st.aveCentreBin, 1.0);
            st.centreBin = (c != c) ? 0 : (c >= 2147483647.0 ? 2147483647 : (c <= -2147483648.0 ? (int)0x80000000 : (int)c));
        }
        if (st.centreBin < 102) st.centreBin = 102;                                    // :453
        state[ch] = st;
        s_centre = st.centreBin;
    }
    __syncthreads();
    const int c0 = s_centre - 102;                                                     // :458
    if (tid < 204) {
        const int k = c0 + tid;
        rev[(size_t)ch * N + tid] = (k >= 0 && k < N) ? x[k] : make_double2(0.0, 0.0);
    }
}

// :461-463 RxDownSample(re, re) on the inverse transform's real part (scaled by 1/N as
// complexInverse(.., true) does), decimator FIR in the reference order; one thread per output.
__global__ void __launch_bounds__(128) k_at_decim(const double2 *__restrict__ inv, int N, double inv_scale,
                                                  const double2 *__restrict__ hist_in, double2 *__restrict__ hist_out,
                                                  const double *__restrict__ taps, int ntaps, int D, int n0, int NO,
                                                  double2 *__restrict__ ds_out, int max_ds)
{
    const int ch = blockIdx.y;
    const int H = ntaps - 1;
    const double2 *x = inv + (size_t)ch * N;
    auto sample = [&](int n) {                         // local sample n (negative: previous block)
        if (n < 0) {
            const int k = n + H;
            return (k >= 0) ? hist_in[(size_t)ch * kMaxDsTaps + k].x : 0.0;
        }
        return __dmul_rn(x[n].x, inv_scale);
    };
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m < NO) {
        const int n = n0 + m * D;
        double a = 0.0;
        for (int k = 0; k < ntaps; k++) a = __dadd_rn(a, __dmul_rn(sample(n - k), taps[k]));   // :479-483
        const double o = __dmul_rn(a, 0.9 * 32768.0);                                          // :486
        ds_out[(size_t)ch * max_ds + m] = make_double2(o, o);
    }
    if (blockIdx.x == 0 && threadIdx.x < H) {          // new history: the last H inputs
        const int n = N - H + threadIdx.x;
        const double v = sample(n);
        hist_out[(size_t)ch * kMaxDsTaps + threadIdx.x] = make_double2(v, v);
    }
}

// ------------------------------------------------------------------ matched filter
struct DmParams {
    const double2 *ds;         // [nchan][max_ds]
    int max_ds, NO;
    const uint8_t *vco_ix;
    const double2 *hist_in;    // [nchan][64], entry k is local sample k-64
    double2 *hist_out;
    const double *dmtaps;
    const double *cossin;
    int base65;                // cntDS before this block, mod 65
    double2 *dm_out;
};

__device__ __forceinline__ double2 vco_mix(const DmParams &p, const double *sTab, int ch, int m)
{   // :515-516
    double2 d = p.ds[(size_t)ch * p.max_ds + m];
    int ix = p.vco_ix[m];
    return make_double2(__dmul_rn(d.x, sTab[ix]), __dmul_rn(d.y, sTab[256 + ix]));
}

// One CTA = one channel x 2080 outputs, five warps.  Lane t of warp w computes the 13 outputs
// 65t + 13w .. 65t + 13w + 12 of the tile.  The reference sums by buffer slot
// (:519-523): output m visits ages a0, a0+1, .., 64, 0, .., a0-1 with a0 = (m + 1 + calls before
// this block) mod 65, tap = dmFilter[age], sample = v[m - age].  For 13 consecutive outputs the
// age at step n is c + r (c = a0 + n mod 65, r = 0..12): the same sample v[m0 - c] serves every
// output that has not wrapped yet (tap dmFilter[c + r]) and v[m0 - c + 65] those that have.  So
// a step is two 16-byte loads for 52 multiply-adds, and because the threads of a warp are 65
// outputs apart, a0 — and with it the set of steps where some outputs have wrapped — is the same
// for all of them: no divergence, and the taps are warp-uniform (shared-memory broadcast).
// Every output still accumulates in the reference's order, so the result is bit-identical.
constexpr int kDm2R = 13;                                 // outputs per thread
constexpr int kDm2Warps = 65 / kDm2R;                     // warp w computes outputs 13w .. 13w+12 of every 65
constexpr int kDm2Threads = 32 * kDm2Warps;
constexpr int kDm2Tile = 32 * 65;                         // 2080 outputs per CTA

__global__ void __launch_bounds__(kDm2Threads) k_matched(const DmParams p)
{
    extern __shared__ __align__(16) unsigned char dm_smem[];
    double2 *sV = reinterpret_cast<double2 *>(dm_smem);              // VCO-mixed samples, tile index i <-> m = m0 - 64 + i
    __shared__ double sTab[512];
    __shared__ double sT2[2 * kDmTaps];                              // dmFilter twice back to back (:58-67)
    const int tid = threadIdx.x, ch = blockIdx.y;
    const int m0 = blockIdx.x * kDm2Tile;
    const int cnt = min(kDm2Tile, p.NO - m0);
    for (int i = tid; i < 512; i += kDm2Threads) sTab[i] = p.cossin[i];
    for (int i = tid; i < 2 * kDmTaps; i += kDm2Threads) sT2[i] = p.dmtaps[i % kDmTaps];
    __syncthreads();
    // staging: 8 loads in flight per thread (one warp per CTA: the latency has to be covered here)
    for (int i0 = 0; i0 < kDm2Tile + 64; i0 += 8 * kDm2Threads) {
        double2 d[8];
        int ix[8];
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const int ii = i0 + u * kDm2Threads + tid, m = m0 - 64 + ii;
            d[u] = make_double2(0.0, 0.0);
            ix[u] = -1;
            if (ii < kDm2Tile + 64) {
                if (m < 0) d[u] = p.hist_in[(size_t)ch * 64 + 64 + m];
                else if (m < p.NO) {
                    d[u] = p.ds[(size_t)ch * p.max_ds + m];
                    ix[u] = p.vco_ix[m];
                }
            }
        }
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const int ii = i0 + u * kDm2Threads + tid;
            if (ii < kDm2Tile + 64) {
                double2 v = d[u];
                if (ix[u] >= 0) v = make_double2(__dmul_rn(v.x, sTab[ix[u]]), __dmul_rn(v.y, sTab[256 + ix[u]]));   // :515-516
                sV[ii] = v;
            }
        }
    }
    __syncthreads();
    {
        const int lo = 65 * (tid & 31) + kDm2R * (tid >> 5);         // first of this thread's 13 outputs (tile local)
        if (lo >= cnt) return;
        const int a0 = (p.base65 + m0 + lo + 1) % 65;                // uniform across the warp (lanes are 65 outputs apart)
        double ai[kDm2R], aq[kDm2R];
#pragma unroll
        for (int r = 0; r < kDm2R; r++) ai[r] = aq[r] = 0.0;
        const double2 *vb = sV + lo + 64;                            // v[m] of output lo
#pragma unroll 1
        for (int n = 0; n < kDmTaps; n++) {
            int c = a0 + n;
            if (c >= 65) c -= 65;
            const double2 xa = vb[-c];
            const double *h = sT2 + c;
            if (c + kDm2R - 1 < 65) {                                // nobody has wrapped: one sample for all
#pragma unroll
                for (int r = 0; r < kDm2R; r++) {
                    ai[r] = __dadd_rn(ai[r], __dmul_rn(xa.x, h[r]));
                    aq[r] = __dadd_rn(aq[r], __dmul_rn(xa.y, h[r]));
                }
            } else {
                const double2 xb = vb[65 - c];                       // (needs c >= 53: index <= lo + 76, staged)
#pragma unroll
                for (int r = 0; r < kDm2R; r++) {
                    const bool w = c + r >= 65;
                    const double xi = w ? xb.x : xa.x, xq = w ? xb.y : xa.y;
                    ai[r] = __dadd_rn(ai[r], __dmul_rn(xi, h[r]));
                    aq[r] = __dadd_rn(aq[r], __dmul_rn(xq, h[r]));
                }
            }
        }
        double2 *o = p.dm_out + (size_t)ch * p.max_ds + m0 + lo;
#pragma unroll
        for (int r = 0; r < kDm2R; r++)
            if (lo + r < cnt) o[r] = make_double2(ai[r], aq[r]);
    }
}

__global__ void k_dm_tail(const DmParams p)
{
    __shared__ double sTab[512];
    const int ch = blockIdx.x, k = threadIdx.x;
    for (int i = threadIdx.x; i < 512; i += blockDim.x) sTab[i] = p.cossin[i];
    __syncthreads();
    if (k >= 64) return;
    int m = p.NO - 64 + k;
    double2 v = (m < 0) ? p.hist_in[(size_t)ch * 64 + k + p.NO] : vco_mix(p, sTab, ch, m);
    p.hist_out[(size_t)ch * 64 + k] = v;
}

// ------------------------------------------------------------------ bit timing + decision
struct TimingParams {
    const double2 *dm;
    int max_ds, NO, nchan;
    const uint8_t *bit_roll;
    TimingState *ts;
    int8_t *bits;
    long long *bit_at;
    int32_t *nbits;
    int max_bits;
    long long cnt_ds0;
};

constexpr int kTimingTile = 8;       // 9600 S/s samples per channel per step of the outer loop

// :533-595, one lane per channel, one warp per CTA (the recurrence is latency bound, so the
// warps are spread over as many SMs as there are).  No shared memory and few registers, so that
// these CTAs fit beside whatever else is resident (the kernel runs on the auxiliary stream, next to
// the following block's tuner and matched filter): every lane reads its own row of the
// matched-filter output, 16 bytes per sample, a tile of 8 samples ahead in registers.
__global__ void __launch_bounds__(32) k_timing(const TimingParams p)
{
    __shared__ double sE[8][32];                       // dmEnergy[], indexed by the running bit position
    const int lane = threadIdx.x;
    const int ch0 = blockIdx.x * 32;
    const int ch = min(ch0 + lane, p.nchan - 1);
    const bool live = ch0 + lane < p.nchan;
    TimingState st = p.ts[ch];
#pragma unroll
    for (int i = 0; i < 8; i++) sE[i][lane] = st.dmEnergy[i];
    const double S1 = 1.0 / 200.0, S2 = 1.0 / 800.0;
    const double C1 = 1.0 - S1, C2 = 1.0 - S2;
    double eOut = st.dmEnergyOut, lastI = st.lastI, lastQ = st.lastQ;
    int bitPos = st.bitPos, peakPos = st.peakPos, newPeak = st.newPeak;
    int nb = 0;
    int8_t *bits = p.bits + (size_t)ch * p.max_bits;
    long long *bit_at = p.bit_at + (size_t)ch * p.max_bits;
    const double2 *row = p.dm + (size_t)ch * p.max_ds;

    const int ntiles = (p.NO + kTimingTile - 1) / kTimingTile;
    double2 cur[kTimingTile], nxt[kTimingTile];
    auto load_tile = [&](int t, double2 (&dst)[kTimingTile]) {
#pragma unroll
        for (int j = 0; j < kTimingTile; j++) {
            const int m = t * kTimingTile + j;
            dst[j] = (m < p.NO) ? row[m] : make_double2(0.0, 0.0);
        }
    };
    if (ntiles > 0) load_tile(0, nxt);
    for (int t = 0; t < ntiles; t++) {
#pragma unroll
        for (int j = 0; j < kTimingTile; j++) cur[j] = nxt[j];
        if (t + 1 < ntiles) load_tile(t + 1, nxt);
        const int cnt = min(kTimingTile, p.NO - t * kTimingTile);
        // bit-phase roll-overs of this tile (the same for every channel): one bit per sample
        unsigned rollmask = 0;
#pragma unroll
        for (int j = 0; j < kTimingTile; j++) {
            const int m = t * kTimingTile + j;
            if (m < p.NO && p.bit_roll[m] != 0) rollmask |= 1u << j;
        }
        // Decisions of different channels fall on different samples (bitPos == peakPos), and two
        // decisions of one channel are at least 5 samples apart.  The per-sample part therefore
        // only notes the decision sample; the expensive part (:538-574) runs for all lanes
        // together once every 4 samples instead of diverging on every sample.
#pragma unroll
        for (int j0 = 0; j0 < cnt; j0 += 4) {
            bool pend = false;
            double2 pf = make_double2(0.0, 0.0);
            double pe1 = 0.0;
            int pm = 0;
#pragma unroll
            for (int jj = 0; jj < 4; jj++) {
                const int j = j0 + jj;
                if (j < cnt) {
                    const double2 f = cur[j];
                    const double energy1 = __dadd_rn(__dmul_rn(f.x, f.x), __dmul_rn(f.y, f.y));            // :534
                    sE[bitPos][lane] = __dadd_rn(__dmul_rn(sE[bitPos][lane], C1), __dmul_rn(energy1, S1));   // :535
                    if (bitPos == peakPos) {                                                               // :537
                        pend = true;
                        pf = f;
                        pe1 = energy1;
                        pm = t * kTimingTile + j;
                    }
                    if (bitPos == ((peakPos + 4) & 7)) peakPos = newPeak;      // :577 dmHalfTable = {4,5,6,7,0,1,2,3}
                    bitPos = (bitPos + 1) & 7;                                 // :579
                    if ((rollmask >> j) & 1u) {                                // :582-592 (same for every channel)
                        bitPos = 0;
                        double eMax = -1.0e10;                                 // (double)-1.0e10F, exact
#pragma unroll
                        for (int n = 0; n < 8; n++) {
                            double e = sE[n][lane];
                            if (e > eMax) { newPeak = n; eMax = e; }
                        }
                    }
                }
            }
            if (pend) {
                eOut = __dadd_rn(__dmul_rn(eOut, C2), __dmul_rn(pe1, S2));                 // :538
                double di = -__dadd_rn(__dmul_rn(lastI, pf.x), __dmul_rn(lastQ, pf.y));    // :539
                double dq = __dadd_rn(__dmul_rn(lastI, pf.y), -__dmul_rn(lastQ, pf.x));    // :540
                lastI = pf.x;
                lastQ = pf.y;
                double energy2 = __dsqrt_rn(__dadd_rn(__dmul_rn(di, di), __dmul_rn(dq, dq)));
                if (energy2 > 100.0) {                                                     // :544
                    if (nb < p.max_bits && live) {
                        bits[nb] = (di < 0.0) ? 1 : -1;                                    // :545,554
                        bit_at[nb] = p.cnt_ds0 + pm;
                    }
                    nb++;
                }
            }
        }
    }
    if (!live) return;
#pragma unroll
    for (int i = 0; i < 8; i++) st.dmEnergy[i] = sE[i][lane];
    st.dmEnergyOut = eOut;
    st.lastI = lastI;
    st.lastQ = lastQ;
    st.bitPos = bitPos;
    st.peakPos = peakPos;
    st.newPeak = newPeak;
    st.cntBit += nb;
    p.ts[ch] = st;
    p.nbits[ch] = nb;
}

}  // namespace bpsk
}  // namespace jsdr

// =========================================================================== host
using namespace jsdr;
using namespace jsdr::bpsk;

namespace {

// Per-sample advance of x = phase*256/(2*pi) in 2^-48 units, modulo 256, in extended
// precision (used by k_mixdecim's integer fast path).  0 selects the exact path:
// non-positive or non-finite increments (mixer bypass, :388).
unsigned long long index_step_fixed(double inc)
{
    if (!(inc > 0.0) || !(inc < 1e6)) return 0ull;
    const long double c = 256.0L / (long double)(2.0 * M_PI);
    long double d = fmodl((long double)inc * c, 256.0L);
    unsigned long long v = (unsigned long long)(d * 281474976710656.0L + 0.5L);
    return v ? v : 1ull;
}

// The same step in 8.56 fixed point for the streaming kernel.  0 selects exact replay:
// increments that are not positive and below pi (two wraps in a row, mixer bypass).
unsigned long long index_step_fixed56(double inc)
{
    if (!(inc > 0.0) || !(inc < 3.1)) return 0ull;
    const long double c = 256.0L / (long double)(2.0 * M_PI);
    long double d = fmodl((long double)inc * c, 256.0L);
    unsigned long long v = (unsigned long long)(d * 72057594037927936.0L + 0.5L);
    return v ? v : 1ull;
}

// The exact wrap thresholds of the pair form (see k_tuner_scout): th1 = the largest double p in
// [0, 2pi] for which the reference's first step does NOT wrap (fl(p + inc) > 2pi is false), th2 the
// same for the second step of a pair whose first did not wrap.  Rounding is monotone, so both sets
// are down-sets and bisection over the bit patterns (non-negative doubles order like their
// integers) with the reference's own additions finds them.  -1 = the step wraps from every phase.
static void scout_thresholds(double inc, double &th1, double &th2)
{
    auto from_bits = [](unsigned long long u) { double x; memcpy(&x, &u, 8); return x; };
    auto to_bits = [](double x) { unsigned long long u; memcpy(&u, &x, 8); return u; };
    auto wraps1 = [&](double p) { volatile double t = p + inc; return t > kTwoPi; };
    auto wraps2 = [&](double p) { volatile double t = p + inc; volatile double u = t + inc; return u > kTwoPi; };
    auto last_false = [&](auto f) -> double {
        if (f(0.0)) return -1.0;
        if (!f(kTwoPi)) return kTwoPi;
        unsigned long long lo = 0, hi = to_bits(kTwoPi);          // f(lo) false, f(hi) true
        while (hi - lo > 1) {
            const unsigned long long mid = lo + (hi - lo) / 2;
            if (f(from_bits(mid))) hi = mid;
            else lo = mid;
        }
        return from_bits(lo);
    };
    th1 = last_false(wraps1);
    th2 = last_false(wraps2);
}

static ScoutChan scout_chan(double inc)
{
    ScoutChan c;
    c.inc = inc;
    c.th1 = c.th2 = c.pad = 0.0;
    if (inc > 0.0 && inc < 3.1) scout_thresholds(inc, c.th1, c.th2);
    return c;
}

// Replay the tuner phase over the next S samples from the committed phase into `P`
// (side stream).
int launch_scout(jsdr_bpsk *b, jsdr_bpsk::TunerPlan &P, int S, bool pump)
{
    jsdr_ctx *ctx = b->ctx;
    ProfScope prof(ctx, JSDR_K_SCOUT, ctx->side);
    const int st = scout_threads(b, pump);
    // The replay is a latency-bound chain that wants its share of a sub-partition's FP64 pipe, and
    // CTAs of a high-priority stream are placed wherever a slot frees up: sixteen of these small
    // CTAs fit in the space one retiring data CTA leaves, and stacked like that they run nine
    // times slower.  A shared-memory request the kernel never touches rules the stacking out:
    // one scout CTA per SM (kScoutSmem, see there).
    static int scout_smem = 0;
    if (!scout_smem) scout_smem = env_int("JSDR_SCOUT_SMEM_KB", 1, 200, kScoutSmem / 1024) * 1024;
    static PerDeviceFlag attr_done;
    JSDR_TRY(attr_done.once(ctx->device, [&]() -> int {
        JSDR_CUDA(cudaFuncSetAttribute(k_tuner_scout, cudaFuncAttributeMaxDynamicSharedMemorySize, scout_smem));
        return JSDR_OK;
    }));
    const int grid = (b->nchan + st - 1) / st;
    k_tuner_scout<<<grid, st, scout_smem, ctx->side>>>(b->d_tu_par.get(), b->d_tu_phase, P.phase_end.get(), P.ckpt.get(), b->nchan, S);
    JSDR_TRY(launched(ctx, "k_tuner_scout"));
    JSDR_CUDA(cudaEventRecord(P.ready, ctx->side));
    P.S = S;
    P.valid = true;
    return JSDR_OK;
}

// Replay vcoPhase (:511-516) and dmBitPhase (:581-584) for NO samples from the committed state
// into buffer kb (side stream).  The committed state is not touched: the output state becomes the
// committed one when the block is actually consumed.
int launch_vco_scout(jsdr_bpsk *b, int NO, int kb)
{
    jsdr_ctx *ctx = b->ctx;
    const double vco_inc = 2.0 * M_PI * 1200.0 / (double)9600;      // :88
    const double bit_inc = 1.0 / (double)9600, bit_time = 1.0 / (double)1200;   // :91-92
    // (the bit-timing kernel of two blocks ago may still be reading this buffer)
    // Own stream: a one-CTA serial chain of about a third of the tuner scout's length; behind that
    // scout on the same stream it made the side stream the critical path of the whole chain.
    if (b->bits_used[kb]) JSDR_CUDA(cudaStreamWaitEvent(ctx->side2, b->stage.ev_bits_done[kb], 0));
    // (and the matched filter that last read this buffer, two blocks ago, is done: the event is the
    // newer one of the previous block)
    if (b->stage.ev_dm_ready) JSDR_CUDA(cudaStreamWaitEvent(ctx->side2, b->stage.ev_dm_ready, 0));
    const int c = b->vco_state_cur;
    k_vco_scout<<<1, 64, 0, ctx->side2>>>(b->d_vco_state.get() + 2 * c, b->d_vco_state.get() + 2 * (c ^ 1), b->stage.d_vco_ix[kb].get(),
                                         b->stage.d_bit_roll[kb].get(), NO, vco_inc, bit_inc, bit_time);
    JSDR_TRY(launched(ctx, "k_vco_scout"));
    JSDR_CUDA(cudaEventRecord(b->stage.ev_vco_ready, ctx->side2));
    return JSDR_OK;
}

// Buffers of the 9600 S/s stages, allocated when a receive first needs them (a
// stages==1 bank, e.g. the mix+FIR benchmark, never pays for them).
int ensure_stage_buffers(jsdr_bpsk *b)
{
    if (b->stage.d_bits) return JSDR_OK;
    jsdr_ctx *ctx = b->ctx;
    const char *what = "stage buffers";
    const size_t nc = (size_t)b->nchan;
    jsdr_bpsk::Stages g;
    for (int i = 0; i < 2; i++) JSDR_TRY(g.d_vco_ix[i].alloc_zeroed((size_t)b->max_ds, ctx->stream, what));
    for (int i = 0; i < 2; i++) JSDR_TRY(g.d_bit_roll[i].alloc_zeroed((size_t)b->max_ds, ctx->stream, what));
    for (int i = 0; i < 2; i++) JSDR_TRY(g.d_dm_hist[i].alloc_zeroed(sizeof(double2) * 64 * nc, ctx->stream, what));
    JSDR_TRY(g.d_bits.alloc_zeroed(nc * b->max_bits, ctx->stream, what));
    JSDR_TRY(g.d_bit_at.alloc_zeroed(sizeof(long long) * nc * b->max_bits, ctx->stream, what));
    for (int i = 0; i < 2; i++) JSDR_TRY(g.d_dm_buf[i].alloc_zeroed(sizeof(double2) * nc * b->max_ds, ctx->stream, what));
    JSDR_TRY(g.ev_dm_ready.create(what));
    JSDR_TRY(g.ev_vco_ready.create(what));
    for (int i = 0; i < 2; i++) JSDR_TRY(g.ev_bits_done[i].create(what));
    // the bit stage starts on the auxiliary stream: order it behind the clears above
    JSDR_CUDA(cudaEventRecord(g.ev_dm_ready, ctx->stream));
    JSDR_CUDA(cudaStreamWaitEvent(ctx->aux, g.ev_dm_ready, 0));
    b->stage = std::move(g);
    b->d_dm_out = b->stage.d_dm_buf[0].get();
    return JSDR_OK;
}

int bpsk_reset_ds(jsdr_bpsk *b)
{
    jsdr_ctx *ctx = b->ctx;
    for (int i = 0; i < 2; i++)
        JSDR_CUDA(cudaMemsetAsync(b->d_ds_hist[i].get(), 0, sizeof(double2) * kMaxDsTaps * (size_t)b->nchan, ctx->stream));
    b->ds_cnt = 0;
    b->ds_hist_cur = 0;
    return JSDR_OK;
}

// The streaming tuner + decimator: one lane per channel, one warp per segment of R outputs.
template <int FMT, int PREC, int NTAPS, int DD>
int launch_stream_shape(jsdr_bpsk *b, const stream::Params &sp)
{
    jsdr_ctx *ctx = b->ctx;
    constexpr int W = (FMT == FMT_S16) ? stream::kWarps : stream::kWarpsF32;
    auto kern = stream::k_mixdecim_stream<FMT, PREC, NTAPS, DD, W>;
    constexpr size_t smem = stream::smem_bytes<FMT, W, DD>();
    static PerDeviceFlag attr_done;
    JSDR_TRY(attr_done.once(ctx->device, [&]() -> int {
        JSDR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        return JSDR_OK;
    }));
    const int warps = sp.ncw * sp.nseg;
    const int grid = std::min((warps + W - 1) / W, sp.grid);
    JSDR_CUDA(cudaMemsetAsync(sp.work_counter, 0, sizeof(unsigned), ctx->stream));
    ProfScope prof(ctx, JSDR_K_MIXDECIM, ctx->stream);
    kern<<<grid, W * 32, smem, ctx->stream>>>(sp);
    return launched(ctx, "k_mixdecim_stream");
}

template <int FMT>
int launch_stream(jsdr_bpsk *b, const MixParams &mp, int S, bool pump)
{
    stream::Params sp;
    sp.in = mp.in;
    sp.chan_stride = mp.chan_stride;
    sp.S = S;
    sp.ic = mp.ic;
    sp.qc = mp.qc;
    sp.tu_dx56 = b->d_tu_dx56.get();
    sp.tu_inc = mp.tu_inc;
    sp.ckpt = mp.ckpt;
    sp.nchan = mp.nchan;
    sp.nchunks = (S + 31) / 32;
    sp.hist_in = mp.hist_in;
    sp.cossin = mp.cossin;
    sp.n0 = mp.n0;
    sp.NO = mp.NO;
    sp.ncw = (mp.nchan + 31) / 32;
    // one CTA per SM, warps loop over segments; the SMs the phase scout needs (on the
    // high-priority side stream) are left free so that the two never share an SM.  Segments:
    // about ten per resident warp (round 2; three before): SMs that join late, when the scout
    // lets go of them, and the last wave then balance to within a tenth of a warp's share, for
    // (NQ-1)/R = 2 % of warm-up periods (3.91 -> 3.72 ms in the pump, profiles/r02_stream_segs.txt).
    const int scout_ctas = (mp.nchan + scout_threads(b, pump) - 1) / scout_threads(b, pump);
    // stand-alone, the replay of the next block runs beside this kernel: leave it its SMs.  In the
    // pump it runs beside the FFT that precedes this kernel and is normally done by now, so every SM
    // is taken; work is handed out dynamically, so an SM the scout still holds just joins late.
    sp.grid = pump ? b->ctx->sm_count : std::max(b->ctx->sm_count - scout_ctas, b->ctx->sm_count / 2);
    sp.warps_per_cta = (FMT == FMT_S16) ? stream::kWarps : stream::kWarpsF32;
    const int resident = sp.grid * sp.warps_per_cta;
    static int segs_per_warp = 0;
    if (!segs_per_warp) segs_per_warp = env_int("JSDR_STREAM_SEGS", 1, 64, 10);   // (tuning aid)
    int nseg = std::max(1, segs_per_warp * resident / sp.ncw);
    int R = (mp.NO + nseg - 1) / nseg;
    if (R < 64) R = 64;
    sp.R = R;
    sp.nseg = (mp.NO + R - 1) / R;
    sp.ds_out = mp.ds_out;
    sp.max_ds = mp.max_ds;
    sp.work_counter = reinterpret_cast<unsigned *>(b->d_nbits.get() + b->nchan);   // one spare word behind nbits[]
    for (int k = 0; k < stream::kMaxTaps; k++) {
        sp.taps[k] = (k < b->ntaps) ? b->h_taps[k] : 0.0;
        sp.tapsf[k] = (float)sp.taps[k];
    }
    const bool f32 = b->precision == JSDR_PREC_F32;
    if (b->ntaps == 27 && mp.D == 10)
        return f32 ? launch_stream_shape<FMT, stream::PREC_F32, 27, 10>(b, sp) : launch_stream_shape<FMT, stream::PREC_F64, 27, 10>(b, sp);
    if (b->ntaps == 27 && mp.D == 20)
        return f32 ? launch_stream_shape<FMT, stream::PREC_F32, 27, 20>(b, sp) : launch_stream_shape<FMT, stream::PREC_F64, 27, 20>(b, sp);
    return f32 ? launch_stream_shape<FMT, stream::PREC_F32, 64, 20>(b, sp) : launch_stream_shape<FMT, stream::PREC_F64, 64, 20>(b, sp);
}

// doBufferFFT (:406-464) for every channel of the bank: binary64 forward transform, search,
// 204 bins to DC, inverse transform, decimator on the real part.  The tuner phase is not
// advanced (the reference's FFT variant never calls RxMixTuner).
// k_at_search keeps the N/4 magnitudes of the scanned band (+ 64 words) in shared memory as doubles
constexpr int kAutoTuneMaxN = 115712;                  // 8 * (N/4 + 64) <= 232448 bytes

template <int FMT>
int autotune_block(jsdr_bpsk *b, const void *d_in, int S, long long chan_stride, int ic, int qc, int n0, int NO)
{
    jsdr_ctx *ctx = b->ctx;
    const int nchan = b->nchan, N = S;
    const size_t bytes = sizeof(double2) * (size_t)nchan * (size_t)N;
    if (!b->at.d_at_state) {
        const char *what = "auto-tune workspace";
        jsdr_bpsk::AutoTune g;
        for (int i = 0; i < 2; i++) JSDR_TRY(g.d_at_work[i].alloc(bytes, what));
        for (int i = 0; i < 2; i++) JSDR_TRY(g.d_at_rev[i].alloc(bytes, what));
        JSDR_TRY(g.d_at_state.alloc_zeroed(sizeof(AutoTuneState) * (size_t)nchan, ctx->stream, what));
        b->at = std::move(g);
    }
    double2 *work[2] = {b->at.d_at_work[0].get(), b->at.d_at_work[1].get()};
    double2 *rev[2] = {b->at.d_at_rev[0].get(), b->at.d_at_rev[1].get()};
    JSDR_REQUIRE(fftg::make_plan(N).nstages > 0, JSDR_EUNSUPPORTED, "block length has a prime factor other than 2, 3, 5, 7");
    JSDR_REQUIRE(N >= 1024 && N <= kAutoTuneMaxN, JSDR_EUNSUPPORTED, "auto-tune needs blocks of 1024 to 115712 samples");
    const long long total = (long long)nchan * N;
    k_at_load<FMT><<<(unsigned)((total + 255) / 256), 256, 0, ctx->stream>>>(d_in, chan_stride, S, nchan, ic, qc, work[0]);
    JSDR_TRY(launched(ctx, "k_at_load"));
    int rc = JSDR_OK;
    double2 *fwd = fftg::run<double>(ctx, ctx->stream, work[0], work[1], N, nchan, -1, &rc);   // :422-423
    if (rc != JSDR_OK) return rc;
    JSDR_CUDA(cudaMemsetAsync(rev[0], 0, bytes, ctx->stream));                                         // :419-420
    const size_t smem = sizeof(double) * (size_t)(N / 4 + 64);
    JSDR_CUDA(cudaFuncSetAttribute(k_at_search, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_at_search<<<nchan, 256, smem, ctx->stream>>>(fwd, rev[0], N, b->doUp, b->at.d_at_state.get());
    JSDR_TRY(launched(ctx, "k_at_search"));
    double2 *inv = fftg::run<double>(ctx, ctx->stream, rev[0], rev[1], N, nchan, +1, &rc);     // :459
    if (rc != JSDR_OK) return rc;
    dim3 grid((std::max(NO, 1) + 127) / 128, nchan);
    k_at_decim<<<grid, 128, 0, ctx->stream>>>(inv, N, 1.0 / (double)N, b->d_ds_hist[b->ds_hist_cur].get(),
                                              b->d_ds_hist[b->ds_hist_cur ^ 1].get(), b->d_taps.get(), b->ntaps, b->D, n0, NO,
                                              b->d_ds_out.get(), b->max_ds);
    return launched(ctx, "k_at_decim");
}

// The tuner + decimator of one block behind its phase replay (checkpoints `ckpt`): the streaming
// kernel or the tile kernel, then the history tail.
template <int FMT>
int mix_decimate(jsdr_bpsk *b, const void *d_in, int S, long long chan_stride, int ic, int qc, int n0, int NO,
                 const double *ckpt, bool pump)
{
    jsdr_ctx *ctx = b->ctx;
    const int D = b->D;
    const int nchan = b->nchan;
    MixParams mp;
    mp.in = d_in;
    mp.chan_stride = chan_stride;
    mp.S = S;
    mp.ic = ic;
    mp.qc = qc;
    mp.tu_inc = b->d_tu_inc.get();
    mp.tu_dx = b->d_tu_dx.get();
    mp.ckpt = ckpt;
    mp.nchan = nchan;
    mp.hist_in = b->d_ds_hist[b->ds_hist_cur].get();
    mp.hist_out = b->d_ds_hist[b->ds_hist_cur ^ 1].get();
    mp.ntaps = b->ntaps;
    mp.cossin = b->d_cossin2.get();
    mp.D = D;
    mp.n0 = n0;
    mp.NO = NO;
    mp.magicD = (unsigned)(4294967296ULL / (unsigned)D) + 1u;
    mp.pad = (D & 1) ? 0 : 1;          // even D: one pad slot per D samples makes the lane stride odd
    mp.ds_out = b->d_ds_out.get();
    mp.max_ds = b->max_ds;
    memcpy(mp.taps, b->h_taps, sizeof(mp.taps));
    {
        const int H = b->ntaps - 1;
        for (int k = 0; k < kMaxDsTaps; k++) {
            const int d = (k <= H) ? H - k : 0;
            mp.off[k] = (int)sizeof(double2) * (d + mp.pad * (d / D));
        }
    }
    bool streamed = false;
    if (NO > 0 && b->kernel_mode != JSDR_KERNEL_TILE) {
        // many channels: the streaming kernel (bpsk_stream.cuh); needs a compiled (taps, D) shape
        const bool shape_ok = (b->ntaps == 27 && D == 10) || (b->ntaps == 27 && D == 20) || (b->ntaps == 64 && D == 20);
        const bool want = b->kernel_mode == JSDR_KERNEL_STREAM || (nchan >= 32 && NO >= 64) ||
                          (b->precision == JSDR_PREC_F32 && nchan >= 8);
        if (shape_ok && want) {
            JSDR_TRY(launch_stream<FMT>(b, mp, S, pump));
            streamed = true;
        }
    }
    if (NO > 0 && !streamed) {
        const int span = (kTileOut - 1) * D + b->ntaps;
        const size_t m_bytes = sizeof(double2) * (size_t)(span + mp.pad * (span / D) + 2);
        mp.ix_off = (int)m_bytes;
        const size_t smem = m_bytes + sizeof(uint16_t) * (size_t)(span + 64 + (span + 64) / 32 + 4);
        dim3 grid((NO + kTileOut - 1) / kTileOut, nchan);
        // compile-time (taps, D) for the shapes that matter; anything else runs the generic loop
        void (*kern)(const MixParams) = k_mixdecim<FMT, 0, 0>;
        if (b->ntaps == 27 && D == 10) kern = k_mixdecim<FMT, 27, 10>;
        else if (b->ntaps == 27 && D == 20) kern = k_mixdecim<FMT, 27, 20>;
        else if (b->ntaps == 64 && D == 20) kern = k_mixdecim<FMT, 64, 20>;
        JSDR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ProfScope prof(ctx, JSDR_K_MIXDECIM, ctx->stream);
        kern<<<grid, kTileThreads, smem, ctx->stream>>>(mp);
        JSDR_TRY(launched(ctx, "k_mixdecim"));
    }
    if (b->ntaps > 1) {
        k_tuner_tail<FMT><<<nchan, 128, 0, ctx->stream>>>(mp);
        JSDR_TRY(launched(ctx, "k_tuner_tail"));
    }
    return JSDR_OK;
}

}  // namespace

// jsdr_bpsk_receive_* in two halves, so that the pump (pump.cu) can enqueue its own kernels between
// them, beside the phase replay on the side stream.  The first half checks, forks this block's
// data-independent replays onto the side streams and puts the input on the device: *d_in is what
// the second half reads, or nullptr after an empty block, which is then complete.
int jsdr::bpsk::receive_begin(jsdr_bpsk *b, const void *in, int fmt, int S, long long chan_stride, int mem,
                              bool pump, const void **d_in)
{
    *d_in = nullptr;
    JSDR_REQUIRE(b && in, JSDR_EINVAL, "null argument");
    JSDR_REQUIRE(S >= 0 && S <= b->max_block, JSDR_EINVAL, "nsamples exceeds max_block_samples");
    JSDR_REQUIRE(chan_stride == 0 || chan_stride >= S, JSDR_EINVAL, "chan_stride smaller than nsamples");
    JSDR_REQUIRE(mem == JSDR_MEM_HOST || mem == JSDR_MEM_DEVICE, JSDR_EINVAL, "bad mem");
    jsdr_ctx *ctx = b->ctx;
    JSDR_TRY(ctx->bind());
    if (b->ds_read_pending) {      // an asynchronous read of the previous block's output is still draining
        JSDR_CUDA(cudaStreamWaitEvent(ctx->stream, b->ev_ds_read, 0));
        b->ds_read_pending = 0;
    }
    b->last_nds = 0;
    if (b->stages >= 2) JSDR_TRY(ensure_stage_buffers(b));   // (before the empty-block return: the reads that follow an
                                                             //  empty FIRST block answer "nothing", not "stage has not run")
    if (S == 0) {
        JSDR_CUDA(cudaMemsetAsync(b->d_nbits.get(), 0, sizeof(int32_t) * b->nchan, ctx->aux));
        if (b->fec && b->stages >= 3 && b->stage.d_bits) JSDR_TRY(jsdr_fec_after_bits(b));   // no bits: no frames either
        return JSDR_OK;
    }
    const int NO = (b->ds_cnt + S) / b->D;

    // ---- fork: data-independent work on the side stream.  The tuner plan for this
    // block was normally computed while the previous block was being processed.
    jsdr_bpsk::TunerPlan &P = b->plan[b->plan_cur];
    const bool autotune = b->dofft != 0;               // :358-364 receive(): doBufferFFT instead of doBufferTune
    if (autotune) JSDR_REQUIRE(S == b->max_block, JSDR_EINVAL, "auto-tune needs whole blocks of max_block_samples");
    JSDR_CUDA(cudaEventRecord(ctx->ev_fork, ctx->stream));
    JSDR_CUDA(cudaStreamWaitEvent(ctx->side, ctx->ev_fork, 0));
    JSDR_CUDA(cudaStreamWaitEvent(ctx->side2, ctx->ev_fork, 0));
    if (!autotune && !(P.valid && P.S == S)) JSDR_TRY(launch_scout(b, P, S, pump));
    const int kb = b->bit_cur;                         // buffer of the 9600 S/s stages for this block
    if (b->stages >= 2 && NO > 0) {
        // normally replayed already, behind the previous block's tuner scout (look-ahead below)
        if (!(b->vco_ahead_valid && b->vco_ahead_NO == NO && b->vco_ahead_kb == kb)) JSDR_TRY(launch_vco_scout(b, NO, kb));
        b->vco_ahead_valid = false;
    }
    JSDR_CUDA(cudaEventRecord(ctx->ev_join, ctx->side));

    // ---- input
    if (mem == JSDR_MEM_HOST) {
        const size_t esz = (fmt == FMT_S16) ? 4 : 8;
        const size_t bytes = esz * ((chan_stride == 0) ? (size_t)S : (size_t)chan_stride * (b->nchan - 1) + S);
        JSDR_TRY(b->d_in.grow(bytes, "tuner bank staging"));
        JSDR_CUDA(cudaMemcpyAsync(b->d_in.get(), in, bytes, cudaMemcpyHostToDevice, ctx->stream));
        in = b->d_in.get();
    }
    *d_in = in;
    return JSDR_OK;
}

// The second half: the tuner + decimator behind this block's phase replay, the next block's
// replay, the 9600 S/s stages.
int jsdr::bpsk::receive_end(jsdr_bpsk *b, const void *d_in, int fmt, int S, long long chan_stride, int ic, int qc,
                            int mem, bool pump)
{
    jsdr_ctx *ctx = b->ctx;
    const int D = b->D;
    const int NO = (b->ds_cnt + S) / D;
    const int n0 = D - 1 - b->ds_cnt;
    const int nchan = b->nchan;
    const int kb = b->bit_cur;
    const bool s16 = fmt == FMT_S16;
    if (b->dofft) {
        JSDR_TRY(s16 ? autotune_block<FMT_S16>(b, d_in, S, chan_stride, ic, qc, n0, NO)
                     : autotune_block<FMT_F32>(b, d_in, S, chan_stride, ic, qc, n0, NO));
    } else {
        jsdr_bpsk::TunerPlan &P = b->plan[b->plan_cur];
        JSDR_CUDA(cudaStreamWaitEvent(ctx->stream, P.ready, 0));
        // (ev_join — the VCO / bit-phase replay of this block — is only needed by the matched filter:
        // the tuner + decimator runs beside it)
        JSDR_TRY(s16 ? mix_decimate<FMT_S16>(b, d_in, S, chan_stride, ic, qc, n0, NO, P.ckpt.get(), pump)
                     : mix_decimate<FMT_F32>(b, d_in, S, chan_stride, ic, qc, n0, NO, P.ckpt.get(), pump));
        // this plan is consumed: its end phase becomes the committed phase, and the
        // scout starts on the next block (same length assumed) while the rest of this
        // one is still in flight
        JSDR_CUDA(cudaEventRecord(P.consumed, ctx->stream));
        P.used = true;
        P.valid = false;
        b->d_tu_phase = P.phase_end.get();
        b->plan_cur ^= 1;
        jsdr_bpsk::TunerPlan &Pn = b->plan[b->plan_cur];
        if (Pn.used) JSDR_CUDA(cudaStreamWaitEvent(ctx->side, Pn.consumed, 0));
        JSDR_TRY(launch_scout(b, Pn, S, pump));
    }
    b->ds_hist_cur ^= 1;
    b->ds_cnt = (b->ds_cnt + S) % D;
    b->cnt_raw += S;
    b->last_nds = NO;

    // ---- matched filter, bit timing
    if (b->stages >= 2 && NO > 0) {
        JSDR_CUDA(cudaStreamWaitEvent(ctx->stream, b->stage.ev_vco_ready, 0));
        b->vco_state_cur ^= 1;                         // this block's replay is consumed: its end state is committed
        DmParams dp;
        dp.ds = b->d_ds_out.get();
        dp.max_ds = b->max_ds;
        dp.NO = NO;
        dp.vco_ix = b->stage.d_vco_ix[kb].get();
        dp.hist_in = b->stage.d_dm_hist[b->dm_hist_cur].get();
        dp.hist_out = b->stage.d_dm_hist[b->dm_hist_cur ^ 1].get();
        dp.dmtaps = b->d_dmtaps.get();
        dp.cossin = b->d_cossin.get();
        dp.base65 = (int)(b->cnt_ds % 65);
        dp.dm_out = b->stage.d_dm_buf[kb].get();
        b->d_dm_out = b->stage.d_dm_buf[kb].get();
        if (b->bits_used[kb]) JSDR_CUDA(cudaStreamWaitEvent(ctx->stream, b->stage.ev_bits_done[kb], 0));
        dim3 grid((NO + kDm2Tile - 1) / kDm2Tile, nchan);
        const size_t dm_smem = sizeof(double2) * (size_t)(kDm2Tile + 64 + 16);
        static PerDeviceFlag dm_attr;
        JSDR_TRY(dm_attr.once(ctx->device, [&]() -> int {
            JSDR_CUDA(cudaFuncSetAttribute(k_matched, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dm_smem));
            return JSDR_OK;
        }));
        {
            ProfScope prof(ctx, JSDR_K_MATCHED, ctx->stream);
            k_matched<<<grid, kDm2Threads, dm_smem, ctx->stream>>>(dp);
        }
        JSDR_TRY(launched(ctx, "k_matched"));
        k_dm_tail<<<nchan, 64, 0, ctx->stream>>>(dp);
        JSDR_TRY(launched(ctx, "k_dm_tail"));
        b->dm_hist_cur ^= 1;
        if (b->stages >= 3) {
            // bit timing on the auxiliary stream: it overlaps the next block's tuner + matched filter
            JSDR_CUDA(cudaEventRecord(b->stage.ev_dm_ready, ctx->stream));
            JSDR_CUDA(cudaStreamWaitEvent(ctx->aux, b->stage.ev_dm_ready, 0));
            TimingParams tp;
            tp.dm = b->stage.d_dm_buf[kb].get();
            tp.max_ds = b->max_ds;
            tp.NO = NO;
            tp.nchan = nchan;
            tp.bit_roll = b->stage.d_bit_roll[kb].get();
            tp.ts = b->d_ts.get();
            tp.bits = b->stage.d_bits.get();
            tp.bit_at = b->stage.d_bit_at.get();
            tp.nbits = b->d_nbits.get();
            tp.max_bits = b->max_bits;
            tp.cnt_ds0 = b->cnt_ds;
            {
                ProfScope prof(ctx, JSDR_K_TIMING, ctx->aux);
                k_timing<<<(nchan + 31) / 32, 32, 0, ctx->aux>>>(tp);
            }
            JSDR_TRY(launched(ctx, "k_timing"));
        }
        b->bit_cur ^= 1;
        // look ahead: the VCO / bit-phase replay of the next block (same length assumed), on the
        // side stream behind the next block's tuner scout
        const int no_next = (b->ds_cnt + S) / D;       // ds_cnt already carries this block
        if (no_next > 0) {
            JSDR_TRY(launch_vco_scout(b, no_next, b->bit_cur));
            b->vco_ahead_valid = true;
            b->vco_ahead_NO = no_next;
            b->vco_ahead_kb = b->bit_cur;
        }
    }
    if (NO == 0)   // nothing reached the 9600 S/s stage in this call: no bits either
        JSDR_CUDA(cudaMemsetAsync(b->d_nbits.get(), 0, sizeof(int32_t) * nchan, ctx->aux));
    if (b->fec && b->stages >= 3 && b->stage.d_bits) JSDR_TRY(jsdr_fec_after_bits(b));   // :553-574, auxiliary stream
    if (b->stages >= 3 && NO > 0) {
        JSDR_CUDA(cudaEventRecord(b->stage.ev_bits_done[kb], ctx->aux));
        b->bits_used[kb] = true;
    }
    b->cnt_ds += NO;
    if (mem == JSDR_MEM_HOST) {
        JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
        JSDR_CUDA(cudaStreamSynchronize(ctx->aux));
    }
    return JSDR_OK;
}

int jsdr::bpsk::receive(jsdr_bpsk *b, const void *in, int fmt, int S, long long chan_stride, int ic, int qc, int mem,
                        bool pump)
{
    const void *d_in;
    JSDR_TRY(receive_begin(b, in, fmt, S, chan_stride, mem, pump, &d_in));
    return d_in ? receive_end(b, d_in, fmt, S, chan_stride, ic, qc, mem, pump) : JSDR_OK;
}

extern "C" int jsdr_bpsk_create(jsdr_ctx *ctx, int rate, int nchan, const double *tuning_hz,
                                int max_block_samples, jsdr_bpsk **out)
try {
    JSDR_REQUIRE(ctx && out && tuning_hz, JSDR_EINVAL, "null argument");
    JSDR_REQUIRE(rate >= 9600 && rate <= 64 * 9600 && nchan > 0 && nchan <= 65535 && max_block_samples > 0,
                 JSDR_EINVAL, "need 9600 <= rate <= 614400, 0 < nchan < 65536, max_block_samples > 0");
    for (int c = 0; c < nchan; c++)
        JSDR_REQUIRE(std::isfinite(tuning_hz[c]), JSDR_EINVAL, "every tuning must be a finite frequency (the reference's comes from an int config key or the dialog, :175-195)");
    JSDR_TRY(ctx->bind());
    std::unique_ptr<jsdr_bpsk> b(new jsdr_bpsk(ctx));
    b->rate = rate;
    b->D = rate / 9600;                 // :476 adsc.rate/DOWN_SAMPLE_RATE (integer division)
    b->nchan = nchan;
    b->max_block = max_block_samples;
    b->max_ds = max_block_samples / b->D + 2;
    b->max_words = (int)((max_block_samples + 31LL) / 32 + 1);
    b->max_bits = b->max_ds;
    b->h_tuning.assign(tuning_hz, tuning_hz + nchan);
    const size_t nc = (size_t)nchan;
    const char *what = "jsdr_bpsk_create";
    cudaStream_t st = ctx->stream;
    JSDR_TRY(b->d_taps.alloc_zeroed(sizeof(double) * kMaxDsTaps, st, what));
    JSDR_TRY(b->d_dmtaps.alloc_zeroed(sizeof(double) * kDmTaps, st, what));
    JSDR_TRY(b->d_cossin.alloc_zeroed(sizeof(double) * 512, st, what));
    JSDR_TRY(b->d_cossin2.alloc_zeroed(sizeof(double2) * 257, st, what));
    JSDR_TRY(b->d_tu_inc.alloc_zeroed(sizeof(double) * nc, st, what));
    JSDR_TRY(b->d_tu_par.alloc_zeroed(sizeof(ScoutChan) * nc, st, what));
    JSDR_TRY(b->d_tu_dx.alloc_zeroed(sizeof(unsigned long long) * nc, st, what));
    JSDR_TRY(b->d_tu_dx56.alloc_zeroed(sizeof(unsigned long long) * nc, st, what));
    JSDR_TRY(b->d_tu_phase0.alloc_zeroed(sizeof(double) * nc, st, what));
    b->d_tu_phase = b->d_tu_phase0.get();
    for (jsdr_bpsk::TunerPlan &P : b->plan) {
        JSDR_TRY(P.ckpt.alloc_zeroed(sizeof(double) * nc * b->max_words, st, what));
        JSDR_TRY(P.phase_end.alloc_zeroed(sizeof(double) * nc, st, what));
        JSDR_TRY(P.ready.create(what));
        JSDR_TRY(P.consumed.create(what));
    }
    for (int i = 0; i < 2; i++) JSDR_TRY(b->d_ds_hist[i].alloc_zeroed(sizeof(double2) * kMaxDsTaps * nc, st, what));
    JSDR_TRY(b->d_ds_out.alloc_zeroed(sizeof(double2) * nc * b->max_ds, st, what));
    JSDR_TRY(b->d_vco_state.alloc_zeroed(sizeof(double) * 4, st, what));
    JSDR_TRY(b->d_ts.alloc_zeroed(sizeof(TimingState) * nc, st, what));
    JSDR_TRY(b->d_nbits.alloc_zeroed(sizeof(int32_t) * (nc + 1), st, what));   // + the streaming kernel's work counter
    // tables and constants, computed on the host exactly as the reference's setup code does
    std::vector<double> cossin(512);
    for (int n = 0; n < 256; n++) {                       // :159-162
        cossin[n] = cos(n * 2.0 * M_PI / 256);
        cossin[256 + n] = sin(n * 2.0 * M_PI / 256);
    }
    std::vector<double> taps(kMaxDsTaps, 0.0), dmt(kDmTaps);
    for (int i = 0; i < 27; i++) taps[i] = (double)kDsFilterF[i];
    for (int i = 0; i < kDmTaps; i++) dmt[i] = (double)kDmFilterF[i];
    std::vector<double> inc(nchan);
    std::vector<unsigned long long> dx(nchan), dx56(nchan);
    for (int c = 0; c < nchan; c++) {
        inc[c] = 2.0 * M_PI * tuning_hz[c] / (double)rate;   // :196
        dx[c] = index_step_fixed(inc[c]);
        dx56[c] = index_step_fixed56(inc[c]);
    }
    std::vector<double> cs2(2 * 257);
    for (int n = 0; n < 256; n++) {
        cs2[2 * n] = cossin[n];
        cs2[2 * n + 1] = cossin[256 + n];
    }
    cs2[512] = cs2[513] = 1.0;     // bypass entry: x*1.0 is exact
    for (int i = 0; i < kMaxDsTaps; i++) b->h_taps[i] = taps[i];
    std::vector<TimingState> ts(nchan);
    memset(ts.data(), 0, sizeof(TimingState) * nc);
    for (int c = 0; c < nchan; c++) ts[c].dmEnergyOut = 1.0;                             // :499
    std::vector<ScoutChan> par(nchan);
    for (int c = 0; c < nchan; c++) par[c] = scout_chan(inc[c]);
    JSDR_TRY(upload(ctx, b->d_cossin.get(), cossin.data(), sizeof(double) * 512));
    JSDR_TRY(upload(ctx, b->d_taps.get(), taps.data(), sizeof(double) * kMaxDsTaps));
    JSDR_TRY(upload(ctx, b->d_dmtaps.get(), dmt.data(), sizeof(double) * kDmTaps));
    JSDR_TRY(upload(ctx, b->d_tu_inc.get(), inc.data(), sizeof(double) * nc));
    JSDR_TRY(upload(ctx, b->d_tu_par.get(), par.data(), sizeof(ScoutChan) * nc));
    JSDR_TRY(upload(ctx, b->d_tu_dx.get(), dx.data(), sizeof(unsigned long long) * nc));
    JSDR_TRY(upload(ctx, b->d_tu_dx56.get(), dx56.data(), sizeof(unsigned long long) * nc));
    JSDR_TRY(upload(ctx, b->d_cossin2.get(), cs2.data(), sizeof(double) * 2 * 257));
    JSDR_TRY(upload(ctx, b->d_ts.get(), ts.data(), sizeof(TimingState) * nc));
    *out = b.release();
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_bpsk_destroy(jsdr_bpsk *b)
try {
    delete b;
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_bpsk_set_stages(jsdr_bpsk *b, int stages)
try {
    JSDR_REQUIRE(b && stages >= 1 && stages <= 3, JSDR_EINVAL, "stages must be 1..3");
    b->stages = stages;
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_bpsk_set_autotune(jsdr_bpsk *b, int dofft, int do_upper)
try {
    JSDR_REQUIRE(b, JSDR_EINVAL, "null argument");
    if (dofft) {                                       // the transform length is the block length (:421)
        const int N = b->max_block;
        JSDR_REQUIRE(N >= 1024, JSDR_EUNSUPPORTED, "auto-tune needs blocks of at least 1024 samples");
        JSDR_REQUIRE(N <= kAutoTuneMaxN, JSDR_EUNSUPPORTED,
                     "auto-tune supports blocks of up to 115712 samples (the band search keeps N/4 bins in shared memory)");
        JSDR_REQUIRE(fftg::make_plan(N).nstages > 0, JSDR_EUNSUPPORTED, "block length has a prime factor other than 2, 3, 5, 7");
    }
    b->dofft = dofft != 0;
    b->doUp = do_upper != 0;
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_bpsk_read_centre(jsdr_bpsk *b, int32_t *centre_bin)
try {
    JSDR_REQUIRE(b && centre_bin, JSDR_EINVAL, "null argument");
    jsdr_ctx *ctx = b->ctx;
    JSDR_TRY(ctx->bind());
    for (int c = 0; c < b->nchan; c++) centre_bin[c] = 0;
    if (!b->at.d_at_state) return JSDR_OK;                // no auto-tune block yet (centreBin = 0, :405)
    std::vector<AutoTuneState> st(b->nchan);
    JSDR_CUDA(cudaMemcpyAsync(st.data(), b->at.d_at_state.get(), sizeof(AutoTuneState) * (size_t)b->nchan, cudaMemcpyDeviceToHost, ctx->stream));
    JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int c = 0; c < b->nchan; c++) centre_bin[c] = st[c].centreBin;
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_bpsk_set_precision(jsdr_bpsk *b, int precision)
try {
    JSDR_REQUIRE(b && (precision == JSDR_PREC_F64 || precision == JSDR_PREC_F32), JSDR_EINVAL, "bad precision");
    b->precision = precision;
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_bpsk_set_kernel(jsdr_bpsk *b, int mode)
try {
    JSDR_REQUIRE(b && mode >= JSDR_KERNEL_AUTO && mode <= JSDR_KERNEL_STREAM, JSDR_EINVAL, "bad kernel mode");
    b->kernel_mode = mode;
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_bpsk_set_tuning(jsdr_bpsk *b, int chan, double hz)
try {
    JSDR_REQUIRE(b && chan >= 0 && chan < b->nchan, JSDR_EINVAL, "bad channel");
    JSDR_REQUIRE(std::isfinite(hz), JSDR_EINVAL, "tuning must be a finite frequency (the reference's comes from an int config key or the dialog, :175-195)");
    JSDR_TRY(b->ctx->bind());
    // the scout may be running ahead with the old increment: let it finish and drop its plan
    JSDR_CUDA(cudaStreamSynchronize(b->ctx->side));
    JSDR_CUDA(cudaStreamSynchronize(b->ctx->side2));
    b->plan[0].valid = b->plan[1].valid = false;
    b->h_tuning[chan] = hz;
    double inc = 2.0 * M_PI * hz / (double)b->rate;       // :188
    unsigned long long dx = index_step_fixed(inc);
    JSDR_TRY(upload(b->ctx, b->d_tu_dx.get() + chan, &dx, sizeof(dx)));
    unsigned long long dx56 = index_step_fixed56(inc);
    JSDR_TRY(upload(b->ctx, b->d_tu_dx56.get() + chan, &dx56, sizeof(dx56)));
    const ScoutChan sc = scout_chan(inc);
    JSDR_TRY(upload(b->ctx, b->d_tu_par.get() + chan, &sc, sizeof(sc)));
    return upload(b->ctx, b->d_tu_inc.get() + chan, &inc, sizeof(double));
} JSDR_CATCH_ALL

extern "C" int jsdr_bpsk_set_ds_filter(jsdr_bpsk *b, const double *taps, int ntaps)
try {
    JSDR_REQUIRE(b && taps && ntaps >= 1 && ntaps <= kMaxDsTaps, JSDR_EINVAL, "1..128 taps");
    JSDR_TRY(b->ctx->bind());
    std::vector<double> t(kMaxDsTaps, 0.0);
    for (int i = 0; i < ntaps; i++) t[i] = taps[i];
    JSDR_TRY(upload(b->ctx, b->d_taps.get(), t.data(), sizeof(double) * kMaxDsTaps));
    for (int i = 0; i < kMaxDsTaps; i++) b->h_taps[i] = t[i];
    b->ntaps = ntaps;
    return bpsk_reset_ds(b);
} JSDR_CATCH_ALL

extern "C" int jsdr_bpsk_receive_f32(jsdr_bpsk *b, const float *iq, int nsamples, int64_t chan_stride, int mem)
try {
    return bpsk::receive(b, iq, FMT_F32, nsamples, chan_stride, 0, 0, mem, false);
} JSDR_CATCH_ALL

extern "C" int jsdr_bpsk_receive_s16(jsdr_bpsk *b, const int16_t *raw, int nsamples, int64_t chan_stride,
                                     int ic, int qc, int mem)
try {
    return bpsk::receive(b, raw, FMT_S16, nsamples, chan_stride, ic, qc, mem, false);
} JSDR_CATCH_ALL

extern "C" int jsdr_bpsk_last_counts(jsdr_bpsk *b, int32_t *n_ds)
try {
    JSDR_REQUIRE(b && n_ds, JSDR_EINVAL, "null argument");
    *n_ds = b->last_nds;
    return JSDR_OK;
} JSDR_CATCH_ALL

namespace {
int read_rows(jsdr_bpsk *b, const double2 *src, double *out, int mem)
{
    JSDR_REQUIRE(b && out, JSDR_EINVAL, "null argument");
    jsdr_ctx *ctx = b->ctx;
    JSDR_TRY(ctx->bind());
    if (b->last_nds == 0) return JSDR_OK;
    JSDR_CUDA(cudaMemcpy2DAsync(out, sizeof(double2) * b->last_nds, src, sizeof(double2) * b->max_ds,
                                sizeof(double2) * b->last_nds, b->nchan,
                                mem == JSDR_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice,
                                ctx->stream));
    if (mem == JSDR_MEM_HOST) JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
    return JSDR_OK;
}
}  // namespace

extern "C" int jsdr_bpsk_read_ds(jsdr_bpsk *b, double *out, int mem) { return read_rows(b, b ? b->d_ds_out.get() : nullptr, out, mem); }

// The same rows, copied on the download stream behind the decimator and without waiting: the
// copy overlaps whatever the caller submits next (the upload of the following block, in the
// pump); jsdr_ctx_sync -- or the next synchronous read -- completes it.
extern "C" int jsdr_bpsk_read_ds_async(jsdr_bpsk *b, double *out, int mem)
try {
    JSDR_REQUIRE(b && out, JSDR_EINVAL, "null argument");
    JSDR_REQUIRE(mem == JSDR_MEM_HOST || mem == JSDR_MEM_DEVICE, JSDR_EINVAL, "bad mem");
    jsdr_ctx *ctx = b->ctx;
    JSDR_TRY(ctx->bind());
    if (!b->ev_ds_read) {
        Event ready, read;
        JSDR_TRY(ready.create("jsdr_bpsk_read_ds_async"));
        JSDR_TRY(read.create("jsdr_bpsk_read_ds_async"));
        b->ev_ds_ready = std::move(ready);
        b->ev_ds_read = std::move(read);
    }
    if (b->last_nds == 0) return JSDR_OK;
    JSDR_CUDA(cudaEventRecord(b->ev_ds_ready, ctx->stream));
    JSDR_CUDA(cudaStreamWaitEvent(ctx->copy_out, b->ev_ds_ready, 0));
    JSDR_CUDA(cudaMemcpy2DAsync(out, sizeof(double2) * b->last_nds, b->d_ds_out.get(), sizeof(double2) * b->max_ds,
                                sizeof(double2) * b->last_nds, b->nchan,
                                mem == JSDR_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice,
                                ctx->copy_out));
    JSDR_CUDA(cudaEventRecord(b->ev_ds_read, ctx->copy_out));
    b->ds_read_pending = 1;
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_bpsk_read_dm(jsdr_bpsk *b, double *out, int mem)
try {
    JSDR_REQUIRE(b && b->stages >= 2 && b->d_dm_out, JSDR_ESTATE, "matched filter stage is disabled or has not run");
    return read_rows(b, b->d_dm_out, out, mem);
} JSDR_CATCH_ALL

extern "C" int jsdr_bpsk_read_bits(jsdr_bpsk *b, int8_t *bits, int64_t *bit_at, int32_t *nbits,
                                   int max_bits, int mem)
try {
    JSDR_REQUIRE(b && nbits, JSDR_EINVAL, "null argument");
    JSDR_REQUIRE(b->stages >= 3 && b->stage.d_bits, JSDR_ESTATE, "bit decision stage is disabled or has not run");
    JSDR_REQUIRE(max_bits >= 0, JSDR_EINVAL, "negative max_bits");
    jsdr_ctx *ctx = b->ctx;
    JSDR_TRY(ctx->bind());
    const cudaMemcpyKind kind = mem == JSDR_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    JSDR_CUDA(cudaMemcpyAsync(nbits, b->d_nbits.get(), sizeof(int32_t) * b->nchan, kind, ctx->aux));
    const int w = max_bits < b->max_bits ? max_bits : b->max_bits;
    if (bits && w > 0)
        JSDR_CUDA(cudaMemcpy2DAsync(bits, (size_t)max_bits, b->stage.d_bits.get(), (size_t)b->max_bits, (size_t)w,
                                    b->nchan, kind, ctx->aux));
    if (bit_at && w > 0)
        JSDR_CUDA(cudaMemcpy2DAsync(bit_at, sizeof(int64_t) * max_bits, b->stage.d_bit_at.get(),
                                    sizeof(long long) * b->max_bits, sizeof(int64_t) * w, b->nchan, kind,
                                    ctx->aux));
    if (mem == JSDR_MEM_HOST) JSDR_CUDA(cudaStreamSynchronize(ctx->aux));
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_bpsk_read_counters(jsdr_bpsk *b, int64_t *counters)
try {
    JSDR_REQUIRE(b && counters, JSDR_EINVAL, "null argument");
    jsdr_ctx *ctx = b->ctx;
    JSDR_TRY(ctx->bind());
    std::vector<TimingState> ts(b->nchan);
    JSDR_CUDA(cudaMemcpyAsync(ts.data(), b->d_ts.get(), sizeof(TimingState) * (size_t)b->nchan,
                              cudaMemcpyDeviceToHost, ctx->aux));
    JSDR_CUDA(cudaStreamSynchronize(ctx->aux));
    for (int c = 0; c < b->nchan; c++) {
        counters[4 * c + 0] = b->cnt_raw;
        counters[4 * c + 1] = b->cnt_ds;
        counters[4 * c + 2] = ts[c].cntBit;
        counters[4 * c + 3] = 0;
    }
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_bpsk_ds_device_ptr(jsdr_bpsk *b, double **dev_ptr)
try {
    JSDR_REQUIRE(b && dev_ptr, JSDR_EINVAL, "null argument");
    *dev_ptr = reinterpret_cast<double *>(b->d_ds_out.get());
    return JSDR_OK;
} JSDR_CATCH_ALL

// The decimator and matched-filter taps as the kernels use them ((double)(float) of the
// F-suffixed literals, FUNcubeBPSKDemod.java:27-77), for the reference-pinning tests
// (tests/test_ref_tables.py compares every entry with the literals parsed from the Java source).
// Host only: no device needed.
extern "C" int jsdr_probe_taps(double *ds27, double *dm65)
try {
    JSDR_REQUIRE(ds27 && dm65, JSDR_EINVAL, "null argument");
    for (int i = 0; i < 27; i++) ds27[i] = (double)jsdr::bpsk::kDsFilterF[i];
    for (int i = 0; i < 65; i++) dm65[i] = (double)jsdr::bpsk::kDmFilterF[i];
    return JSDR_OK;
} JSDR_CATCH_ALL

// The exact wrap thresholds the phase scout uses for one tuner increment (scout_thresholds):
// host only, for tests/test_scout_thresholds.py, which checks on the CPU that `p > th1` / `p > th2`
// ARE the reference's comparisons (FUNcubeBPSKDemod.java:385) for every double around them.
extern "C" int jsdr_probe_scout_thresholds(double inc, double *th1, double *th2)
try {
    JSDR_REQUIRE(th1 && th2, JSDR_EINVAL, "null argument");
    JSDR_REQUIRE(inc > 0.0 && inc < 3.1, JSDR_EINVAL, "the pair form covers 0 < inc < 3.1");
    scout_thresholds(inc, *th1, *th2);
    return JSDR_OK;
} JSDR_CATCH_ALL
