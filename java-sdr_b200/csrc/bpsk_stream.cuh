// bpsk_stream.cuh — the streaming form of the FUNcube tuner + decimator
// (FUNcubeBPSKDemod.java:382-397 RxMixTuner, :467-492 RxDownSample) for banks of
// many channels.  Included by bpsk.cu (uses its phase / conversion helpers).
//
// Mapping: one LANE per channel, one WARP per (32 consecutive channels, segment of
// R decimated outputs).  Every lane walks its own channel backwards in time, one
// "period" of D input samples at a time.  A sample is converted and mixed ONCE, in
// registers, and feeds the ceil(NTAPS/D) outputs whose windows contain it ("roles":
// role q of period t is output t-q of the segment and uses taps q*D .. q*D+D-1).
// Walking newest -> oldest makes every output accumulate its taps in the order
// k = 0, 1, .. exactly as RxDownSample does (:479-483), so the binary64 variant is
// bit-identical to the Java arithmetic; at the end of a period the oldest role is
// complete, is scaled (:486) and stored, and the roles rotate.
//
// Memory: raw s16 IQ goes HBM -> registers -> shared memory as whole, aligned
// 128-byte row chunks (32 samples; 8 lanes x 16 B per row, 4 rows per warp
// instruction), one chunk ahead of the arithmetic, into a 64-sample ring per row;
// each lane then reads its own row (odd pitch, no bank conflicts).  Nothing but the decimated output is written back: 4 B in and 16/D B
// out per input sample.  The cos/sin table sits in shared memory in 8 (binary64) or
// 16 (binary32) interleaved copies so that the per-lane lookups never conflict.
//
// Tuner phase: the table index of sample s is the integer part of
// x = tuPhase*256/2pi.  x is carried in 8.56 fixed point, anchored at the scout's
// exact checkpoint (bpsk.cu) and stepped by integer adds.  The reference's rounding
// can move the true value by < 2^-39 over the <= 64 steps from an anchor, so the
// integer part is the reference's index unless x is within 2^-24 of an integer; such
// samples (about one in 2^23), and channels whose increment has no fixed-point form,
// are resolved by replaying the reference's own double arithmetic from the checkpoint.
#pragma once

namespace jsdr {
namespace bpsk {
namespace stream {

constexpr int kWarps = 16;            // s16 input: one CTA per SM (231552 B of shared memory, 128 registers); fewer warps do not help (DESIGN.md §9)
constexpr int kWarpsF32 = 8;          // float input: the ring rows are twice as wide
constexpr int kMaxTaps = 64;
enum { PREC_F64 = 0, PREC_F32 = 1 };

struct Params {
    const void *in;                     // [nchan][chan_stride] s16 IQ pairs (uint32) or float IQ pairs (float2)
    long long chan_stride;
    int S, ic, qc;
    const unsigned long long *tu_dx56;  // [nchan] index step per sample, 8.56 fixed point; 0: exact replay only
    const double *tu_inc;               // [nchan]
    const double *ckpt;                 // [nchunks][nchan] tuPhase before each 32-sample chunk
    int nchan, nchunks;
    const double2 *hist_in;             // [nchan][kMaxDsTaps], entry k is local sample k-H
    const double2 *cossin;              // [257] (cos, sin); entry 256 = (1, 1), the mixer bypass
    int n0, NO, R, nseg, ncw;           // first output's sample, outputs, outputs per segment, segments, channel groups
    int grid;                           // CTAs to launch (host side only)
    int warps_per_cta;                  // kWarps or kWarpsF32 (host side only)
    unsigned *work_counter;             // zeroed before the launch
    double2 *ds_out;
    int max_ds;
    double taps[kMaxTaps];
    float tapsf[kMaxTaps];
};

__device__ __forceinline__ unsigned long long u64_of(float2 a) { return *reinterpret_cast<unsigned long long *>(&a); }
__device__ __forceinline__ float2 f2_of(unsigned long long a) { return *reinterpret_cast<float2 *>(&a); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c)
{   // per-half a*b+c in one FFMA2
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(u64_of(a)), "l"(u64_of(b)), "l"(u64_of(c)));
    return f2_of(r);
}
__device__ __forceinline__ float2 add2(float2 a, float2 b)
{
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(u64_of(a)), "l"(u64_of(b)));
    return f2_of(r);
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b)
{
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(u64_of(a)), "l"(u64_of(b)));
    return f2_of(r);
}

// tuPhase -> x = tuPhase*256/2pi in 8.56 fixed point (mod 256), to within 2^-47
__device__ __forceinline__ unsigned long long phase_to_x56(double ph)
{
    const double hi = __dmul_rn(ph, kIdxScaleHi);
    const double lo = __fma_rn(ph, kIdxScaleLo, __fma_rn(ph, kIdxScaleHi, -hi));
    const unsigned long long x48 = (unsigned long long)(__double2ll_rn(hi * 281474976710656.0) +
                                                        __double2ll_rn(lo * 281474976710656.0));
    return x48 << 8;
}

// The reference's own arithmetic for the D samples s_hi, s_hi-1, .. of one lane:
// replay tuPhase from the checkpoint and leave the table index of sample s_hi-j in
// out[j] (256 = mixer bypass).
__device__ __noinline__ void exact_period_indices(const double *__restrict__ ckpt, double inc, int nchan, int S, int ch,
                                                  int s_hi, int D, uint16_t *out)
{
    for (int j = 0; j < D; j++) out[j] = 0;
    const int s_lo = max(s_hi - D + 1, 0), s_top = min(s_hi, S - 1);
    if (s_top < s_lo) return;
    const int c = s_lo >> 5;
    double ph = ckpt[(size_t)c * nchan + ch];
    for (int s = c << 5; s <= s_top; s++) {
        ph = phase_step(ph, inc);
        if (s >= s_lo) out[s_hi - s] = (uint16_t)tuner_index(ph);
    }
}

template <int PREC>
struct Acc;
template <>
struct Acc<PREC_F64> {
    double i, q;
    __device__ __forceinline__ void zero() { i = 0.0; q = 0.0; }
};
template <>
struct Acc<PREC_F32> {
    float i, q;
    __device__ __forceinline__ void zero() { i = 0.f; q = 0.f; }
};

// The raw element the ring holds: one s16 I/Q pair (IRawHandler bytes) or one float I/Q pair
// (IAudioHandler floats).  A staging piece is 16 bytes (4 or 2 samples), a chunk is 8 pieces
// (128 bytes per row: 32 or 16 samples), so the staging code is the same for both.
template <int FMT> struct Raw;
template <> struct Raw<FMT_S16> { typedef uint32_t type; };
template <> struct Raw<FMT_F32> { typedef float2 type; };
template <int FMT> __host__ __device__ constexpr int raw_words() { return FMT == FMT_S16 ? 1 : 2; }   // 32-bit words per sample
template <int FMT> __host__ __device__ constexpr int piece_samples() { return 4 / raw_words<FMT>(); }
template <int FMT> __host__ __device__ constexpr int chunk_samples() { return 8 * piece_samples<FMT>(); }

constexpr int kRing = 64;                 // samples per row in the ring: two (s16) or four (float) chunks
// The first D (rounded up to 4) positions of the ring are mirrored behind its end, so that a
// period that would wrap can be read at fixed offsets below position p+64 instead.
template <int DD> __host__ __device__ constexpr int mirror_len() { return (DD + 3) & ~3; }
template <int DD> __host__ __device__ constexpr int row_pitch() { return (kRing + mirror_len<DD>()) | 1; }   // odd (samples): no bank conflicts
constexpr int kScratch = 24;              // uint16 per lane for the exact-replay path (>= D)
constexpr int kTabBytes = 257 * 128;      // 8 x double2 or 16 x float2 copies of each of the 257 entries

template <int FMT, int W, int DD>
constexpr size_t smem_bytes()
{
    return (size_t)kTabBytes + (size_t)W * (32 * row_pitch<DD>() * 4 * raw_words<FMT>() + 32 * kScratch * 2);
}

__device__ __forceinline__ double2 lds_d2(unsigned addr)
{
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ float2 lds_f2(unsigned addr)
{
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
    return v;
}

// One period (D samples, newest first) of one lane: table lookups, mix, and the
// multiply-accumulates of the NQ live outputs.  FAST = every sample of the period
// is a sample of this call (not history), the period does not wrap in the ring and
// there is no I/Q correction, so the reads are at fixed offsets below `top`;
// otherwise each sample checks for itself.
template <int FMT, int PREC, int NTAPS, int DD, bool FAST>
__device__ __forceinline__ void period_body(const Params &p, const typename Raw<FMT>::type *myrow,
                                            const unsigned (&taddr)[DD], int s_hi, int ch,
                                            Acc<PREC> (&acc)[(NTAPS + DD - 1) / DD])
{
    typedef typename Raw<FMT>::type raw_t;
    constexpr int NQ = (NTAPS + DD - 1) / DD;
    constexpr int H = NTAPS - 1;
    const int ptop = s_hi & (kRing - 1);
    const raw_t *top = myrow + (ptop >= DD - 1 ? ptop : ptop + kRing);   // wrapping periods read the mirror
#pragma unroll
    for (int j = 0; j < DD; j++) {
        const int s = s_hi - j;
        bool hist = false;
        raw_t rw = raw_t();
        if constexpr (FAST) {
            rw = top[-j];
        } else {
            hist = s < 0;
            if (!hist) rw = myrow[s & (kRing - 1)];
        }
        // f2 = (I, Q) as floats: the s16 values themselves (the 1/32767 comes below), or the floats
        float2 f2;
        if constexpr (FMT == FMT_S16) {
            uint32_t w = rw;
            if constexpr (!FAST)
                w = (((w & 0xffffu) + (unsigned)p.ic) & 0xffffu) | ((((w >> 16) + (unsigned)p.qc) & 0xffffu) << 16);
            w ^= 0x80008000u;          // exact s16 -> float: splice into the mantissa of 2^23
            // (I, Q) as one packed pair: the bias subtraction and the division below are one FADD2 /
            // FMUL2 / FFMA2 each for both halves
            f2 = add2(make_float2(__uint_as_float(__byte_perm(w, 0x4b000000u, 0x7410)),
                                  __uint_as_float(__byte_perm(w, 0x4b000000u, 0x7432))),
                      make_float2(-8421376.0f, -8421376.0f));
        } else {
            f2 = rw;
        }
        const float fi = f2.x, fq = f2.y;
        if constexpr (PREC == PREC_F64) {
            double xi, xq;
            if constexpr (FMT == FMT_S16) {
                // (float)s / 32767f, correctly rounded (JavaAudio.java:283): fma(s, r_hi, s*r_lo), the
                // s16_over_32767 of common.cuh on both halves at once
                const float2 q2 = fma2(f2, make_float2(3.0518509447574615e-05f, 3.0518509447574615e-05f),
                                       mul2(f2, make_float2(2.8422576792141996e-14f, 2.8422576792141996e-14f)));
                xi = (double)q2.x;
                xq = (double)q2.y;
            } else {
                xi = (double)fi;       // :372-373 (double)buf[n*2]
                xq = (double)fq;
            }
            const double2 cs = lds_d2(taddr[j]);
            double mi = __dmul_rn(xi, cs.x);   // :389-390 i*cosTab[ix], q*sinTab[ix]
            double mq = __dmul_rn(xq, cs.y);
            if (!FAST && hist) {
                const int k = s + H;
                double2 hv = make_double2(0.0, 0.0);
                if (k >= 0) hv = p.hist_in[(size_t)ch * kMaxDsTaps + k];
                mi = hv.x;
                mq = hv.y;
            }
#pragma unroll
            for (int q = 0; q < NQ; q++) {
                const int k = j + q * DD;
                if (k < NTAPS) {
                    acc[q].i = __dadd_rn(acc[q].i, __dmul_rn(mi, p.taps[k]));   // :479-483, age order
                    acc[q].q = __dadd_rn(acc[q].q, __dmul_rn(mq, p.taps[k]));
                }
            }
        } else {
            const float2 cs = lds_f2(taddr[j]);
            float mi = fi * cs.x;
            float mq = fq * cs.y;
            if (!FAST && hist) {
                const int k = s + H;
                double2 hv = make_double2(0.0, 0.0);
                if (k >= 0) hv = p.hist_in[(size_t)ch * kMaxDsTaps + k];
                mi = (float)hv.x;
                mq = (float)hv.y;
            }
#pragma unroll
            for (int q = 0; q < NQ; q++) {
                const int k = j + q * DD;
                if (k < NTAPS) {
                    acc[q].i = fmaf(mi, p.tapsf[k], acc[q].i);
                    acc[q].q = fmaf(mq, p.tapsf[k], acc[q].q);
                }
            }
        }
    }
}

template <int FMT, int PREC, int NTAPS, int DD, int W>
__global__ void __launch_bounds__(W * 32, 1) k_mixdecim_stream(const Params p)
{
    typedef typename Raw<FMT>::type raw_t;
    constexpr int NQ = (NTAPS + DD - 1) / DD;          // live outputs per sample
    constexpr int kPitch = row_pitch<DD>();            // samples
    constexpr int MIR = mirror_len<DD>();
    constexpr int SPP = piece_samples<FMT>();          // samples per 16-byte staging piece
    constexpr int CH = chunk_samples<FMT>();           // samples per staged chunk (128 bytes per row)
    constexpr int CHLOG = (CH == 32) ? 5 : 4;
    constexpr int NSLOT = kRing / CH;
    constexpr int WARP_BYTES = 32 * kPitch * (int)sizeof(raw_t) + 32 * kScratch * 2;
    static_assert(DD <= kScratch && DD <= 32, "period");
    static_assert(NTAPS <= kMaxTaps && NQ <= 4, "taps");

    extern __shared__ __align__(16) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // ---- table copies: copy c of entry e at byte e*128 + c*(128/NCOPY)
    if constexpr (PREC == PREC_F64) {
        double2 *tab = reinterpret_cast<double2 *>(smem);
        for (int i = tid; i < 257 * 8; i += W * 32) tab[i] = p.cossin[i >> 3];
    } else {
        float2 *tab = reinterpret_cast<float2 *>(smem);
        // s16 input: the 1/32767 of the conversion (JavaAudio.java:283) is folded into the table
        const double scale = (FMT == FMT_S16) ? 32767.0 : 1.0;
        for (int i = tid; i < 257 * 16; i += W * 32) {
            const double2 cs = p.cossin[i >> 4];
            tab[i] = make_float2((float)(cs.x / scale), (float)(cs.y / scale));
        }
    }
    __syncthreads();
    // shared-window address of this lane's copy of table entry 0 (128-byte aligned base: the index is or-ed in)
    const unsigned lane_tab = (unsigned)__cvta_generic_to_shared(smem) + ((PREC == PREC_F64) ? (lane & 7) * 16 : (lane & 15) * 8);

    raw_t *ring = reinterpret_cast<raw_t *>(smem + kTabBytes + warp * WARP_BYTES);
    uint16_t *scratch = reinterpret_cast<uint16_t *>(smem + kTabBytes + warp * WARP_BYTES + 32 * kPitch * (int)sizeof(raw_t)) + lane * kScratch;
    const raw_t *myrow = ring + lane * kPitch;

    // staging role of this lane: rows 4i + (lane>>3), 16-byte piece (lane&7) of a chunk
    const int srow = lane >> 3, spiece = lane & 7;
    const long long stride4 = 4 * p.chan_stride;       // samples between this lane's consecutive staging rows
    const bool aligned = ((reinterpret_cast<size_t>(p.in) & 15) == 0) && ((p.chan_stride * (long long)sizeof(raw_t)) % 16 == 0);
    const bool iqcorr = FMT == FMT_S16 && (p.ic | p.qc) != 0;

    // warps take (channel group, segment) items from a shared counter: an SM that became free
    // late (the phase scout ran on it) simply takes fewer
    for (;;) {
        int wg = 0;
        if (lane == 0) wg = (int)atomicAdd(p.work_counter, 1u);
        wg = __shfl_sync(0xffffffffu, wg, 0);
        if (wg >= p.ncw * p.nseg) break;
        const int cw = wg % p.ncw, seg = wg / p.ncw;
        const int ch0 = cw * 32;
        const int rows = min(32, p.nchan - ch0);
        const int ch = min(ch0 + lane, p.nchan - 1);
        const bool lane_live = ch0 + lane < p.nchan;
        const int m_top = (seg + 1) * p.R - 1;         // newest output of the segment (may lie beyond NO)
        const int n_top = p.n0 + m_top * DD;           // its newest input sample
        const int nper = p.R + NQ - 1;
        const unsigned long long dx = p.tu_dx56[ch];
        const bool exact_lane = (dx == 0ull);
        const raw_t *stage0 = reinterpret_cast<const raw_t *>(p.in) + (long long)(ch0 + srow) * p.chan_stride + spiece * SPP;

        // ---- staging: chunk c = samples [CH*c, CH*c+CH) of 32 rows -> ring slot c mod NSLOT
        uint4 pre[8];
        auto load_chunk = [&](int c) {
            const int s0 = c * CH + spiece * SPP;
            if (c >= 0 && aligned && c * CH + CH <= p.S && rows == 32) {
                const raw_t *src = stage0 + c * CH;
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    pre[i] = ldg_stream_u4(reinterpret_cast<const uint4 *>(src));
                    src += stride4;
                }
            } else {                                   // block edges, short or unaligned rows
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    const bool rok = c >= 0 && (srow + 4 * i) < rows;
                    const uint32_t *src = reinterpret_cast<const uint32_t *>(stage0 + (long long)i * stride4 + c * CH);
                    uint32_t v[4];
#pragma unroll
                    for (int e = 0; e < 4; e++) {
                        v[e] = 0u;
                        if (rok && s0 + e / raw_words<FMT>() < p.S) v[e] = src[e];
                    }
                    pre[i] = make_uint4(v[0], v[1], v[2], v[3]);
                }
            }
        };
        auto store_chunk = [&](int c) {
            const int pos = (c & (NSLOT - 1)) * CH + spiece * SPP;      // ring position of this lane's piece
            uint32_t *dst = reinterpret_cast<uint32_t *>(ring + srow * kPitch + pos);
            constexpr int RW = 4 * kPitch * raw_words<FMT>();             // words between staging rows of one lane
#pragma unroll
            for (int i = 0; i < 8; i++) {
                if constexpr (FMT == FMT_S16) {
                    dst[i * RW + 0] = pre[i].x;
                    dst[i * RW + 1] = pre[i].y;
                    dst[i * RW + 2] = pre[i].z;
                    dst[i * RW + 3] = pre[i].w;
                } else {
                    uint2 *d2 = reinterpret_cast<uint2 *>(dst + i * RW);
                    d2[0] = make_uint2(pre[i].x, pre[i].y);
                    d2[1] = make_uint2(pre[i].z, pre[i].w);
                }
            }
            // mirror of ring positions 0 .. MIR-1: a branch of its own, so that the chunks that
            // land in the other ring slots (every second one, or three in four) skip it entirely
            if (pos < MIR) {
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    if constexpr (FMT == FMT_S16) {
                        dst[i * RW + kRing + 0] = pre[i].x;
                        dst[i * RW + kRing + 1] = pre[i].y;
                        dst[i * RW + kRing + 2] = pre[i].z;
                        dst[i * RW + kRing + 3] = pre[i].w;
                    } else {
                        uint2 *d2 = reinterpret_cast<uint2 *>(dst + i * RW);
                        d2[kRing + 0] = make_uint2(pre[i].x, pre[i].y);
                        d2[kRing + 1] = make_uint2(pre[i].z, pre[i].w);
                    }
                }
            }
        };

        Acc<PREC> acc[NQ];
#pragma unroll
        for (int q = 0; q < NQ; q++) acc[q].zero();

        // x = tuPhase*256/2pi (8.56 fixed point) of the newest sample of the current period.  It is
        // re-anchored at an exact checkpoint every kReanchor periods and stepped by integer adds
        // in between (at most kReanchor*D + 32 steps from an anchor: drift < 2^-36, guard 2^-24).
        constexpr int kReanchor = 12;
        const unsigned long long dxD = dx * (unsigned long long)DD;
        unsigned long long x_top = 0;
        bool bad_anchor = false;

        int staged_lo = (n_top >> CHLOG) + 1;          // lowest chunk in the ring
        __syncwarp();                                  // (the previous segment's reads are done)
        load_chunk(staged_lo - 1);
        store_chunk(staged_lo - 1);
        staged_lo--;
        load_chunk(staged_lo - 1);
        __syncwarp();

#pragma unroll 1
        for (int tt = 0; tt < nper; tt++) {
            const int s_hi = n_top - tt * DD;          // newest sample of the period (uniform)
            const int s_lo = s_hi - DD + 1;
            while ((s_lo >> CHLOG) < staged_lo) {      // uniform: the period enters the next chunk(s) down
                __syncwarp();                          // (twice in a row only when D > chunk: float input, D = 20)
                store_chunk(staged_lo - 1);
                staged_lo--;
                load_chunk(staged_lo - 1);
                __syncwarp();
            }

            // ---- table addresses of the period's samples
            unsigned taddr[DD];
            {
                if (tt % kReanchor == 0) {             // uniform
                    const int c = min(max(s_hi >> 5, 0), p.nchunks - 1);
                    const double ck = p.ckpt[(size_t)c * p.nchan + ch];
                    x_top = phase_to_x56(ck) + (unsigned long long)((long long)(s_hi - (c << 5) + 1)) * dx;
                    // The index is extrapolated backwards from this anchor over the next kReanchor
                    // periods.  Samples whose phase is <= 0 take the mixer bypass (:395) instead of a
                    // table entry; that only happens while the phase climbs from below zero after a
                    // retune from a negative frequency, so the whole anchor window is clear of it as
                    // soon as the checkpoint of its OLDEST chunk is non-negative (inc > 0: the phase
                    // only grows from there).  Otherwise the lane replays exactly.
                    const int c_lo = min(max((s_hi - kReanchor * DD + 1) >> 5, 0), p.nchunks - 1);
                    const double ck_lo = p.ckpt[(size_t)c_lo * p.nchan + ch];
                    bad_anchor = !(ck >= 0.0) || !(ck_lo >= 0.0);
                }
                // Sample j of the period sits j steps below the top: hi32(x_top - j*dx) lies in
                // [X - j, X] for X = hi32(x_top) - j*hi32(dx) (the low words can borrow at most j), so
                // the index is X's top byte unless X's 24 fraction bits are within j + 1 of an
                // integer -- one multiply-add per sample instead of a 64-bit running difference,
                // and no chain from sample to sample.  `near` lanes replay exactly (about one
                // period in 2^14 per lane).
                const unsigned xt = (unsigned)(x_top >> 32), ndx = 0u - (unsigned)(dx >> 32);
                const unsigned nt = (xt << 8) + 256u, ndx8 = ndx << 8;
                x_top -= dxD;
                bool near = exact_lane || bad_anchor;
#pragma unroll
                for (int j = 0; j < DD; j++) {
                    const unsigned xj = xt + (unsigned)j * ndx;
                    taddr[j] = lane_tab + ((xj >> 17) & 0x7f80u);   // entry (index) of this lane's copy
                    near |= (nt + (unsigned)j * ndx8) <= 256u * (unsigned)(DD + 2);   // fraction in [-1, DD] * 2^-24
                }
                if (__any_sync(0xffffffffu, near)) {
                    if (near) {
                        exact_period_indices(p.ckpt, p.tu_inc[ch], p.nchan, p.S, ch, s_hi, DD, scratch);
#pragma unroll
                        for (int j = 0; j < DD; j++) taddr[j] = lane_tab + ((unsigned)scratch[j] << 7);
                    }
                }
            }

            // ---- convert, mix, accumulate
            if (s_lo >= 0 && !iqcorr) period_body<FMT, PREC, NTAPS, DD, true>(p, myrow, taddr, s_hi, ch, acc);
            else period_body<FMT, PREC, NTAPS, DD, false>(p, myrow, taddr, s_hi, ch, acc);

            // ---- the oldest role is complete: scale (:469,486), store, rotate
            const int r_out = tt - (NQ - 1);
            const int m = m_top - r_out;
            if (r_out >= 0 && m < p.NO && lane_live) {
                double2 o;
                if constexpr (PREC == PREC_F64) {
                    o = make_double2(__dmul_rn(acc[NQ - 1].i, 0.9 * 32768.0), __dmul_rn(acc[NQ - 1].q, 0.9 * 32768.0));
                } else {
                    o = make_double2((double)acc[NQ - 1].i * (0.9 * 32768.0), (double)acc[NQ - 1].q * (0.9 * 32768.0));
                }
                p.ds_out[(size_t)ch * p.max_ds + m] = o;
            }
#pragma unroll
            for (int q = NQ - 1; q > 0; q--) acc[q] = acc[q - 1];
            acc[0].zero();
        }
    }
}

}  // namespace stream
}  // namespace bpsk
}  // namespace jsdr
