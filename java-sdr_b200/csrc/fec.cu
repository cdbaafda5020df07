// fec.cu — the frame stage behind the FUNcube bit stream (SURVEY §8f-1):
//   sync correlator   FUNcubeBPSKDemod.java:553-574  (65-point correlation against
//                     SYNC_VECTOR at stride 80 over the last 5200 bits, >= 45 starts a decode)
//   FECDecode         FECDecoder.java:703-852        (de-interleave 80x65, Viterbi K=7 r=1/2,
//                     de-scramble, 2 x RS(160,128) = CCSDS (255,223) shortened by 95,
//                     re-encode and count channel errors)
// All integer work, bit-exact.  The reference shifts a 5200-byte array per bit (:553); here
// the last 5199 bits of every channel stay on the device and every new bit's correlation
// is an independent thread.  A detected frame is decoded by one warp: the 64-state
// add-compare-select runs one butterfly per lane with the path metrics exchanged by
// shuffles, the decisions of a step are two ballots, lanes 0/1 run the two RS decoders.
//
// Tables: GF(256), scrambler, convolutional-code symbols, RS generator and the sync
// vector are generated from their defining polynomials (FECDecoder.java:40-57,105-181,
// 544-546, 600-605).  The Viterbi metric table (FECDecoder.java:67-100) is a literal in
// the reference, not a formula: it is an INPUT of jsdr_bpsk_enable_fec (the Java shim
// passes the reference's own array).
#include <string.h>

#include <algorithm>
#include <vector>

#include "handles.h"

namespace jsdr {
namespace fec {

constexpr int NN = 255, KK = 223, NROOTS = 32, FCR = 112, PRIM = 11, IPRIM = 116, A0 = 255;
constexpr int RSBLOCKS = 2, RSPAD = 95;
constexpr int NBITS = (256 + NROOTS * RSBLOCKS) * 8 + 6;      // 2566
constexpr int ROWS = 80, COLS = 65;                           // interleaver (FECDecoder "ROWS"=80, "COLUMNS"=65)
constexpr int SYMS = 5200, SYNC_LEN = 65, HIST = SYMS - 1;
constexpr int CPOLYA = 0x4f, CPOLYB = 0x6d, SYNC_POLY = 0x48;

// Generated from their defining polynomials; identical for every bank, so they are written to
// the constant bank once per device and never again (the caller-supplied Viterbi metric table
// lives in per-bank global memory instead: another bank's decode may be running when a bank is
// enabled).
struct Tables {
    uint8_t partab[256];
    uint8_t syms[128];
    uint8_t scrambler[320];
    uint8_t alpha_to[256], index_of[256];
    uint8_t rs_poly[16];
    int8_t sync[SYNC_LEN];        // +1 / -1 (FUNcubeBPSKDemod.SYNC_VECTOR, :79-81)
};

__constant__ Tables c_tab;

static int parity8(int x) { x ^= x >> 4; x ^= x >> 2; x ^= x >> 1; return x & 1; }
__host__ __device__ static inline int mod255(int x)
{
    while (x >= 255) { x -= 255; x = (x >> 8) + (x & 255); }
    return x;
}

static void build_tables(Tables &t)
{
    for (int i = 0; i < 256; i++) t.partab[i] = (uint8_t)parity8(i);
    // symbol pair of encoder state s; the second symbol is inverted (FECDecoder.java:105-114, 564)
    for (int s = 0; s < 128; s++) t.syms[s] = (uint8_t)((parity8(s & CPOLYA) << 1) | (1 - parity8(s & CPOLYB)));
    int sr = 1;                                               // GF(256), x^8+x^7+x^2+x+1 (:145-181)
    for (int i = 0; i < 255; i++) {
        t.alpha_to[i] = (uint8_t)sr;
        t.index_of[sr] = (uint8_t)i;
        sr <<= 1;
        if (sr & 0x100) sr ^= 0x187;
    }
    t.alpha_to[255] = 0;
    t.index_of[0] = A0;
    int st = 0xff;                                            // CCSDS randomiser, x^8+x^7+x^5+x^3+1 (:118-139)
    for (int i = 0; i < 320; i++) {
        int byte = 0;
        for (int b = 0; b < 8; b++) {
            byte = (byte << 1) | ((st >> 7) & 1);
            const int fb = ((st >> 7) ^ (st >> 4) ^ (st >> 2) ^ st) & 1;
            st = ((st << 1) | fb) & 0xff;
        }
        t.scrambler[i] = (uint8_t)byte;
    }
    int g[NROOTS + 1];                                        // RS generator, roots alpha^(PRIM*(FCR+i)) (:544-546)
    memset(g, 0, sizeof(g));
    g[0] = 1;
    int root = FCR * PRIM;
    for (int i = 0; i < NROOTS; i++, root += PRIM) {
        g[i + 1] = 1;
        for (int j = i; j > 0; j--) {
            if (g[j] != 0) g[j] = g[j - 1] ^ t.alpha_to[mod255(t.index_of[g[j]] + root)];
            else g[j] = g[j - 1];
        }
        g[0] = t.alpha_to[mod255(t.index_of[g[0]] + root)];
    }
    for (int j = 0; j < 16; j++) t.rs_poly[j] = t.index_of[g[j + 1]];
    int s7 = 0x7f;                                            // sync LFSR (:600-605)
    for (int i = 0; i < SYNC_LEN; i++) {
        t.sync[i] = (s7 & 64) ? 1 : -1;
        s7 = ((s7 << 1) | t.partab[s7 & SYNC_POLY]) & 0xff;
    }
}

// The systematic RS encoder (:614-655) as a linear map: row i of par is the parity (x^32 * x^(127-i))
// mod g(x) that a single 1 in data byte i of a block leaves, lowest-order parity byte first, so
// the parity of a block is the GF(256) combination of the rows selected by its data bytes.
// Row 127 is g(x) without its leading term; row i-1 is row i advanced by one zero byte.
static void build_rs_parity_map(const Tables &t, uint8_t par[128][NROOTS])
{
    uint8_t g[NROOTS + 1];                                    // g[k], k = 1..32: palindromic, monic
    for (int k = 1; k <= 16; k++) g[k] = t.alpha_to[t.rs_poly[k - 1]];
    for (int k = 17; k < NROOTS; k++) g[k] = g[NROOTS - k];
    g[NROOTS] = 1;
    auto gmul = [&](int a, int b) { return (a && b) ? t.alpha_to[mod255(t.index_of[a] + t.index_of[b])] : 0; };
    uint8_t reg[NROOTS];
    for (int k = 0; k < NROOTS; k++) reg[k] = g[k + 1];
    for (int i = 127; i >= 0; i--) {
        memcpy(par[i], reg, NROOTS);
        const int fb = reg[0];
        for (int k = 0; k < NROOTS - 1; k++) reg[k] = (uint8_t)(reg[k + 1] ^ gmul(fb, g[k + 1]));
        reg[NROOTS - 1] = (uint8_t)fb;
    }
}

// ------------------------------------------------------------------ sync correlator
struct FrameMeta {
    int chan;
    int corr;
    long long bit_index;      // cntBit of the bit that completed the frame
    int start;                // position of the frame's first bit in the channel's (history ++ new bits) sequence
    int errors;               // FECDecode's return: channel errors, or -1
};

// the bit sequence of one channel as the correlator sees it: 5199 old bits, then this call's
__device__ __forceinline__ int seq_bit(const int8_t *__restrict__ hist, const int8_t *__restrict__ bits, int pos)
{
    return pos < HIST ? hist[pos] : bits[pos - HIST];
}

// :556-562 for every new bit of every channel: one thread each
__global__ void __launch_bounds__(256) k_sync(const int8_t *__restrict__ hist, const int8_t *__restrict__ bits,
                                              const int32_t *__restrict__ nbits, int max_bits, int nchan,
                                              const long long *__restrict__ cnt_bit_after, int ts_stride_ll,
                                              FrameMeta *__restrict__ frames, int *__restrict__ nframes, int max_frames,
                                              long long *__restrict__ cnt_fec)
{
    const int ch = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int nb = min(nbits[ch], max_bits);
    if (i >= nb) return;
    const int8_t *h = hist + (size_t)ch * HIST;
    const int8_t *b = bits + (size_t)ch * max_bits;
    int corr = 0;
#pragma unroll 5
    for (int n = 0; n < SYNC_LEN; n++) corr += seq_bit(h, b, i + 80 * n) * c_tab.sync[n];
    if (corr >= 45) {
        atomicAdd((unsigned long long *)&cnt_fec[ch], 1ull);
        const int slot = atomicAdd(nframes, 1);
        if (slot < max_frames) {
            FrameMeta m;
            m.chan = ch;
            m.corr = corr;
            m.bit_index = cnt_bit_after[(size_t)ch * ts_stride_ll] - nb + i;
            m.start = i;
            m.errors = -2;
            frames[slot] = m;
        }
    }
}

// new history = the last 5199 bits of (history ++ new bits)
__global__ void __launch_bounds__(256) k_sync_shift(const int8_t *__restrict__ hist_in, int8_t *__restrict__ hist_out,
                                                    const int8_t *__restrict__ bits, const int32_t *__restrict__ nbits,
                                                    int max_bits)
{
    const int ch = blockIdx.y;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= HIST) return;
    const int nb = min(nbits[ch], max_bits);
    hist_out[(size_t)ch * HIST + k] = (int8_t)seq_bit(hist_in + (size_t)ch * HIST, bits + (size_t)ch * max_bits, k + nb);
}

// ------------------------------------------------------------------ FECDecode, one warp per frame
struct RsScratch {
    uint8_t syn[NROOTS];          // S_i
    uint8_t lam[NROOTS + 1];      // lambda coefficients (values)
    uint8_t om[NROOTS];           // omega coefficients
    uint8_t root[NROOTS], loc[NROOTS];
};

struct DecodeSmem {
    uint8_t raw[SYMS];                       // dmFECBits: 0xc0 / 0x40 (:564-566)
    uint8_t symbols[NBITS * 2 + 65 + 3];     // de-interleaved
    unsigned dec[NBITS][2];                  // decisions of states 2b (even) and 2b+1 (odd), bit b
    uint8_t vit[(NBITS - 6) / 8];
    uint8_t rs[RSBLOCKS][NN + 1];
    uint8_t out[256];
    uint8_t enc[324];                        // the 320 scrambled bytes the convolutional encoder sees, then zeros
    int16_t mettab[2][256];                  // FECDecoder.java:67-100, the caller's copy (per bank)
    uint8_t gf_exp2[512], gf_lg[256];
    RsScratch rsw;
    int rserr[RSBLOCKS];
};

// ---- GF(256) arithmetic on shared-memory tables (lane-divergent look-ups; the constant bank
// would serialise them).  exp2[i] = alpha^i for i < 510 (two periods, so that the sum of two
// logarithms needs no reduction), lg[v] = log_alpha v, lg[0] unused.
struct GF {
    const uint8_t *exp2, *lg;
    __device__ __forceinline__ int mul(int a, int b) const { return (a && b) ? exp2[lg[a] + lg[b]] : 0; }
    __device__ __forceinline__ int mul_exp(int a, int e) const { return a ? exp2[lg[a] + e] : 0; }   // a * alpha^e, e < 255
    __device__ __forceinline__ int div(int a, int b) const { return a ? exp2[lg[a] + 255 - lg[b]] : 0; }   // b != 0
};

// RS(255,223) over GF(256), CCSDS roots alpha^(11*(112+i)), errors only — the whole warp decodes
// one code word (FECDecoder.java:325-519 is the reference's sequential form of the same
// mathematics; nothing of its structure is kept):
//   syndromes        lane i evaluates the word at root i (Horner over the 160 stored symbols)
//   Berlekamp-Massey lane l holds the coefficient lambda[l+1] and b[l]; the discrepancy is one
//                    warp XOR-reduction, x*b(x) and lambda(x)/d are one shuffle
//   root search      lane-parallel over the 255 field elements, roots compacted by ballot
//   error values     lane i builds omega[i]; lane j evaluates Forney's quotient for root j
// Returns what the reference returns: 0 for a clean word, the number of roots when
// deg(lambda) roots were found and every derivative is non-zero, -1 otherwise.  The
// Berlekamp-Massey recurrence is the textbook one the reference also runs, so lambda — and
// with it the outcome for words with more than 16 errors — is the same polynomial.
__device__ int rs_decode_warp(uint8_t *cw, RsScratch &R, const GF gf, int lane)
{
    const unsigned FULL = 0xffffffffu;
    // ---- syndromes: S_i = cw(beta_i), beta_i = alpha^(PRIM*(FCR+i)); the 95 pad symbols are zero
    {
        const int be = ((FCR + lane) * PRIM) % NN;
        int s = 0;
        for (int j = RSPAD; j < NN; j++) s = cw[j] ^ gf.mul_exp(s, be);
        R.syn[lane] = (uint8_t)s;
        if (__ballot_sync(FULL, s != 0) == 0u) return 0;
    }
    __syncwarp();
    // ---- Berlekamp-Massey.  lambda(x) = 1 + sum lam_l x^(l+1); b(x) = sum bq_l x^l
    int lam = 0, bq = (lane == 0) ? 1 : 0, L = 0;
    for (int r = 1; r <= NROOTS; r++) {
        // discrepancy d = S[r-1] + sum_{i=1}^{r-1} lambda[i] S[r-1-i]
        const int term = (lane <= r - 2) ? gf.mul(lam, R.syn[r - 2 - lane]) : 0;
        const int d = __reduce_xor_sync(FULL, (unsigned)term) ^ R.syn[r - 1];
        int b_up = __shfl_up_sync(FULL, bq, 1);              // x * b(x)
        if (lane == 0) b_up = 0;
        if (d == 0) {
            bq = b_up;
        } else {
            int l_up = __shfl_up_sync(FULL, lam, 1);         // coefficient `lane` of the old lambda
            if (lane == 0) l_up = 1;
            const int lam_new = lam ^ gf.mul(d, bq);         // lambda - d * x * b
            if (2 * L <= r - 1) {
                L = r - L;
                bq = gf.div(l_up, d);                        // b = old lambda / d
            } else {
                bq = b_up;
            }
            lam = lam_new;
        }
    }
    const unsigned nz = __ballot_sync(FULL, lam != 0);
    const int deg = nz ? 32 - __clz(nz) : 0;                  // highest non-zero coefficient
    R.lam[lane + 1] = (uint8_t)lam;
    if (lane == 0) R.lam[0] = 1;
    __syncwarp();
    // ---- roots of lambda among alpha^i, i = 1..255; error location of root i is (IPRIM*i - 1) mod 255
    int count = 0;
    for (int t = 0; t < 8; t++) {
        const int i = 32 * t + lane + 1;
        int q = 1;
        if (i <= NN) {
            for (int j = 1; j <= deg; j++) q ^= gf.mul_exp(R.lam[j], (j * i) % NN);
        }
        const bool hit = (i <= NN) && (q == 0);
        const unsigned m = __ballot_sync(FULL, hit);
        if (hit) {
            const int pos = count + __popc(m & ((1u << lane) - 1u));
            if (pos < NROOTS) {
                R.root[pos] = (uint8_t)i;
                R.loc[pos] = (uint8_t)((IPRIM * i - 1) % NN);
            }
        }
        count += __popc(m);
    }
    if (count != deg) return -1;
    // ---- omega(x) = S(x) lambda(x) mod x^32
    {
        int om = 0;
        const int jm = min(deg, lane);
        for (int j = 0; j <= jm; j++) om ^= gf.mul(R.syn[lane - j], R.lam[j]);
        R.om[lane] = (uint8_t)om;
    }
    __syncwarp();
    // ---- error values (Forney): lane j corrects location loc[j]
    bool bad = false;
    if (lane < count) {
        const int rt = R.root[lane];
        int num1 = 0;
        for (int i = 0; i < NROOTS; i++) num1 ^= gf.mul_exp(R.om[i], (i * rt) % NN);
        int den = 0;                                          // lambda'(x) keeps the odd coefficients
        for (int i = 0; i <= (min(deg, NROOTS - 1) & ~1); i += 2) den ^= gf.mul_exp(R.lam[i + 1], (i * rt) % NN);
        if (den == 0) {
            bad = true;
        } else if (num1 != 0) {
            const int num2e = (rt * (FCR - 1)) % NN;          // alpha^(root*(FCR-1))
            cw[R.loc[lane]] ^= (uint8_t)gf.div(gf.mul_exp(num1, num2e), den);
        }
    }
    if (__any_sync(FULL, bad)) return -1;
    __syncwarp();
    return count;
}

// Re-encoding for the channel-error count (FECDecoder.java:831-847 calls encode_FEC40, :527-688),
// without building the 5200-symbol frame: the encoder is a fixed map from the 320 scrambled
// bytes to frame positions, so every lane compares its own positions directly.
//   RS parity   the systematic encoder is GF-linear: parity byte k of a block is the dot
//               product of its 128 data bytes with column k of rs_par (x^(32+127-i) mod g(x),
//               built on the host) — lane k owns parity byte k, no shift register
//   symbols     frame position p = row*80 + col holds sync bit `row` in column 0 and otherwise
//               encoder output number col*65 + row - 65: symbol (n & 1) of input bit n >> 1,
//               a parity of the 7-bit window that ends at that bit
__device__ int reencode_count_errors(const uint8_t *out, const uint8_t *raw, uint8_t *enc /* 322 */,
                                     const uint8_t *__restrict__ rs_par, const GF gf, int lane)
{
    for (int r = 0; r < RSBLOCKS; r++) {
        int par = 0;
        for (int i = 0; i < 128; i++) par ^= gf.mul(out[2 * i + r], rs_par[i * NROOTS + lane]);
        enc[256 + 2 * lane + r] = (uint8_t)(par ^ c_tab.scrambler[256 + 2 * lane + r]);
    }
    for (int i = lane; i < 256; i += 32) enc[i] = out[i] ^ c_tab.scrambler[i];
    if (lane < 2) enc[320 + lane] = 0;                        // the six flush bits (:670)
    __syncwarp();
    int errors = 0;
    for (int p = lane; p < SYMS; p += 32) {
        const int row = p / ROWS, col = p - row * ROWS;
        int sym = 0;
        if (col == 0) {
            sym = c_tab.sync[row] > 0;
        } else {
            const int k = col * COLS + row - COLS;            // encoder output number
            if (k < 2 * NBITS) {
                const int n = k >> 1, byte = n >> 3;
                const int two = ((byte ? enc[byte - 1] : 0) << 8) | enc[byte];
                const int win = (two >> (7 - (n & 7))) & 0x7f;   // input bits n-6 .. n, newest lowest
                sym = (k & 1) ? 1 - (__popc(win & CPOLYB) & 1) : (__popc(win & CPOLYA) & 1);
            }
        }
        errors += (sym != (raw[p] >> 7));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) errors += __shfl_xor_sync(0xffffffffu, errors, o);
    return errors;
}

__global__ void __launch_bounds__(32) k_fec_decode(const int8_t *__restrict__ hist, const int8_t *__restrict__ bits,
                                                   int max_bits, FrameMeta *__restrict__ frames,
                                                   const int *__restrict__ nframes, int max_frames,
                                                   uint8_t *__restrict__ data_out, long long *__restrict__ cnt_dec,
                                                   const int16_t *__restrict__ mettab, const uint8_t *__restrict__ rs_par)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DecodeSmem &S = *reinterpret_cast<DecodeSmem *>(smem_raw);
    const int slot = blockIdx.x, lane = threadIdx.x;
    if (slot >= min(*nframes, max_frames)) return;
    const FrameMeta m = frames[slot];
    for (int i = lane; i < 512; i += 32) {
        S.gf_exp2[i] = c_tab.alpha_to[i < NN ? i : (i < 2 * NN ? i - NN : 0)];
        (&S.mettab[0][0])[i] = mettab[i];
    }
    for (int i = lane; i < 256; i += 32) S.gf_lg[i] = c_tab.index_of[i];
    const GF gf = {S.gf_exp2, S.gf_lg};
    const int8_t *h = hist + (size_t)m.chan * HIST;
    const int8_t *b = bits + (size_t)m.chan * max_bits;
    // :564-566 dmFECBits[n] = dmFECCorr[n]==1 ? 0xc0 : 0x40
    for (int n = lane; n < SYMS; n += 32) S.raw[n] = (seq_bit(h, b, m.start + n) == 1) ? 0xc0 : 0x40;
    for (int n = lane; n < (int)sizeof(S.symbols); n += 32) S.symbols[n] = 0;
    __syncwarp();
    // :707-723 de-interleave, skipping the sync column: symbols[(col-1)*65 + row] = raw[row*80 + col]
    for (int n = lane; n < (ROWS - 1) * COLS; n += 32) {
        const int col = 1 + n / COLS, row = n % COLS;
        S.symbols[n] = S.raw[row * ROWS + col];
    }
    __syncwarp();

    // ---- viterbi27 (:203-278).  Lane b owns butterfly b: predecessors b and b+32, successors 2b, 2b+1.
    {
        int lo = (lane == 0) ? 0 : -999999, hi = -999999;     // cmetric[b], cmetric[b+32]
        const int sym_e = c_tab.syms[2 * lane], sym_o = c_tab.syms[2 * lane + 1];
        for (int bit = 0; bit < NBITS; bit++) {
            const int s0 = S.symbols[2 * bit], s1 = S.symbols[2 * bit + 1];
            int mets[4];
#pragma unroll
            for (int i = 0; i < 4; i++) mets[i] = S.mettab[(i >> 1) & 1][s0] + S.mettab[i & 1][s1];
            int b1 = mets[sym_e];
            const int b2 = mets[sym_o];
            int m0 = lo + b1;                                  // nmetric[2b] candidates
            int m1 = hi + b2;
            b1 -= b2;
            const bool d_e = m1 > m0;
            const int n_e = d_e ? m1 : m0;
            m0 -= b1;                                          // nmetric[2b+1] candidates
            m1 += b1;
            const bool d_o = m1 > m0;
            const int n_o = d_o ? m1 : m0;
            const unsigned be = __ballot_sync(0xffffffffu, d_e), bo = __ballot_sync(0xffffffffu, d_o);
            if (lane == 0) {
                S.dec[bit][0] = be;
                S.dec[bit][1] = bo;
            }
            // next step: cmetric[b] = nmetric[b] (lane b>>1, even/odd), cmetric[b+32] = nmetric[b+32] (lane 16 + (b>>1))
            const int src_lo = lane >> 1, src_hi = 16 + (lane >> 1);
            const int e_lo = __shfl_sync(0xffffffffu, n_e, src_lo), o_lo = __shfl_sync(0xffffffffu, n_o, src_lo);
            const int e_hi = __shfl_sync(0xffffffffu, n_e, src_hi), o_hi = __shfl_sync(0xffffffffu, n_o, src_hi);
            lo = (lane & 1) ? o_lo : e_lo;
            hi = (lane & 1) ? o_hi : e_hi;
        }
    }
    __syncwarp();
    for (int i = lane; i < (NBITS - 6) / 8; i += 32) S.vit[i] = 0;
    __syncwarp();
    if (lane == 0) {                                           // trace back from state 0 (:262-277)
        int state = 0;
        for (int i = NBITS - 7, bit = NBITS - 1; i >= 0; i--, bit--) {
            // decision of `state` at step `bit`: state = 2b + e
            const unsigned w = S.dec[bit][state & 1];
            if ((w >> (state >> 1)) & 1u) {
                state |= 64;
                S.vit[i >> 3] |= (uint8_t)(0x80 >> (i & 7));
            }
            state >>= 1;
        }
    }
    __syncwarp();
    // ---- de-scramble into the two RS code blocks (:762-771)
    for (int n = lane; n < RSBLOCKS * (NN + 1); n += 32) (&S.rs[0][0])[n] = 0;
    __syncwarp();
    for (int n = lane; n < (NN - RSPAD) * RSBLOCKS; n += 32) {
        const int col = RSPAD + n / RSBLOCKS, row = n % RSBLOCKS;
        S.rs[row][col] = S.vit[n] ^ c_tab.scrambler[n];
    }
    __syncwarp();
    int rserr[RSBLOCKS];
    for (int r = 0; r < RSBLOCKS; r++) {                                // :774-777, the warp decodes one word at a time
        rserr[r] = rs_decode_warp(S.rs[r], S.rsw, gf, lane);
        __syncwarp();
    }
    int rc = (rserr[0] == -1 || rserr[1] == -1) ? -1 : 0;
    if (rc == 0) {
        for (int j = lane; j < 256; j += 32) S.out[j] = S.rs[j % RSBLOCKS][RSPAD + j / RSBLOCKS];   // :783-789
        __syncwarp();
        rc = reencode_count_errors(S.out, S.raw, S.enc, rs_par, gf, lane);   // :831-847
        for (int j = lane; j < 256; j += 32) data_out[(size_t)slot * 256 + j] = S.out[j];
        if (lane == 0) atomicAdd((unsigned long long *)&cnt_dec[m.chan], 1ull);
    } else {
        for (int j = lane; j < 256; j += 32) data_out[(size_t)slot * 256 + j] = 0;
    }
    if (lane == 0) frames[slot].errors = rc;
}

}  // namespace fec
}  // namespace jsdr

// =========================================================================== host
using namespace jsdr;

struct jsdr_fec_state {
    int max_frames = 0;                       // frame slots on the device (>= what the caller asked for)
    DevBuf<int16_t> d_mettab;                 // [2][256], this bank's copy of the caller's metric table
    DevBuf<int8_t> d_hist[2];                 // [nchan][5199]
    int cur = 0;
    DevBuf<fec::FrameMeta> d_frames;
    DevBuf<int> d_nframes;
    const uint8_t *d_rs_par = nullptr;        // [128][32] parity map (per device, shared)
    DevBuf<uint8_t> d_data;                   // [max_frames][256]
    DevBuf<long long> d_cnt;                  // [2][nchan] cntFEC, cntDec (:567,571)
};

void jsdr_fec_delete::operator()(jsdr_fec_state *f) const { delete f; }

extern "C" int jsdr_bpsk_enable_fec(jsdr_bpsk *b, const int16_t *mettab, int max_frames)
try {
    JSDR_REQUIRE(b && mettab && max_frames > 0, JSDR_EINVAL, "bad argument");
    jsdr_ctx *ctx = b->ctx;
    JSDR_TRY(ctx->bind());
    // generated tables and the parity map: once per device, then read-only
    static PerDeviceFlag tables_done;
    static uint8_t *d_rs_par[64] = {nullptr};
    JSDR_TRY(tables_done.once(ctx->device, [&]() -> int {
        fec::Tables t;
        fec::build_tables(t);
        JSDR_CUDA(cudaMemcpyToSymbol(fec::c_tab, &t, sizeof(t)));
        uint8_t par[128][fec::NROOTS];
        fec::build_rs_parity_map(t, par);
        if (!d_rs_par[ctx->device & 63]) JSDR_CUDA(cudaMalloc(&d_rs_par[ctx->device & 63], sizeof(par)));
        JSDR_CUDA(cudaMemcpy(d_rs_par[ctx->device & 63], par, sizeof(par), cudaMemcpyHostToDevice));
        JSDR_CUDA(cudaDeviceSynchronize());        // tables are in place before anyone's kernel reads them
        return JSDR_OK;
    }));
    if (b->fec) {                                               // metric table refreshed, state kept: behind this bank's own work
        JSDR_CUDA(cudaMemcpyAsync(b->fec->d_mettab.get(), mettab, 512 * sizeof(int16_t), cudaMemcpyHostToDevice, ctx->aux));
        JSDR_CUDA(cudaStreamSynchronize(ctx->aux));
        return JSDR_OK;
    }
    const char *what = "jsdr_bpsk_enable_fec";
    std::unique_ptr<jsdr_fec_state, jsdr_fec_delete> f(new jsdr_fec_state());
    // Every detection of a call is decoded (cntDec must follow cntFEC as in :563-571): a channel
    // can complete at most one frame per 5200 bits of signal, so nchan * (max_bits/5200 + 2)
    // slots cover everything but a correlator firing on noise more than twice per frame time.
    f->max_frames = std::max(max_frames, b->nchan * (b->max_bits / fec::SYMS + 2));
    f->d_rs_par = d_rs_par[ctx->device & 63];
    max_frames = f->max_frames;
    const size_t nc = (size_t)b->nchan;
    JSDR_TRY(f->d_hist[0].alloc_zeroed(nc * fec::HIST, ctx->stream, what));      // dmFECCorr starts as zeros (:503)
    JSDR_TRY(f->d_hist[1].alloc(nc * fec::HIST, what));
    JSDR_TRY(f->d_frames.alloc(sizeof(fec::FrameMeta) * (size_t)max_frames, what));
    JSDR_TRY(f->d_nframes.alloc_zeroed(sizeof(int), ctx->stream, what));
    JSDR_TRY(f->d_data.alloc((size_t)max_frames * 256, what));
    JSDR_TRY(f->d_cnt.alloc_zeroed(sizeof(long long) * 2 * nc, ctx->stream, what));
    JSDR_TRY(f->d_mettab.alloc(512 * sizeof(int16_t), what));
    JSDR_CUDA(cudaMemcpy(f->d_mettab.get(), mettab, 512 * sizeof(int16_t), cudaMemcpyHostToDevice));
    JSDR_CUDA(cudaStreamSynchronize(ctx->stream));            // the stage itself runs on the auxiliary stream
    b->fec = std::move(f);
    return JSDR_OK;
} JSDR_CATCH_ALL

// called by bpsk_receive after the bit-timing stage; like that stage it runs on the auxiliary stream
int jsdr_fec_after_bits(jsdr_bpsk *b)
{
    jsdr_fec_state *f = b->fec.get();
    jsdr_ctx *ctx = b->ctx;
    const int nchan = b->nchan, max_bits = b->max_bits;
    int8_t *const bits = b->stage.d_bits.get();
    int8_t *const hist = f->d_hist[f->cur].get(), *const hist_next = f->d_hist[f->cur ^ 1].get();
    int32_t *const nbits = b->d_nbits.get();
    JSDR_CUDA(cudaMemsetAsync(f->d_nframes.get(), 0, sizeof(int), ctx->aux));
    if (max_bits > 0) {
        dim3 grid((max_bits + 255) / 256, nchan);
        // cntBit lives at the end of each TimingState
        const long long *cnt_bit = reinterpret_cast<const long long *>(
            reinterpret_cast<const char *>(b->d_ts.get()) + offsetof(jsdr::bpsk::TimingState, cntBit));
        ProfScope prof(ctx, JSDR_K_SYNC, ctx->aux);
        fec::k_sync<<<grid, 256, 0, ctx->aux>>>(hist, bits, nbits, max_bits, nchan, cnt_bit,
                                                   (int)(sizeof(jsdr::bpsk::TimingState) / sizeof(long long)), f->d_frames.get(),
                                                   f->d_nframes.get(), f->max_frames, f->d_cnt.get());
        JSDR_TRY(launched(ctx, "k_sync"));
    }
    const size_t smem = sizeof(fec::DecodeSmem);
    static PerDeviceFlag attr_done;
    JSDR_TRY(attr_done.once(ctx->device, [&]() -> int {
        JSDR_CUDA(cudaFuncSetAttribute(fec::k_fec_decode, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        return JSDR_OK;
    }));
    {
        ProfScope prof(ctx, JSDR_K_FEC, ctx->aux);
        fec::k_fec_decode<<<f->max_frames, 32, smem, ctx->aux>>>(hist, bits, max_bits, f->d_frames.get(),
                                                                   f->d_nframes.get(), f->max_frames, f->d_data.get(),
                                                                   f->d_cnt.get() + nchan, f->d_mettab.get(), f->d_rs_par);
        JSDR_TRY(launched(ctx, "k_fec_decode"));
    }
    dim3 g2((fec::HIST + 255) / 256, nchan);
    fec::k_sync_shift<<<g2, 256, 0, ctx->aux>>>(hist, hist_next, bits, nbits, max_bits);
    JSDR_TRY(launched(ctx, "k_sync_shift"));
    f->cur ^= 1;
    return JSDR_OK;
}

extern "C" int jsdr_bpsk_read_frames(jsdr_bpsk *b, int32_t *nframes, int32_t *chan, int64_t *bit_index,
                                     int32_t *errors, uint8_t *data, int max_frames)
try {
    JSDR_REQUIRE(b && nframes, JSDR_EINVAL, "null argument");
    JSDR_REQUIRE(b->fec, JSDR_ESTATE, "jsdr_bpsk_enable_fec has not been called");
    jsdr_fec_state *f = b->fec.get();
    jsdr_ctx *ctx = b->ctx;
    JSDR_TRY(ctx->bind());
    int n = 0;
    JSDR_CUDA(cudaMemcpyAsync(&n, f->d_nframes.get(), sizeof(int), cudaMemcpyDeviceToHost, ctx->aux));
    JSDR_CUDA(cudaStreamSynchronize(ctx->aux));
    const int have = std::min(n, f->max_frames);
    std::vector<fec::FrameMeta> meta(have);
    std::vector<uint8_t> dat((size_t)have * 256);
    if (have > 0) {
        JSDR_CUDA(cudaMemcpyAsync(meta.data(), f->d_frames.get(), sizeof(fec::FrameMeta) * have, cudaMemcpyDeviceToHost, ctx->aux));
        JSDR_CUDA(cudaMemcpyAsync(dat.data(), f->d_data.get(), (size_t)have * 256, cudaMemcpyDeviceToHost, ctx->aux));
        JSDR_CUDA(cudaStreamSynchronize(ctx->aux));
    }
    // detection order on the device is not deterministic: report by (channel, bit)
    std::vector<int> order(have);
    for (int i = 0; i < have; i++) order[i] = i;
    std::sort(order.begin(), order.end(), [&](int x, int y) {
        if (meta[x].chan != meta[y].chan) return meta[x].chan < meta[y].chan;
        return meta[x].bit_index < meta[y].bit_index;
    });
    const int give = std::min(have, std::max(max_frames, 0));
    for (int i = 0; i < give; i++) {
        const fec::FrameMeta &m = meta[order[i]];
        if (chan) chan[i] = m.chan;
        if (bit_index) bit_index[i] = m.bit_index;
        if (errors) errors[i] = m.errors;
        if (data) memcpy(data + (size_t)i * 256, dat.data() + (size_t)order[i] * 256, 256);
    }
    *nframes = n;                                               // detections this call (may exceed what fitted)
    return JSDR_OK;
} JSDR_CATCH_ALL

extern "C" int jsdr_bpsk_read_fec_counters(jsdr_bpsk *b, int64_t *cnt_fec, int64_t *cnt_dec)
try {
    JSDR_REQUIRE(b && cnt_fec && cnt_dec, JSDR_EINVAL, "null argument");
    JSDR_REQUIRE(b->fec, JSDR_ESTATE, "jsdr_bpsk_enable_fec has not been called");
    jsdr_ctx *ctx = b->ctx;
    JSDR_TRY(ctx->bind());
    const size_t nc = (size_t)b->nchan;
    JSDR_CUDA(cudaMemcpyAsync(cnt_fec, b->fec->d_cnt.get(), sizeof(long long) * nc, cudaMemcpyDeviceToHost, ctx->aux));
    JSDR_CUDA(cudaMemcpyAsync(cnt_dec, b->fec->d_cnt.get() + nc, sizeof(long long) * nc, cudaMemcpyDeviceToHost, ctx->aux));
    JSDR_CUDA(cudaStreamSynchronize(ctx->aux));
    return JSDR_OK;
} JSDR_CATCH_ALL

// ---- the tables this library builds for itself, for the reference-pinning tests (host only, no
// device needed): tests/test_ref_tables.py compares every entry with the literals of
// FECDecoder.java:40-57,105-181,544-546 and FUNcubeBPSKDemod.java:79-81.
extern "C" int jsdr_probe_table(int which, int32_t *out, int n)
try {
    JSDR_REQUIRE(out && n >= 0, JSDR_EINVAL, "null argument");
    fec::Tables t;
    fec::build_tables(t);
    const int sizes[] = {256, 128, 320, 256, 256, 16, fec::SYNC_LEN};
    JSDR_REQUIRE(which >= 0 && which < 7 && n <= sizes[which], JSDR_EINVAL, "no such table or too many entries");
    for (int i = 0; i < n; i++) {
        switch (which) {
        case 0: out[i] = t.partab[i]; break;
        case 1: out[i] = t.syms[i]; break;
        case 2: out[i] = t.scrambler[i]; break;
        case 3: out[i] = t.alpha_to[i]; break;
        case 4: out[i] = t.index_of[i]; break;
        case 5: out[i] = t.rs_poly[i]; break;
        default: out[i] = t.sync[i]; break;
        }
    }
    return JSDR_OK;
} JSDR_CATCH_ALL
