// handles.h — the opaque handle types behind include/jsdrcuda.h.
#pragma once

#include <stddef.h>
#include <stdint.h>

#include <vector>

#include "common.cuh"

struct jsdr_fft {
    jsdr_ctx *ctx = nullptr;
    int n = 0, rate = 0, max_batch = 0;
    void *launch = nullptr;          // jsdr::fft::launch_fn of the plan
    float2 *d_tw = nullptr;          // exp(-2*pi*i*t/n)
    float2 *d_work[2] = {nullptr, nullptr};   // workspace of the four-step / staged paths (no single-CTA plan)
    unsigned long long *d_best = nullptr;     // [max_batch] packed block maxima (four-step path)
    int fs_n1 = 0;                            // four-step factor N1 (128 or 256), 0 otherwise
    int split = 0;                            // 2: split plan — two n/2-point transforms per block (fft_kernel SPLIT)
    float2 *d_tw2 = nullptr;                  // split plan: exp(-2*pi*i*c/n), c in [0, n/2)
    unsigned *d_cnt = nullptr;                // split plan: halves reported per block (zero between launches)
    // staging for host-pointer calls (allocated on first use)
    void *d_in = nullptr;
    float *d_out = nullptr;
    int32_t *d_peak = nullptr;
    size_t in_cap = 0, out_cap = 0;
    int32_t *d_pix = nullptr;        // pixel rows of jsdr_pump_waterfall_s16's host path
    size_t pix_cap = 0;
};

namespace jsdr {
namespace bpsk {

// per-channel state of the bit-timing state machine (FUNcubeBPSKDemod.java:497-502)
struct TimingState {
    double dmEnergy[8];
    double dmEnergyOut;
    double lastI, lastQ;
    int bitPos, peakPos, newPeak, pad;
    long long cntBit;
};

// per-channel state of the auto-tune search (FUNcubeBPSKDemod.java:403-405)
struct AutoTuneState {
    double avePeakPower, aveCentreBin;
    int centreBin, pad;
};

enum { FMT_F32 = 0, FMT_S16 = 1 };   // input: (float I, float Q) or s16le (I, Q) pairs
struct ScoutChan;                    // bpsk.cu
constexpr int kMaxDsTaps = 128;
constexpr int kDmTaps = 65;          // MATCHED_FILTER_SIZE

}  // namespace bpsk
}  // namespace jsdr

struct jsdr_fec_state;   // fec.cu
int jsdr_launch_waterfall(jsdr_ctx *ctx, const float *d_psd, int n, int rows, int width, uint32_t peak_rgb,
                          int32_t *d_pix, cudaStream_t st);   // demod_fir.cu

struct jsdr_bpsk {
    jsdr_ctx *ctx = nullptr;
    jsdr_fec_state *fec = nullptr;   // sync correlator + FEC stage, when enabled
    int rate = 0, D = 0, nchan = 0, max_block = 0, stages = 3;
    int ntaps = 27;
    int max_ds = 0, max_words = 0, max_bits = 0;
    std::vector<double> h_tuning;

    double *d_taps = nullptr;        // [kMaxDsTaps] decimator low-pass
    double *d_dmtaps = nullptr;      // [65] matched filter
    double *d_cossin = nullptr;      // cosTab[256] then sinTab[256]
    double2 *d_cossin2 = nullptr;    // (cos, sin) pairs, plus entry 256 = (1, 1) for the mixer bypass

    double *d_tu_inc = nullptr;      // [nchan] tuPhaseInc
    jsdr::bpsk::ScoutChan *d_tu_par = nullptr;   // [nchan] increment and exact wrap thresholds (phase scout)
    unsigned long long *d_tu_dx = nullptr;   // [nchan] table-index step per sample, 8.48 fixed point
    unsigned long long *d_tu_dx56 = nullptr; // [nchan] the same in 8.56 fixed point (streaming kernel)
    int precision = 0;               // JSDR_PREC_F64 (exact) or JSDR_PREC_F32 (decimator in binary32)
    int kernel_mode = 0;             // JSDR_KERNEL_AUTO / _TILE / _STREAM
    double *d_tu_phase0 = nullptr;   // [nchan] initial tuPhase (zeros)
    const double *d_tu_phase = nullptr;   // committed tuPhase: phase0 or the phase_end of the last plan used
    // Scout output ("plan") for one block.  Two of them: while the data kernels work
    // through block k, the scout already replays block k+1 on the side stream.
    struct TunerPlan {
        double *ckpt = nullptr;      // [max_words][nchan] tuPhase before each 32-sample chunk
        double *phase_end = nullptr; // [nchan] tuPhase after the block
        int S = 0;
        bool valid = false;          // holds the plan for the next S samples from d_tu_phase
        bool used = false;           // `consumed` has been recorded at least once
        cudaEvent_t ready = nullptr, consumed = nullptr;
    } plan[2];
    int plan_cur = 0;
    double h_taps[128] = {0};        // host copy of the decimator taps (kernel parameter)
    double2 *d_ds_hist[2] = {nullptr, nullptr};   // [nchan][kMaxDsTaps] last ntaps-1 mixed samples
    int ds_hist_cur = 0;
    int ds_cnt = 0;                  // dsCnt carry (identical for all channels)
    int64_t cnt_raw = 0, cnt_ds = 0; // cntRaw / cntDS (identical for all channels)
    double2 *d_ds_out = nullptr;     // [nchan][max_ds]
    int last_nds = 0;

    double *d_vco_state = nullptr;   // [2][2] vcoPhase, dmBitPhase (channel independent): committed state and the replay's output
    int vco_state_cur = 0;           // which half is the committed state
    bool vco_ahead_valid = false;    // the replay of the NEXT block is already on the side stream
    int vco_ahead_NO = 0, vco_ahead_kb = 0;
    cudaEvent_t ev_vco_ready = nullptr;
    // jsdr_bpsk_read_ds_async: decimator done -> copy stream, copy done -> next block's decimator
    cudaEvent_t ev_ds_ready = nullptr, ev_ds_read = nullptr;
    int ds_read_pending = 0;
    // The bit-timing stage (and the frame stage behind it) runs on the context's auxiliary stream,
    // beside the next block's tuner / matched filter on the main stream.  What it reads is therefore
    // double buffered: matched-filter output, VCO table indices and bit-phase roll-overs of block k
    // live in buffer k&1 until the timing kernel of block k has finished (ev_bits_done[k&1]).
    uint8_t *d_vco_ix[2] = {nullptr, nullptr};     // [max_ds] table index per 9600 S/s sample
    uint8_t *d_bit_roll[2] = {nullptr, nullptr};   // [max_ds] 1 where dmBitPhase rolled over
    double2 *d_dm_buf[2] = {nullptr, nullptr};     // [nchan][max_ds] matched-filter output
    cudaEvent_t ev_dm_ready = nullptr, ev_bits_done[2] = {nullptr, nullptr};
    bool bits_used[2] = {false, false};
    int bit_cur = 0;
    double2 *d_dm_hist[2] = {nullptr, nullptr};   // [nchan][64] last 64 VCO-mixed samples
    int dm_hist_cur = 0;
    double2 *d_dm_out = nullptr;     // the buffer of d_dm_buf[] the last receive filled

    jsdr::bpsk::TimingState *d_ts = nullptr;   // [nchan]
    int8_t *d_bits = nullptr;        // [nchan][max_bits]
    long long *d_bit_at = nullptr;   // [nchan][max_bits]
    int32_t *d_nbits = nullptr;      // [nchan]

    void *d_in = nullptr;            // staging for host-pointer calls
    size_t in_cap = 0;

    // auto-tune variant (doBufferFFT, FUNcubeBPSKDemod.java:406-464)
    int dofft = 0, doUp = 0;
    double2 *d_at_work[2] = {nullptr, nullptr};   // [nchan][max_block] forward transform ping-pong
    double2 *d_at_rev[2] = {nullptr, nullptr};    // [nchan][max_block] 204 bins at DC, inverse ping-pong
    jsdr::bpsk::AutoTuneState *d_at_state = nullptr;   // [nchan]
};

struct jsdr_demod {
    jsdr_ctx *ctx = nullptr;
    int rate = 0, nchan = 0, max_block = 0, max_chunks = 0;
    int dofir = 1, dodwn = 1;
    std::vector<float> h_w;          // [nchan][21]
    std::vector<float> h_phi;        // [nchan]
    float *d_w = nullptr;            // [nchan][21]
    float *d_phi = nullptr;          // [nchan]
    float *d_car = nullptr;          // [nchan] carried phase
    float *d_chunk_car = nullptr;    // [max_chunks][nchan]
    float2 *d_hist[2] = {nullptr, nullptr};   // [nchan][20] last 20 input samples
    int hist_cur = 0;
    void *d_in = nullptr;
    float *d_out = nullptr;
    size_t in_cap = 0, out_cap = 0;
    // detectors + AGC (demod.java:405-481)
    int mode = 0, doagc = 0;         // MODE_OFF (:87 default)
    float2 *d_lilq = nullptr;        // [2][nchan] li, lq of the FM discriminator (:67-68); the second half is
                                     // k_detect's output when a row holds several blocks
    float *d_det = nullptr;          // [nchan][S] detector output scratch
    int16_t *d_audio = nullptr;      // host-call staging: s16 audio + max/avg
    size_t det_cap = 0, audio_cap = 0;
    // jsdr_pump_demod_s16: the car replay's end (side2 -> main stream) and the audio's (main
    // stream -> download stream)
    cudaEvent_t ev_car_ready = nullptr, ev_audio_ready = nullptr;
};

struct jsdr_fir {
    jsdr_ctx *ctx = nullptr;
    int nchan = 0, max_block = 0;
    double *d_w = nullptr;           // [nchan][21]
    int32_t *d_hist[2] = {nullptr, nullptr};  // [nchan][20]
    int hist_cur = 0;
    int32_t *d_in = nullptr, *d_out = nullptr;
    size_t in_cap = 0, out_cap = 0;
};

// demod_fir.cu: the demod handler of jsdr_pump_demod_s16 (pump.cu)
int jsdr_pump_demod_fork(jsdr_demod *d, int S);
int jsdr_pump_demod_staging(jsdr_demod *d, int S, int nblocks, int16_t **d_audio, float **d_max_avg);
int jsdr_pump_demod_run(jsdr_demod *d, const int16_t *d_raw, int S, int L, int ic, int qc, int16_t *audio,
                        float *max_avg);

int jsdr_fec_after_bits(jsdr_bpsk *b);   // fec.cu: run the frame stage on the bits of the last receive
void jsdr_fec_destroy(jsdr_bpsk *b);

namespace jsdr {
namespace fft {
enum { IN_F32 = 0, IN_S16 = 1 };
enum { OUT_PSD = 0, OUT_SPECTRUM = 1 };
// enqueue one batched transform on `st` (all pointers are device memory)
int launch(jsdr_fft *f, const void *d_in, int in_fmt, int batch, float *d_out, int32_t *d_peak,
           int out_mode, int ic, int qc, cudaStream_t st);
// grow the host-call staging d_in / d_out to at least these sizes; d_peak holds max_batch bins
int ensure_staging(jsdr_fft *f, size_t in_bytes, size_t out_bytes);
}  // namespace fft

namespace bpsk {
// bpsk.cu: jsdr_bpsk_receive_* (`fmt` FMT_F32 / FMT_S16), and the same in two halves for the pump
// (pump.cu), which enqueues its own kernels between them.  `pump` sizes the phase replay and the
// decimator's grid for a pump step (scout_threads, launch_stream).
int receive(jsdr_bpsk *b, const void *in, int fmt, int S, long long chan_stride, int ic, int qc, int mem,
            bool pump);
int receive_begin(jsdr_bpsk *b, const void *in, int fmt, int S, long long chan_stride, int mem, bool pump,
                  const void **d_in);
int receive_end(jsdr_bpsk *b, const void *d_in, int fmt, int S, long long chan_stride, int ic, int qc, int mem,
                bool pump);
}  // namespace bpsk
}  // namespace jsdr
