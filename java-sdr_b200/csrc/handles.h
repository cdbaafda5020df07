// handles.h — the opaque handle types behind include/jsdrcuda.h.
#pragma once

#include <stddef.h>
#include <stdint.h>

#include <memory>
#include <vector>

#include "common.cuh"

struct jsdr_fft {
    explicit jsdr_fft(jsdr_ctx *c) : ctx(c) {}
    ~jsdr_fft() { ctx->bind(); }
    jsdr_ctx *ctx;
    int n = 0, rate = 0, max_batch = 0;
    void *launch = nullptr;          // jsdr::fft::launch_fn of the plan
    jsdr::DevBuf<float2> d_tw;       // exp(-2*pi*i*t/n)
    // workspace of the four-step / staged paths (no single-CTA plan), allocated whole on first use
    struct Work {
        jsdr::DevBuf<float2> z[2];
        jsdr::DevBuf<unsigned long long> best;   // [max_batch] packed block maxima (four-step path)
    } work;
    int fs_n1 = 0;                            // four-step factor N1 (128 or 256), 0 otherwise
    int split = 0;                            // 2: split plan — two n/2-point transforms per block (fft_kernel SPLIT)
    jsdr::DevBuf<float2> d_tw2;               // split plan: exp(-2*pi*i*c/n), c in [0, n/2)
    jsdr::DevBuf<unsigned long long> d_best;  // split plan: [max_batch] packed block maxima
    jsdr::DevBuf<unsigned> d_cnt;             // split plan: halves reported per block (zero between launches)
    jsdr::DevBuf<float> d_win;                // [n] window of jsdr_fft_set_window (kept when the window is removed)
    bool win_on = false;                      // the kernels multiply by d_win
    // staging for host-pointer calls (allocated on first use)
    jsdr::DevBuf<void> d_in;
    jsdr::DevBuf<float> d_out;
    jsdr::DevBuf<int32_t> d_peak;
    jsdr::DevBuf<int32_t> d_pix;     // pixel rows of jsdr_pump_waterfall_s16's host path
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
struct jsdr_fec_delete {
    void operator()(jsdr_fec_state *f) const;   // fec.cu
};
int jsdr_launch_waterfall(jsdr_ctx *ctx, const float *d_psd, int n, int rows, int width, uint32_t peak_rgb,
                          int32_t *d_pix, cudaStream_t st);   // demod_fir.cu

struct jsdr_bpsk {
    explicit jsdr_bpsk(jsdr_ctx *c) : ctx(c) {}
    ~jsdr_bpsk()
    {
        ctx->bind();
        cudaStreamSynchronize(ctx->side);
        cudaStreamSynchronize(ctx->side2);
        cudaStreamSynchronize(ctx->stream);
        cudaStreamSynchronize(ctx->aux);
        if (ds_read_pending) cudaStreamSynchronize(ctx->copy_out);   // an asynchronous read may still be draining
    }
    jsdr_ctx *ctx;
    std::unique_ptr<jsdr_fec_state, jsdr_fec_delete> fec;   // sync correlator + FEC stage, when enabled
    int rate = 0, D = 0, nchan = 0, max_block = 0, stages = 3;
    int ntaps = 27;
    int max_ds = 0, max_words = 0, max_bits = 0;
    std::vector<double> h_tuning;

    jsdr::DevBuf<double> d_taps;     // [kMaxDsTaps] decimator low-pass
    jsdr::DevBuf<double> d_dmtaps;   // [65] matched filter
    jsdr::DevBuf<double> d_cossin;   // cosTab[256] then sinTab[256]
    jsdr::DevBuf<double2> d_cossin2; // (cos, sin) pairs, plus entry 256 = (1, 1) for the mixer bypass

    jsdr::DevBuf<double> d_tu_inc;   // [nchan] tuPhaseInc
    jsdr::DevBuf<jsdr::bpsk::ScoutChan> d_tu_par;   // [nchan] increment and exact wrap thresholds (phase scout)
    jsdr::DevBuf<unsigned long long> d_tu_dx;       // [nchan] table-index step per sample, 8.48 fixed point
    jsdr::DevBuf<unsigned long long> d_tu_dx56;     // [nchan] the same in 8.56 fixed point (streaming kernel)
    int precision = 0;               // JSDR_PREC_F64 (exact) or JSDR_PREC_F32 (decimator in binary32)
    int kernel_mode = 0;             // JSDR_KERNEL_AUTO / _TILE / _STREAM
    jsdr::DevBuf<double> d_tu_phase0;     // [nchan] initial tuPhase (zeros)
    const double *d_tu_phase = nullptr;   // committed tuPhase: phase0 or the phase_end of the last plan used
    // Scout output ("plan") for one block.  Two of them: while the data kernels work
    // through block k, the scout already replays block k+1 on the side stream.
    struct TunerPlan {
        jsdr::DevBuf<double> ckpt;       // [max_words][nchan] tuPhase before each 32-sample chunk
        jsdr::DevBuf<double> phase_end;  // [nchan] tuPhase after the block
        int S = 0;
        bool valid = false;          // holds the plan for the next S samples from d_tu_phase
        bool used = false;           // `consumed` has been recorded at least once
        jsdr::Event ready, consumed;
    } plan[2];
    int plan_cur = 0;
    double h_taps[128] = {0};        // host copy of the decimator taps (kernel parameter)
    jsdr::DevBuf<double2> d_ds_hist[2];   // [nchan][kMaxDsTaps] last ntaps-1 mixed samples
    int ds_hist_cur = 0;
    int ds_cnt = 0;                  // dsCnt carry (identical for all channels)
    int64_t cnt_raw = 0, cnt_ds = 0; // cntRaw / cntDS (identical for all channels)
    jsdr::DevBuf<double2> d_ds_out;  // [nchan][max_ds]
    int last_nds = 0;

    jsdr::DevBuf<double> d_vco_state;   // [2][2] vcoPhase, dmBitPhase (channel independent): committed state and the replay's output
    int vco_state_cur = 0;           // which half is the committed state
    bool vco_ahead_valid = false;    // the replay of the NEXT block is already on the side stream
    int vco_ahead_NO = 0, vco_ahead_kb = 0;
    // jsdr_bpsk_read_ds_async: decimator done -> copy stream, copy done -> next block's decimator
    jsdr::Event ev_ds_ready, ev_ds_read;
    int ds_read_pending = 0;
    // Buffers of the 9600 S/s stages, allocated whole when a receive first needs them.
    // The bit-timing stage (and the frame stage behind it) runs on the context's auxiliary stream,
    // beside the next block's tuner / matched filter on the main stream.  What it reads is therefore
    // double buffered: matched-filter output, VCO table indices and bit-phase roll-overs of block k
    // live in buffer k&1 until the timing kernel of block k has finished (ev_bits_done[k&1]).
    struct Stages {
        jsdr::DevBuf<uint8_t> d_vco_ix[2];     // [max_ds] table index per 9600 S/s sample
        jsdr::DevBuf<uint8_t> d_bit_roll[2];   // [max_ds] 1 where dmBitPhase rolled over
        jsdr::DevBuf<double2> d_dm_hist[2];    // [nchan][64] last 64 VCO-mixed samples
        jsdr::DevBuf<int8_t> d_bits;           // [nchan][max_bits]
        jsdr::DevBuf<long long> d_bit_at;      // [nchan][max_bits]
        jsdr::DevBuf<double2> d_dm_buf[2];     // [nchan][max_ds] matched-filter output
        jsdr::Event ev_dm_ready, ev_vco_ready, ev_bits_done[2];
    } stage;
    bool bits_used[2] = {false, false};
    int bit_cur = 0;
    int dm_hist_cur = 0;
    double2 *d_dm_out = nullptr;     // the buffer of stage.d_dm_buf[] the last receive filled

    jsdr::DevBuf<jsdr::bpsk::TimingState> d_ts;   // [nchan]
    jsdr::DevBuf<int32_t> d_nbits;   // [nchan]

    jsdr::DevBuf<void> d_in;         // staging for host-pointer calls

    // auto-tune variant (doBufferFFT, FUNcubeBPSKDemod.java:406-464)
    int dofft = 0, doUp = 0;
    struct AutoTune {                // allocated whole by the first auto-tune block
        jsdr::DevBuf<double2> d_at_work[2];   // [nchan][max_block] forward transform ping-pong
        jsdr::DevBuf<double2> d_at_rev[2];    // [nchan][max_block] 204 bins at DC, inverse ping-pong
        jsdr::DevBuf<jsdr::bpsk::AutoTuneState> d_at_state;   // [nchan]
    } at;
};

struct jsdr_demod {
    explicit jsdr_demod(jsdr_ctx *c) : ctx(c) {}
    ~jsdr_demod()
    {
        ctx->bind();
        cudaStreamSynchronize(ctx->side);
        cudaStreamSynchronize(ctx->side2);
        cudaStreamSynchronize(ctx->copy_out);
        cudaStreamSynchronize(ctx->stream);
    }
    jsdr_ctx *ctx;
    int rate = 0, nchan = 0, max_block = 0, max_chunks = 0;
    int dofir = 1, dodwn = 1;
    std::vector<float> h_w;          // [nchan][21]
    std::vector<float> h_phi;        // [nchan]
    jsdr::DevBuf<float> d_w;         // [nchan][21]
    jsdr::DevBuf<float> d_phi;       // [nchan]
    jsdr::DevBuf<float> d_car;       // [nchan] carried phase
    jsdr::DevBuf<float> d_chunk_car; // [max_chunks][nchan]
    jsdr::DevBuf<float2> d_hist[2];  // [nchan][20] last 20 input samples
    int hist_cur = 0;
    jsdr::DevBuf<void> d_in;
    jsdr::DevBuf<float2> d_out;
    // detectors + AGC (demod.java:405-481)
    int mode = 0, doagc = 0;         // MODE_OFF (:87 default)
    jsdr::DevBuf<float2> d_lilq;     // [2][nchan] li, lq of the FM discriminator (:67-68); the second half is
                                     // k_detect's output when a row holds several blocks
    jsdr::DevBuf<float> d_det;       // [nchan][S] detector output scratch
    jsdr::DevBuf<int16_t> d_audio;   // host-call staging: s16 audio + max/avg
    // jsdr_pump_demod_s16: the car replay's end (side2 -> main stream) and the audio's (main
    // stream -> download stream)
    jsdr::Event ev_car_ready, ev_audio_ready;
};

struct jsdr_fir {
    explicit jsdr_fir(jsdr_ctx *c) : ctx(c) {}
    ~jsdr_fir()
    {
        ctx->bind();
        cudaStreamSynchronize(ctx->stream);
    }
    jsdr_ctx *ctx;
    int nchan = 0, max_block = 0;
    jsdr::DevBuf<double> d_w;        // [nchan][21]
    jsdr::DevBuf<int32_t> d_hist[2]; // [nchan][20]
    int hist_cur = 0;
    jsdr::DevBuf<int32_t> d_in, d_out;
};

// demod_fir.cu: the demod handler of jsdr_pump_demod_s16 (pump.cu)
int jsdr_pump_demod_fork(jsdr_demod *d, int S);
int jsdr_pump_demod_staging(jsdr_demod *d, int S, int nblocks, int16_t **d_audio, float **d_max_avg);
int jsdr_pump_demod_run(jsdr_demod *d, const int16_t *d_raw, int S, int L, int ic, int qc, int16_t *audio,
                        float *max_avg);

int jsdr_fec_after_bits(jsdr_bpsk *b);   // fec.cu: run the frame stage on the bits of the last receive

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
