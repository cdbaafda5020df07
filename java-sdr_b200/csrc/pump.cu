// pump.cu — JavaAudio.run's fan-out (JavaAudio.java:262-304) for a batch: each channel's blocks go
// to the fft handler, the tuner bank and, in jsdr_pump_demod_s16, the demod handler.
#include <algorithm>

#include "handles.h"

using namespace jsdr;

namespace {

struct PumpPixels {          // jsdr_pump_waterfall_s16: pixel rows and the two trailing floats instead of the PSD
    int width;
    uint32_t rgb;
    int32_t *pixels;         // [batch][width]
    float *peak;             // [batch][2]: psd[N] (peak Hz), psd[N+1] (peak dB)
};
struct PumpDemod {           // jsdr_pump_demod_s16: the demod handler beside the other two
    jsdr_demod *d;
    int16_t *audio;          // [nchan][nblocks*n]
    float *max_avg;          // nullable: [nchan][nblocks][2]
};

// Every refusal of the three calls, before anything is enqueued: the demod's car replay is forked
// first, and the bank's own checks would come after the FFT and the demod had consumed the block.
int pump_check(const jsdr_fft *f, const jsdr_bpsk *b, const int16_t *raw, int nblocks, const float *psd, int mem,
               const PumpPixels *px, const PumpDemod *dm)
{
    JSDR_REQUIRE(f && b && raw && (px ? px->pixels && px->peak : psd != nullptr), JSDR_EINVAL, "null argument");
    JSDR_REQUIRE(mem == JSDR_MEM_HOST || mem == JSDR_MEM_DEVICE, JSDR_EINVAL, "bad mem");
    JSDR_REQUIRE(f->ctx == b->ctx, JSDR_EINVAL, "handlers belong to different contexts");
    JSDR_REQUIRE(nblocks > 0, JSDR_EINVAL, "nblocks must be positive");
    const long long S = (long long)nblocks * f->n;
    JSDR_REQUIRE(S <= b->max_block, JSDR_EINVAL, "nblocks*n exceeds the bank's max_block_samples");
    JSDR_REQUIRE((long long)nblocks * b->nchan <= f->max_batch, JSDR_EINVAL, "nchan*nblocks exceeds the fft's max_batch");
    JSDR_REQUIRE(!b->dofft || S == b->max_block, JSDR_EINVAL, "auto-tune needs whole blocks of max_block_samples");
    if (px) JSDR_REQUIRE(px->width > 0 && px->width <= f->n, JSDR_EINVAL, "need 0 < width <= n");
    if (dm) {
        JSDR_REQUIRE(dm->d && dm->audio, JSDR_EINVAL, "null argument");
        JSDR_REQUIRE(dm->d->ctx == f->ctx, JSDR_EINVAL, "handlers belong to different contexts");
        JSDR_REQUIRE(dm->d->nchan == b->nchan, JSDR_EINVAL, "the demod and the bank need the same channel count");
        JSDR_REQUIRE(S <= dm->d->max_block, JSDR_EINVAL, "nblocks*n exceeds the demod's max_block_samples");
    }
    return JSDR_OK;
}

int pump_receive(jsdr_fft *f, jsdr_bpsk *b, const int16_t *raw, int nblocks, int ic, int qc, float *psd,
                 int32_t *peak_bin, int mem, const PumpPixels *px, const PumpDemod *dm)
{
    JSDR_TRY(pump_check(f, b, raw, nblocks, psd, mem, px, dm));
    jsdr_ctx *ctx = f->ctx;
    JSDR_TRY(ctx->bind());
    // JavaAudio.java:281-288: every handler sees the corrected samples (ic, qc)
    const int S = nblocks * f->n;
    const int batch = nblocks * b->nchan;
    const int N2 = f->n + 2;
    const size_t psd_bytes = sizeof(float) * (size_t)batch * N2;
    if (dm) JSDR_TRY(jsdr_pump_demod_fork(dm->d, S));   // the car replay starts beside everything below

    if (mem == JSDR_MEM_DEVICE) {
        // Between the bank's halves: behind its fork, so that the next block's phase replay (side
        // stream) starts beside this FFT and not behind it; the demod kernels follow the FFT, ahead
        // of the bank's wait for this block's tuner-phase replay.
        if (px) JSDR_TRY(fft::ensure_staging(f, 0, psd_bytes));
        float *d_psd = px ? f->d_out.get() : psd;
        int32_t *d_peak = (px && !peak_bin) ? f->d_peak.get() : peak_bin;
        const void *d_in;
        JSDR_TRY(bpsk::receive_begin(b, raw, bpsk::FMT_S16, S, S, mem, true, &d_in));
        JSDR_TRY(fft::launch(f, d_in, fft::IN_S16, batch, d_psd, d_peak, fft::OUT_PSD, ic, qc, ctx->stream));
        if (px) {   // paintLine and the maxima behind the FFT
            JSDR_TRY(jsdr_launch_waterfall(ctx, d_psd, f->n, batch, px->width, px->rgb, px->pixels, ctx->stream));
            JSDR_CUDA(cudaMemcpy2DAsync(px->peak, 2 * sizeof(float), d_psd + f->n, N2 * sizeof(float),
                                        2 * sizeof(float), (size_t)batch, cudaMemcpyDeviceToDevice, ctx->stream));
        }
        if (dm)
            JSDR_TRY(jsdr_pump_demod_run(dm->d, static_cast<const int16_t *>(d_in), S, f->n, ic, qc, dm->audio,
                                         dm->max_avg));
        return bpsk::receive_end(b, d_in, bpsk::FMT_S16, S, S, ic, qc, mem, true);
    }

    JSDR_TRY(fft::ensure_staging(f, 0, psd_bytes));
    JSDR_TRY(b->d_in.grow((size_t)b->nchan * (size_t)S * 4, "tuner bank staging"));
    if (px) JSDR_TRY(f->d_pix.grow((size_t)batch * px->width * sizeof(int32_t), "pixel staging"));
    char *d_raw = static_cast<char *>(b->d_in.get());   // the batch, resident for all handlers
    float *d_psd = f->d_out.get();
    int32_t *d_peak = f->d_peak.get(), *d_pix = f->d_pix.get();
    // Host path, pipelined over channel chunks: PCIe is full duplex, so the upload of chunk
    // c+1 (copy_in stream) runs beside the FFT of chunk c (main stream) and the download of
    // the results of chunk c-1 (copy_out stream).  The tuner bank runs once the whole batch is in.
    const int nchunk = std::min(16, std::max(1, b->nchan / 8));
    JSDR_CUDA(cudaEventRecord(ctx->ev_fork, ctx->stream));            // staging buffers are free again
    JSDR_CUDA(cudaStreamWaitEvent(ctx->copy_in, ctx->ev_fork, 0));
    for (int c = 0; c < nchunk; c++) {
        const int c0 = (int)((long long)b->nchan * c / nchunk), c1 = (int)((long long)b->nchan * (c + 1) / nchunk);
        if (c1 == c0) continue;
        const size_t in_off = (size_t)c0 * (size_t)S * 4, in_len = (size_t)(c1 - c0) * (size_t)S * 4;
        const size_t blk0 = (size_t)c0 * nblocks, nblk = (size_t)(c1 - c0) * nblocks;
        JSDR_CUDA(cudaMemcpyAsync(d_raw + in_off, (const char *)raw + in_off, in_len,
                                  cudaMemcpyHostToDevice, ctx->copy_in));
        JSDR_CUDA(cudaEventRecord(ctx->ev_chunk_in[c], ctx->copy_in));
        JSDR_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_chunk_in[c], 0));
        JSDR_TRY(fft::launch(f, d_raw + in_off, fft::IN_S16, (int)nblk, d_psd + blk0 * N2, d_peak + blk0, fft::OUT_PSD,
                             ic, qc, ctx->stream));
        if (px)
            JSDR_TRY(jsdr_launch_waterfall(ctx, d_psd + blk0 * N2, f->n, (int)nblk, px->width, px->rgb,
                                           d_pix + blk0 * px->width, ctx->stream));
        JSDR_CUDA(cudaEventRecord(ctx->ev_chunk_done[c], ctx->stream));
        JSDR_CUDA(cudaStreamWaitEvent(ctx->copy_out, ctx->ev_chunk_done[c], 0));
        if (px) {
            JSDR_CUDA(cudaMemcpyAsync(px->pixels + blk0 * px->width, d_pix + blk0 * px->width,
                                      nblk * px->width * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->copy_out));
            JSDR_CUDA(cudaMemcpy2DAsync(px->peak + blk0 * 2, 2 * sizeof(float), d_psd + blk0 * N2 + f->n, N2 * sizeof(float),
                                        2 * sizeof(float), nblk, cudaMemcpyDeviceToHost, ctx->copy_out));
        } else {
            JSDR_CUDA(cudaMemcpyAsync(psd + blk0 * N2, d_psd + blk0 * N2, nblk * N2 * sizeof(float),
                                      cudaMemcpyDeviceToHost, ctx->copy_out));
        }
        if (peak_bin)
            JSDR_CUDA(cudaMemcpyAsync(peak_bin + blk0, d_peak + blk0, sizeof(int32_t) * nblk,
                                      cudaMemcpyDeviceToHost, ctx->copy_out));
    }
    if (dm) {   // the whole batch is in (the main stream waited for every chunk): demod, audio down beside the bank
        jsdr_demod *d = dm->d;
        int16_t *d_audio = nullptr;
        float *d_ma = nullptr;
        JSDR_TRY(jsdr_pump_demod_staging(d, S, nblocks, &d_audio, &d_ma));
        JSDR_TRY(jsdr_pump_demod_run(d, reinterpret_cast<const int16_t *>(d_raw), S, f->n, ic, qc, d_audio,
                                     dm->max_avg ? d_ma : nullptr));
        JSDR_CUDA(cudaEventRecord(d->ev_audio_ready, ctx->stream));
        JSDR_CUDA(cudaStreamWaitEvent(ctx->copy_out, d->ev_audio_ready, 0));
        JSDR_CUDA(cudaMemcpyAsync(dm->audio, d_audio, sizeof(int16_t) * (size_t)b->nchan * S, cudaMemcpyDeviceToHost,
                                  ctx->copy_out));
        if (dm->max_avg)
            JSDR_CUDA(cudaMemcpyAsync(dm->max_avg, d_ma, sizeof(float) * 2 * (size_t)b->nchan * nblocks,
                                      cudaMemcpyDeviceToHost, ctx->copy_out));
    }
    JSDR_TRY(bpsk::receive(b, d_raw, bpsk::FMT_S16, S, S, ic, qc, JSDR_MEM_DEVICE, true));
    JSDR_CUDA(cudaStreamSynchronize(ctx->copy_out));
    JSDR_CUDA(cudaStreamSynchronize(ctx->stream));
    return JSDR_OK;
}

}  // namespace

// The fft handler and the tuner bank over the same resident batch.
extern "C" int jsdr_pump_receive_s16(jsdr_fft *f, jsdr_bpsk *b, const int16_t *raw, int nblocks,
                                     int ic, int qc, float *psd, int32_t *peak_bin, int mem)
try {
    return pump_receive(f, b, raw, nblocks, ic, qc, psd, peak_bin, mem, nullptr, nullptr);
} JSDR_CATCH_ALL

// JavaAudio.run's whole fan-out (JavaAudio.java:298-304): the fft handler, the demod handler and
// the tuner bank over one resident batch.  The demod part equals nblocks successive demod.receive
// calls of n samples per channel.
extern "C" int jsdr_pump_demod_s16(jsdr_fft *f, jsdr_bpsk *b, jsdr_demod *d, const int16_t *raw, int nblocks,
                                   int ic, int qc, float *psd, int32_t *peak_bin, int16_t *audio, float *max_avg,
                                   int mem)
try {
    const PumpDemod dm = {d, audio, max_avg};
    return pump_receive(f, b, raw, nblocks, ic, qc, psd, peak_bin, mem, nullptr, &dm);
} JSDR_CATCH_ALL

// The same fan-out with waterfall.java's paintLine (:90-107) chained behind every block's PSD on
// the device: what returns is the pixel row a waterfall draws and the two published maxima
// (fft.java:223-224), 4*width + 8 bytes per block instead of 4*(N+2).
extern "C" int jsdr_pump_waterfall_s16(jsdr_fft *f, jsdr_bpsk *b, const int16_t *raw, int nblocks, int ic, int qc,
                                       int width, uint32_t peak_rgb, int32_t *pixels, float *peak, int32_t *peak_bin,
                                       int mem)
try {
    const PumpPixels px = {width, peak_rgb, pixels, peak};
    return pump_receive(f, b, raw, nblocks, ic, qc, nullptr, peak_bin, mem, &px, nullptr);
} JSDR_CATCH_ALL
