/*
 * jsdrcuda.h — C ABI of libjsdrcuda.so, the B200 (sm_100a) implementation of
 * java-sdr's IQ front-end hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  Every entry point takes plain
 * pointers and sizes so that java.lang.foreign (or JNI, or ctypes) can bind it
 * without glue; INTEGRATION.md shows the Java-side binding.  Each group cites
 * the reference interface it stands behind (paths relative to the reference
 * checkout).
 *
 * Conventions
 *   - every function returns JSDR_OK (0) or a negative jsdr_status; the text of
 *     the last failure on the calling thread is jsdr_last_error().  Nothing
 *     throws: an exception escaping IAudioHandler.receive would end ingest
 *     (JavaAudio.java:321-323), so the shim only ever sees return codes.
 *   - `mem` says where the data pointers of that call live: JSDR_MEM_HOST
 *     (the call copies in/out and returns with results ready — what the Java
 *     handlers use) or JSDR_MEM_DEVICE (pointers are device memory from
 *     jsdr_dev_alloc; the call only enqueues work on the context's stream,
 *     jsdr_ctx_sync waits for it).
 *   - IQ is interleaved I,Q.  float IQ is the IAudioHandler contract
 *     (IAudioHandler.java:3-5, nominal +-1); int16 IQ is the IRawHandler
 *     contract (IRawHandler.java:3-5, s16le, before I/Q correction), converted
 *     on the device by the rule of JavaAudio.java:276-293.
 *   - threading: a context and the handles created from it are driven by one thread at a
 *     time, like the reference's handlers, which all run on JavaAudio's single "run" thread
 *     (JavaAudio.java:298-304).  Different contexts (one per GPU) are independent.
 *   - there is no CPU fallback: without a CUDA device every create call fails
 *     with JSDR_ECUDA.
 */
#ifndef JSDRCUDA_H
#define JSDRCUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define JSDR_ABI_VERSION 2

typedef enum jsdr_status {
    JSDR_OK = 0,
    JSDR_EINVAL = -1,       /* bad argument */
    JSDR_ECUDA = -2,        /* CUDA runtime error / no device */
    JSDR_ENOMEM = -3,
    JSDR_EUNSUPPORTED = -4, /* e.g. an FFT length with no plan */
    JSDR_ESTATE = -5,       /* call out of order */
    JSDR_EINTERNAL = -6     /* a C++ exception other than out-of-memory was caught at the boundary */
} jsdr_status;

enum { JSDR_MEM_HOST = 0, JSDR_MEM_DEVICE = 1 };

typedef struct jsdr_ctx jsdr_ctx;
typedef struct jsdr_fft jsdr_fft;
typedef struct jsdr_bpsk jsdr_bpsk;
typedef struct jsdr_demod jsdr_demod;
typedef struct jsdr_fir jsdr_fir;

/* ------------------------------------------------------------------ context */
int         jsdr_abi_version(void);
const char *jsdr_last_error(void);
int         jsdr_device_count(int *count);
int         jsdr_ctx_create(int device, jsdr_ctx **out);
int         jsdr_ctx_destroy(jsdr_ctx *ctx);
int         jsdr_ctx_sync(jsdr_ctx *ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
int         jsdr_ctx_launch_count(jsdr_ctx *ctx, int64_t *count);

/* Optional per-kernel timing: while enabled, every launch of the kernels below is
 * bracketed by CUDA events on its own stream; _read waits for the work and returns
 * the summed milliseconds and launch counts per kind since the last read
 * (ms/count hold JSDR_K_COUNT entries; at most 65536 launches are kept between two reads,
 * later ones are not timed).  bench.py's roofline numbers come from here. */
enum { JSDR_K_FFT = 0, JSDR_K_MIXDECIM = 1, JSDR_K_MATCHED = 2, JSDR_K_TIMING = 3, JSDR_K_SCOUT = 4,
       JSDR_K_OTHER = 5, JSDR_K_DEMOD = 6, JSDR_K_FIR = 7, JSDR_K_DETECT = 8, JSDR_K_WATERFALL = 9,
       JSDR_K_SYNC = 10, JSDR_K_FEC = 11, JSDR_K_COUNT = 12 };
int         jsdr_ctx_profile(jsdr_ctx *ctx, int enable);
int         jsdr_ctx_profile_read(jsdr_ctx *ctx, double *ms, int64_t *count, int nkinds);

/* pinned host rings handed to Java as MemorySegments; plain device buffers for
 * device-resident batches */
int jsdr_host_alloc(jsdr_ctx *ctx, size_t bytes, void **out);
int jsdr_host_free(jsdr_ctx *ctx, void *p);
int jsdr_dev_alloc(jsdr_ctx *ctx, size_t bytes, void **out);
int jsdr_dev_free(jsdr_ctx *ctx, void *p);
int jsdr_memcpy_h2d(jsdr_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes);
int jsdr_memcpy_d2h(jsdr_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes);
int jsdr_memset_dev(jsdr_ctx *ctx, void *dst_dev, int value, size_t bytes);
/* CUDA-event timing on the context's stream (bench.py times with these) */
int jsdr_timer_start(jsdr_ctx *ctx);
int jsdr_timer_stop_ms(jsdr_ctx *ctx, float *ms);

/* ------------------------------------------------------------------ fft.java
 * Replaces fft.receive (fft.java:190-228) for `batch` independent blocks of n
 * complex samples: unnormalised forward DFT (the FloatFFT_1D.complexForward
 * contract, fft.java:194-195), psd[k] = 10*log10((re^2+im^2)*(2/n)^2)
 * (:199-207), first strict maximum (:208-211) converted to Hz with wrapping
 * int32 arithmetic (:214-221).  Output per block is the published "fft-psd"
 * array: float[n+2] = n dB values in FFT order, then peak Hz, then peak dB
 * (:223-226).  peak_bin (nullable, int32 per block) additionally exports the
 * arg-max bin (-1 if no bin compared greater), because the Hz value wraps
 * beyond +-53.7 kHz at 192 kS/s (SURVEY Q2).
 * No window is applied unless jsdr_fft_set_window sets one (fft.java never applies
 * win[]; SURVEY Q1).
 */
int jsdr_fft_supported(int n);   /* 1 if a plan exists for n */
int jsdr_fft_create(jsdr_ctx *ctx, int n, int rate, int max_batch, jsdr_fft **out);
int jsdr_fft_destroy(jsdr_fft *f);
int jsdr_fft_receive_f32(jsdr_fft *f, const float *iq, int batch, float *psd,
                         int32_t *peak_bin, int mem);
int jsdr_fft_receive_s16(jsdr_fft *f, const int16_t *raw, int batch, int ic, int qc,
                         float *psd, int32_t *peak_bin, int mem);
/* the spectrum itself (what complexForward leaves in dat[]): float[2n] per block */
int jsdr_fft_forward_f32(jsdr_fft *f, const float *iq, int batch, float *spec, int mem);
/* Multiply each block's sample t (I and Q alike) by win[t] before the transform: what fft.java
 * would publish if receive() applied its win[] (fft.java:72-73) to dat[] ahead of complexForward.
 * win is host memory, float[n]; NULL removes the window.  No gain correction: cf stays (2/n)^2.
 * Applies to jsdr_fft_receive_f32/_s16, jsdr_fft_forward_f32 and the fft part of the three pumps;
 * the bank and the demod handler of a pump still see unwindowed samples.
 *   - stream-ordered on the context's stream: work already enqueued with JSDR_MEM_DEVICE uses the
 *     window in force when it was enqueued, calls after this one use the new window.
 *   - a non-finite entry (JSDR_EINVAL, the message names the first one) or a failed allocation
 *     (JSDR_ENOMEM) leaves the previous window in force.
 *   - arithmetic: one binary32 multiply per component on the converted sample, before any
 *     butterfly: RN(x*win[t]) for float input, RN((float)s*win[t]) for s16 input, s the value after
 *     the ic / qc correction (the 1/32767 stays folded into cf).  Java's order, RN(RN(s/32767f)*w),
 *     differs from this by a few ulps per sample, far inside the 1e-4 parity bar. */
int jsdr_fft_set_window(jsdr_fft *f, const float *win);

/* ------------------------------------------------------- FUNcubeBPSKDemod.java
 * A bank of `nchan` independent FUNcube tuners.  One receive call is one
 * IAudioHandler.receive(buf) (FUNcubeBPSKDemod.java:358-364, doBufferTune
 * :366-379) for every channel at once:
 *   RxMixTuner   :382-397  table NCO, i*cos / q*sin, phase accumulated exactly
 *   RxDownSample :467-492  decimate by rate/9600 with the 27-tap low-pass, x0.9*32768
 *   RxDemodulate :505-595  1200 Hz VCO mix, 65-tap matched filter (slot-ordered
 *                          sum), bit-energy timing, differential decision
 * All in binary64 in the reference's operation order, so every output is
 * bit-identical to the Java arithmetic.  State persists across calls.
 * chan_stride: distance between channels' inputs in complex samples; 0 means
 * one shared stream fans out to every tuner (the reference's own model,
 * jsdr.java:479-483).
 * stages: 1 = tuner + decimator only, 2 = + matched filter, 3 = + bit timing
 * and decisions (default).
 */
int jsdr_bpsk_create(jsdr_ctx *ctx, int rate, int nchan, const double *tuning_hz,
                     int max_block_samples, jsdr_bpsk **out);
int jsdr_bpsk_destroy(jsdr_bpsk *b);
int jsdr_bpsk_set_stages(jsdr_bpsk *b, int stages);
int jsdr_bpsk_set_tuning(jsdr_bpsk *b, int chan, double hz);       /* :174-189 */
/* The FFT auto-tune variant, doBufferFFT (FUNcubeBPSKDemod.java:406-464; config keys
 * "FUNcube<i>-bpsk-dofft" / "-upper", :198-200): when dofft is set every receive call
 * must carry exactly max_block_samples samples (the transform length is the block
 * length, :421; 1024..115712 samples with no prime factor beyond 7 — rate/10 of every
 * supported rate qualifies — otherwise set_autotune answers JSDR_EUNSUPPORTED).  Forward transform in binary64, 100-bin boxcar arg-max over the lower
 * (or, do_upper, upper) quarter band, smoothed / gated / clamped centre bin, 204 bins
 * moved to DC, inverse transform scaled by 1/n, decimator fed (re, re) (:461-463).
 * read_centre returns what the reference publishes as "<name>-bpsk-centre" (:456). */
int jsdr_bpsk_set_autotune(jsdr_bpsk *b, int dofft, int do_upper);
int jsdr_bpsk_read_centre(jsdr_bpsk *b, int32_t *centre_bin /* nchan */);
/* Arithmetic of the tuner + decimator stage.  JSDR_PREC_F64 (default) is the
 * reference's binary64 in the reference's operation order: every output is
 * bit-identical to the Java arithmetic, and the bits that follow are exact.
 * JSDR_PREC_F32 keeps the exact tuner table index sequence but mixes and filters
 * in binary32 (filtered samples within 1e-4 of full scale of the binary64 path);
 * it is meant for channeliser use (stages == 1), not for bit decisions. */
enum { JSDR_PREC_F64 = 0, JSDR_PREC_F32 = 1 };
int jsdr_bpsk_set_precision(jsdr_bpsk *b, int precision);
/* Kernel choice for the tuner + decimator (results are identical): AUTO picks the
 * streaming kernel (one lane per channel) for banks of >= 32 channels of s16 input
 * and the tile kernel (one CTA per channel tile) otherwise. */
enum { JSDR_KERNEL_AUTO = 0, JSDR_KERNEL_TILE = 1, JSDR_KERNEL_STREAM = 2 };
int jsdr_bpsk_set_kernel(jsdr_bpsk *b, int mode);
/* replace the 27-tap decimator low-pass (BASELINE config 4 uses 64 taps); resets
 * the decimator history like a fresh instance */
int jsdr_bpsk_set_ds_filter(jsdr_bpsk *b, const double *taps, int ntaps);
int jsdr_bpsk_receive_f32(jsdr_bpsk *b, const float *iq, int nsamples,
                          int64_t chan_stride, int mem);
int jsdr_bpsk_receive_s16(jsdr_bpsk *b, const int16_t *raw, int nsamples,
                          int64_t chan_stride, int ic, int qc, int mem);
/* what the last receive produced, per channel */
int jsdr_bpsk_last_counts(jsdr_bpsk *b, int32_t *n_ds /* outputs per channel */);
int jsdr_bpsk_read_ds(jsdr_bpsk *b, double *out /* nchan*n_ds*2 */, int mem);   /* fed to RxDemodulate */
/* the same copy without the wait: it runs on the download stream behind the decimator, beside
 * whatever is submitted next (the following block's upload); `out` holds the rows once
 * jsdr_ctx_sync has returned.  The next receive orders itself behind the copy. */
int jsdr_bpsk_read_ds_async(jsdr_bpsk *b, double *out /* nchan*n_ds*2 */, int mem);
int jsdr_bpsk_read_dm(jsdr_bpsk *b, double *out /* nchan*n_ds*2 */, int mem);   /* matched filter fi,fq */
/* bits are +1/-1 (the value written to dmFECCorr, :554); bit_at is the cntDS
 * index of the 9600 S/s sample the decision was taken on.  max_bits is the row
 * pitch of bits/bit_at; nbits[c] is how many channel c produced this call. */
int jsdr_bpsk_read_bits(jsdr_bpsk *b, int8_t *bits, int64_t *bit_at, int32_t *nbits,
                        int max_bits, int mem);
/* cntRaw, cntDS, cntBit, reserved — 4 x int64 per channel (:114, painted at :220) */
int jsdr_bpsk_read_counters(jsdr_bpsk *b, int64_t *counters);
/* device pointer of the decimated output for zero-copy consumers */
int jsdr_bpsk_ds_device_ptr(jsdr_bpsk *b, double **dev_ptr);

/* The frame stage behind the bits (FUNcubeBPSKDemod.java:553-574, FECDecoder.java:703-852):
 * once enabled, every receive call (stages == 3) also runs the sync correlator over the
 * new bits (65-point correlation with SYNC_VECTOR at stride 80 across the last 5200 bits,
 * >= 45 starts a decode) and FECDecode on every hit: de-interleave, Viterbi K=7 r=1/2,
 * de-scramble, two RS(160,128) decoders, re-encode and count channel errors.
 * mettab is the Viterbi metric table int16[2][256] (a literal in FECDecoder.java:67-100;
 * the caller passes the reference's own array).  read_frames returns this call's frames
 * ordered by (channel, bit): errors is FECDecode's return value (channel errors, or -1 if
 * an RS block failed, data then zero); bit_index is cntBit of the bit that completed the
 * frame; *nframes is the number detected (it can exceed max_frames, the rest are dropped).
 * read_fec_counters: cntFEC and cntDec per channel (:567,571). */
int jsdr_bpsk_enable_fec(jsdr_bpsk *b, const int16_t *mettab, int max_frames_per_call);
int jsdr_bpsk_read_frames(jsdr_bpsk *b, int32_t *nframes, int32_t *chan, int64_t *bit_index,
                          int32_t *errors, uint8_t *data /* max_frames*256 */, int max_frames);
int jsdr_bpsk_read_fec_counters(jsdr_bpsk *b, int64_t *cnt_fec, int64_t *cnt_dec);

/* ------------------------------------------------------------------ demod.java
 * FIR band-pass + NCO down-shift part of demod.receive (demod.java:410-434) for
 * nchan channels: 21-tap complex FIR with float taps and float accumulation in
 * the reference order (filter(), :378-396), then the float phase accumulator
 * NCO (:424-433).  weights() follows :341-375 (flo == INT32_MIN gives the
 * all-pass); until it is called the taps are zero (SURVEY Q5).
 */
int jsdr_demod_create(jsdr_ctx *ctx, int rate, int nchan, int max_block_samples, jsdr_demod **out);
int jsdr_demod_destroy(jsdr_demod *d);
int jsdr_demod_weights(jsdr_demod *d, int chan, int flo, int fhi);
int jsdr_demod_get_weights(jsdr_demod *d, int chan, float w[21]);
int jsdr_demod_set_flags(jsdr_demod *d, int dofir, int dodwn);
int jsdr_demod_receive_f32(jsdr_demod *d, const float *iq, int nsamples, int64_t chan_stride,
                           float *out /* nchan*2*nsamples */, int mem);
/* The same on s16 IQ of the IRawHandler contract (what the dongle delivers): each sample is
 * converted on the device as JavaAudio does before it calls its handlers (JavaAudio.java:276-293,
 * ic/qc added with 16-bit wrap, then (float)s/32767f), so the result equals receive_f32 on the
 * converted floats bit for bit.  chan_stride counts complex samples (0: one shared stream).
 * The delay line holds converted floats: s16 and f32 calls may alternate on one handle. */
int jsdr_demod_receive_s16(jsdr_demod *d, const int16_t *raw, int nsamples, int64_t chan_stride,
                           int ic, int qc, float *out /* nchan*2*nsamples */, int mem);

/* The detectors, AGC and s16 narrowing that follow the FIR + NCO in demod.receive
 * (demod.java:405-481): mode 0 off, 1 raw (I), 2 AM (envelope minus its running mean),
 * 3 NFM / 4 WFM (quadrature discriminator, gain rate/5000 or rate/75000); doagc scales
 * by 1.0f/max.  audio is what receive() writes to bbf: one s16 per input sample
 * (the reference writes it to both stereo channels, :474-477), nchan*nsamples;
 * max_avg (nullable) returns max and avg per channel (painted at :544-547). */
int jsdr_demod_set_mode(jsdr_demod *d, int mode, int doagc);
int jsdr_demod_receive_audio_f32(jsdr_demod *d, const float *iq, int nsamples, int64_t chan_stride,
                                 int16_t *audio, float *max_avg /* nchan*2 */, int mem);
/* The whole of demod.receive on s16 IQ, converted as in jsdr_demod_receive_s16. */
int jsdr_demod_receive_audio_s16(jsdr_demod *d, const int16_t *raw, int nsamples, int64_t chan_stride,
                                 int ic, int qc, int16_t *audio, float *max_avg /* nchan*2 */, int mem);

/* -------------------------------------------------------------- waterfall.java
 * paintLine (waterfall.java:90-107) for `rows` published "fft-psd" rows (float[n+2]
 * each): max-decimate to `width` pixels, -100..0 dBFS -> 0..255, tint with peak_rgb
 * (waterfall.java:15, Color.CYAN = 0x00ffff), rotate by width/2, ARGB out
 * [rows][width].  With JSDR_MEM_DEVICE it chains behind jsdr_fft_receive_* so that
 * only the pixel row returns to the host. */
int jsdr_waterfall_rows(jsdr_ctx *ctx, const float *psd, int n, int rows, int width, uint32_t peak_rgb,
                        int32_t *pixels, int mem);

/* ------------------------------------------------------------------ fir.java
 * The four arithmetic methods of the stand-alone fir.java tool:
 *   weights     :169-195  (host, one-off)            jsdr_fir_design
 *   filter      :198-211  int samples x double taps  jsdr_fir_filter_i32
 *   complex_gen :221-228  one period of the integer NCO (host, one-off)
 *   complex_mod :214-218  wrapping int32 complex multiply
 */
int jsdr_fir_design(int f1, int f2, float rate, double w[21]);
int jsdr_fir_nco_table(int freq, float rate, int32_t *sig /* 2*(int)rate */);
int jsdr_fir_create(jsdr_ctx *ctx, int nchan, int max_block_samples, jsdr_fir **out);
int jsdr_fir_destroy(jsdr_fir *f);
int jsdr_fir_set_weights(jsdr_fir *f, int chan, const double w[21]);
int jsdr_fir_filter_i32(jsdr_fir *f, const int32_t *in, int nsamples, int64_t chan_stride,
                        int32_t *out /* nchan*nsamples */, int mem);
int jsdr_fir_complex_mod_i32(jsdr_ctx *ctx, const int32_t *a, const int32_t *b, int32_t *out,
                             int64_t npairs, int mem);

/* ------------------------------------------------------------- constant tables
 * The constants the library builds for itself, readable without a device so that the
 * reference-pinning tests can compare EVERY entry with the literals of the Java sources:
 *   jsdr_probe_table  which = 0 Partab[256] (FECDecoder.java:40-57), 1 Syms[128] (:105-114),
 *                     2 Scrambler[320] (:118-139), 3 ALPHA_TO[256] (:145-162),
 *                     4 INDEX_OF[256] (:164-181), 5 RS_poly[16] (:544-546),
 *                     6 SYNC_VECTOR[65] (FUNcubeBPSKDemod.java:79-81); first n entries
 *   jsdr_probe_taps   dsFilter[27] (FUNcubeBPSKDemod.java:27-55) and the 65 distinct taps of
 *                     dmFilter (:58-77, stored twice there)
 */
int jsdr_probe_table(int which, int32_t *out, int n);
int jsdr_probe_taps(double ds27[27], double dm65[65]);
/* The exact wrap thresholds of the tuner-phase replay for one increment (0 < inc < 3.1):
 * th1 = the largest double p in [0, 2pi] for which `tuPhase += inc; if (tuPhase > 2pi)`
 * (FUNcubeBPSKDemod.java:384-386) does NOT wrap from p, th2 the same for the second of two
 * steps whose first did not wrap (-1: wraps from every phase).  Host only. */
int jsdr_probe_scout_thresholds(double inc, double *th1, double *th2);

/* ------------------------------------------------------------------ the pump
 * JavaAudio.run's fan-out (JavaAudio.java:262-304) for a batch: every channel's
 * block goes to the fft handler and to the tuner bank in one call: the FFT + PSD of every
 * block, then the tuner bank over the same resident input, on one stream (the tuner-phase
 * replay of the NEXT call runs beside them on a side stream).  ic/qc are JavaAudio's I/Q
 * DC corrections (JavaAudio.java:281-288), applied to what both handlers see.
 * raw is [nchan][nblocks*n] s16 IQ; psd is
 * [nchan][nblocks][n+2].  With mem == JSDR_MEM_HOST the copies are inside the
 * call (this is bench.py's e2e path).
 */
int jsdr_pump_receive_s16(jsdr_fft *f, jsdr_bpsk *b, const int16_t *raw, int nblocks,
                          int ic, int qc, float *psd, int32_t *peak_bin, int mem);
/* The same fan-out with waterfall.java's paintLine (waterfall.java:90-107, as in
 * jsdr_waterfall_rows) chained behind every block's PSD on the device: what comes back is the
 * ARGB pixel row a waterfall draws, pixels[nchan*nblocks][width], and the two published maxima
 * of fft.java:223-224, peak[nchan*nblocks][2] = {peak Hz, peak dB} — 4*width + 8 bytes per
 * block instead of 4*(n+2).  For consumers that only paint (waterfall.java:28-47). */
int jsdr_pump_waterfall_s16(jsdr_fft *f, jsdr_bpsk *b, const int16_t *raw, int nblocks,
                            int ic, int qc, int width, uint32_t peak_rgb, int32_t *pixels,
                            float *peak, int32_t *peak_bin, int mem);
/* JavaAudio.run's whole fan-out (JavaAudio.java:298-304): fft + demod + tuner bank over one
 * resident [nchan][nblocks*n] batch.  PSD, peak bins and the bank's outputs are those of
 * jsdr_pump_receive_s16; the demod handler (d->nchan == b->nchan, nblocks*n within its
 * max_block_samples) gives what nblocks successive jsdr_demod_receive_audio_s16 calls of n samples
 * per channel give, in its current mode and flags.
 * audio is [nchan][nblocks*n]; max_avg (nullable) is [nchan][nblocks][2], one pair per block. */
int jsdr_pump_demod_s16(jsdr_fft *f, jsdr_bpsk *b, jsdr_demod *d, const int16_t *raw, int nblocks,
                        int ic, int qc, float *psd, int32_t *peak_bin,
                        int16_t *audio, float *max_avg, int mem);

#ifdef __cplusplus
}
#endif
#endif
