/*
 * jsdr_oracle.h — CPU restatement of java-sdr's IQ front-end arithmetic.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in the product (libjsdrcuda.so, the
 * host mirror, the Java shim) may include, link or call this.  Only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs use it, and only as the checker / reported CPU baseline.
 *
 * PARITY STATUS (what pins this restatement to the reference; DESIGN.md section 2)
 *   - PINNED to reference data, every entry (tests/test_ref_tables.py against
 *     tests/golden/ref_tables.npz, parsed from the Java sources by
 *     tests/golden/make_ref_tables.py): Partab, mettab, Syms, Scrambler,
 *     ALPHA_TO / INDEX_OF, RS_poly (FECDecoder.java:40-181,544-546), the
 *     decimator and matched-filter taps and SYNC_VECTOR
 *     (FUNcubeBPSKDemod.java:27-81) and the scalar constants — the literal
 *     tables ARE the reference's golden data.  On top of them: the
 *     sync-LFSR (FECDecoder.java:600-605) == SYNC_VECTOR identity and the
 *     encode -> modulate -> demodulate -> FECDecode round trip.
 *   - FIR / NCO / tuner / decimator / matched filter / bit timing / FEC:
 *     a line by line restatement in Java numeric semantics (strict IEEE, no
 *     FMA contraction, float-literal taps widened, (int) saturating casts).
 *     The reference ships no tests or golden OUTPUTS and no JVM exists
 *     here, so outputs are pinned through the tables above, the identities
 *     and first-principles known answers, not through recorded reference runs.
 *   - FFT (fft.java:194-195, FUNcubeBPSKDemod.java:422-423,459): the
 *     arithmetic lives in JTransforms 2.4 (reference Makefile:8), which is
 *     absent from /root/reference.  The oracle is the mathematical DFT in
 *     binary64.  PARITY UNPINNED by any reference artefact (stated as the
 *     task requires); Java's Math.sin/cos/log10 likewise (<= 1 ulp, not run).
 *
 * All file:line citations are relative to the reference checkout.
 */
#ifndef JSDR_ORACLE_H
#define JSDR_ORACLE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- JavaAudio.java:276-293 : s16le -> float with I/Q DC correction ---- */
void orc_s16_to_float(const int16_t *raw, int nframes, int chns, int ic, int qc,
                      float *buf /* 2*nframes */);

/* ---- DFT by definition (binary64), any n ------------------------------- */
/* in/out interleaved re,im.  inverse!=0: e^{+i..} and scaled by 1/n
 * (JTransforms complexInverse(x, true) contract). */
void orc_dft_f64(const double *in, double *out, int n, int inverse);
/* O(n^2) direct sum, for pinning orc_dft_f64 at small n */
void orc_dft_direct_f64(const double *in, double *out, int n, int inverse);

/* ---- fft.java:190-224 : fft.receive ------------------------------------ */
/* psd has n+2 floats; peak_bin (may be NULL) receives the arg-max bin or -1.
 * The transform is done in binary64 and rounded to float before the float
 * PSD arithmetic of fft.java:199-212. */
void orc_fft_receive(const float *buf, int n, int rate, float *psd, int *peak_bin);
/* double-precision path: power*cf per bin in binary64 (no log) */
void orc_fft_power_f64(const float *buf, int n, double *pw);
/* CPU-baseline flavour: float32 transform with the plan (twiddle table)
 * rebuilt on every call, as fft.java:194 does. */
void orc_fft_receive_f32plan(const float *buf, int n, int rate, float *psd, int *peak_bin);

/* ---- fir.java:169-228 -------------------------------------------------- */
typedef struct {
    double wfir[21];
    int fir[21];
    int fof;
} orc_fir;
void orc_fir_init(orc_fir *s);
/* f1==f2==INT32_MIN -> all-pass (fir.java:171-174) */
void orc_fir_weights(orc_fir *s, int f1, int f2, float rate);
int  orc_fir_filter(orc_fir *s, int in);
void orc_fir_filter_block(orc_fir *s, const int *in, int *out, int n);
/* wav[0]=freq, wav[1]=running sample counter (updated) */
void orc_fir_complex_gen(int sig[2], int wav[2], float rate);
void orc_fir_complex_mod(const int a[2], const int b[2], int out[2]);

/* ---- demod.java:341-434 ------------------------------------------------ */
typedef struct {
    float wfir[21];
    float fir[42];
    int fof;
    float car, phi;
    int dofir, dodwn;
    int rate;
} orc_demod;
void orc_demod_init(orc_demod *s, int rate);       /* taps zero, fof=0 (Q5) */
void orc_demod_weights(orc_demod *s, int flo, int fhi); /* flo==INT32_MIN -> all-pass */
/* out = the value of sam[] after the FIR and down-shift stages
 * (what demod.java:436-437 copies to dbg[]) */
void orc_demod_receive(orc_demod *s, const float *buf, int nsamples, float *out);
/* The NCO phase alone (:427-429): out[k] = car used by sample k (k < n) from car0, out[n] = the
 * value carried to the next call.  out holds n + 1 floats. */
void orc_demod_phases(float phi, float car0, int n, float *out);

/* The rest of demod.receive (demod.java:405-481) on the FIR/NCO output `sam` (2n floats):
 * detector per mode (0 off, 1 raw, 2 AM, 3 NFM, 4 WFM; :439-463), max/avg, AGC, s16
 * narrowing (:469-473).  lilq carries li/lq across blocks.  audio: n shorts (one channel of
 * the stereo pair the reference writes); max_avg[0]=max (after the AM fix-up), [1]=avg. */
void orc_demod_detect(const float *sam, int nsamples, int mode, int rate, int doagc,
                      float lilq[2], int16_t *audio, float max_avg[2]);

/* waterfall.paintLine (waterfall.java:90-107): one published psd row (float[n+2]) to `width`
 * ARGB pixels, peak colour 0xRRGGBB. */
void orc_waterfall_row(const float *psd, int n, int width, uint32_t peak_rgb, int32_t *pix);

/* ---- FUNcubeBPSKDemod.java:366-595 ------------------------------------- */
#define ORC_MAX_DS_TAPS 128
typedef struct {
    int rate, D;
    double tuning, tuPhaseInc, tuPhase;
    int ds_ntaps;
    double dsFilter[ORC_MAX_DS_TAPS];
    double dsBuf[ORC_MAX_DS_TAPS][2];
    int dsPos, dsCnt;
    double vcoPhase;
    double dmBuf[65][2];
    int dmPos;
    double dmEnergy[10];
    int dmBitPos, dmPeakPos, dmNewPeak;
    double dmEnergyOut, dmBitPhase, dmLastIQ[2];
    double energy1, energy2;
    int64_t cntRaw, cntDS, cntBit, cntFEC, cntDec;
    int dmCorr, dmMaxCorr, dmErrBits, decodeOK;
    int8_t dmFECCorr[5200];
    uint8_t decoded[256];
    int do_fec;                 /* run the sync correlator + FECDecode (f-1) */
    int stages;                 /* 1: stop after RxDownSample (CPU baseline of mix+FIR); 3: full chain */
    /* auto-tune (doBufferFFT) */
    int doUp;
    double avePeakPower, aveCentreBin;
    int centreBin;
    double sinTab[256], cosTab[256];
    /* per-call capture (caller-owned, may be NULL) */
    double *cap_ds;   int cap_ds_n,  cap_ds_max;   /* (i,q) fed to RxDemodulate */
    double *cap_dm;   int cap_dm_n,  cap_dm_max;   /* matched-filter (fi,fq)    */
    int8_t *cap_bits; int64_t *cap_bit_at; int cap_bits_n, cap_bits_max; /* +-1, cntDS index */
    uint8_t *cap_frames; int cap_frames_n, cap_frames_max; /* decoded 256-byte frames */
} orc_bpsk;
void orc_bpsk_init(orc_bpsk *s, int rate, double tuning);
/* replace the 27-tap decimator by an arbitrary low-pass (config-4 shape) */
void orc_bpsk_set_ds_filter(orc_bpsk *s, const double *taps, int ntaps);
void orc_bpsk_set_tuning(orc_bpsk *s, double tuning);
void orc_bpsk_receive(orc_bpsk *s, const float *buf, int nsamples);      /* doBufferTune */
void orc_bpsk_receive_fft(orc_bpsk *s, const float *buf, int nsamples);  /* doBufferFFT  */
int  orc_bpsk_sizeof(void);
void orc_bpsk_default_taps(double *ds27, double *dm65);
void orc_sync_vector(int8_t out[65]);   /* FUNcubeBPSKDemod.java:79-81 literal */

/* ---- FECDecoder.java --------------------------------------------------- */
void orc_fec_sync_lfsr(uint8_t out[65]);                    /* :600-605 */
void orc_fec_encode(const uint8_t data[256], uint8_t sym[5200]); /* :677-688 */
int  orc_fec_decode(const uint8_t raw[5200], uint8_t out[256]);  /* :703-852 */
int  orc_fec_table_probe(int which, int idx);                     /* table self-check */
int  orc_rs_decode(uint8_t data[255]);                            /* decode_rs_8 :325-519, no erasures */

/* ---- CPU baseline drivers (pthreads over channels / blocks) ------------ */
/* returns the number of threads used */
/* 0 (default): the FFT plan and twiddle table are rebuilt for every block, as fft.java:194 does
 * (new FloatFFT_1D per receive); 1: built once per thread and length, modulo-free loops — more
 * favourable to the CPU than the reference's own code (bench.py's CPU arm uses 1) */
void orc_baseline_set_fft_mode(int mode);
int orc_baseline_fft_s16(const int16_t *raw, int nblocks, int n, int rate, float *psd, int nthreads);
/* the benchmark pipeline per (channel, block): JavaAudio conversion, fft.receive
 * (float plan rebuilt per block) and the tuner + decimator */
int orc_baseline_pipeline_s16(const int16_t *raw, int nchan, int nblocks, int n, int rate,
                              const double *tuning, const double *taps, int ntaps,
                              float *psd /* nchan*nblocks*(n+2) */, double *ds /* nchan*(nblocks*n/D)*2 */,
                              int nthreads);
int orc_baseline_mixdecim_s16(const int16_t *raw, int nchan, int nsamples, int rate,
                              const double *tuning, const double *taps, int ntaps,
                              double *out /* nchan * (nsamples/D) * 2 */, int nthreads);

#ifdef __cplusplus
}
#endif
#endif
