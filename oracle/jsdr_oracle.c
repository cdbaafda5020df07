/*
 * jsdr_oracle.c — CPU restatement of java-sdr's IQ front-end arithmetic.
 *
 * TEST INFRASTRUCTURE ONLY — see jsdr_oracle.h for the rules and for the
 * parity status (tables, taps and constants pinned to every literal of the
 * reference; "PARITY UNPINNED" for the FFT, whose arithmetic is JTransforms').
 *
 * Build: gcc -O2 -std=c11 -ffp-contract=off -fno-fast-math -pthread
 * (-ffp-contract=off because Java never fuses a*b+c).
 *
 * file:line citations are relative to the reference checkout.
 */
#define _GNU_SOURCE
#include "jsdr_oracle.h"

#include <limits.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#define TWO_PI (2.0 * M_PI) /* Java: 2.0*Math.PI, same binary64 value */

/* ------------------------------------------------------------------ */
/* Java numeric helpers                                                */
/* ------------------------------------------------------------------ */

/* Java (int)double : NaN -> 0, saturating, truncation toward zero */
static int j_d2i(double d)
{
    if (d != d) return 0;
    if (d >= 2147483647.0) return INT_MAX;
    if (d <= -2147483648.0) return INT_MIN;
    return (int)d;
}

/* Java int multiply: wraps */
static int j_imul(int a, int b)
{
    return (int)((uint32_t)a * (uint32_t)b);
}

/* ------------------------------------------------------------------ */
/* JavaAudio.java:276-293                                              */
/* ------------------------------------------------------------------ */
void orc_s16_to_float(const int16_t *raw, int nframes, int chns, int ic, int qc, float *buf)
{
    int sn = 0;
    const int16_t *p = raw;
    for (int l = 0; l < nframes; l++) {
        int16_t s = *p++;
        s = (int16_t)(s + (int16_t)ic);               /* :282  s += (short)m_ic, 16-bit wrap */
        buf[sn++] = (float)s / (float)32767;          /* :283 */
        if (chns > 1) {
            s = *p++;
            s = (int16_t)(s + (int16_t)qc);           /* :287 */
            buf[sn++] = (float)s / (float)32767;      /* :288 */
        } else {
            buf[sn++] = 0;                            /* :290 */
        }
    }
}

/* ------------------------------------------------------------------ */
/* DFT in binary64 (stands in for JTransforms 2.4 — parity unpinned)   */
/* Stockham autosort, any factorisation, O(n * sum of prime factors).  */
/* ------------------------------------------------------------------ */
static void make_twiddle_f64(double *tw, int n, int inverse)
{
    for (int t = 0; t < n; t++) {
        double a = TWO_PI * (double)t / (double)n;
        tw[2 * t] = cos(a);
        tw[2 * t + 1] = inverse ? sin(a) : -sin(a);
    }
}

static int next_factor(int n)
{
    if (n % 4 == 0) return 4;
    if (n % 2 == 0) return 2;
    for (int p = 3; (long)p * p <= n; p += 2)
        if (n % p == 0) return p;
    return n;
}

void orc_dft_f64(const double *in, double *out, int n, int inverse)
{
    if (n <= 0) return;
    double *tw = (double *)malloc(sizeof(double) * 2 * (size_t)n);
    double *a = (double *)malloc(sizeof(double) * 2 * (size_t)n);
    double *b = (double *)malloc(sizeof(double) * 2 * (size_t)n);
    make_twiddle_f64(tw, n, inverse);
    memcpy(a, in, sizeof(double) * 2 * (size_t)n);
    int ns = 1, rem = n;
    while (rem > 1) {
        int R = next_factor(rem);
        double *v = (double *)malloc(sizeof(double) * 2 * (size_t)R);
        int m = n / R;
        for (int j = 0; j < m; j++) {
            int k = j % ns;
            /* twiddle W(r*k, ns*R) = tw[r*k*(n/(ns*R))] */
            long step = (long)k * (n / (ns * R));
            for (int r = 0; r < R; r++) {
                double xr = a[2 * (j + (long)r * m)], xi = a[2 * (j + (long)r * m) + 1];
                long ti = (step * r) % n;
                double wr = tw[2 * ti], wi = tw[2 * ti + 1];
                v[2 * r] = xr * wr - xi * wi;
                v[2 * r + 1] = xr * wi + xi * wr;
            }
            long j0 = (long)(j / ns) * ns * R + k;
            for (int q = 0; q < R; q++) {
                double sr = 0, si = 0;
                for (int r = 0; r < R; r++) {
                    long ti = ((long)r * q % R) * (n / R);
                    double wr = tw[2 * ti], wi = tw[2 * ti + 1];
                    sr += v[2 * r] * wr - v[2 * r + 1] * wi;
                    si += v[2 * r] * wi + v[2 * r + 1] * wr;
                }
                b[2 * (j0 + (long)q * ns)] = sr;
                b[2 * (j0 + (long)q * ns) + 1] = si;
            }
        }
        free(v);
        double *t = a; a = b; b = t;
        ns *= R;
        rem /= R;
    }
    if (inverse) {
        double s = 1.0 / (double)n;
        for (int i = 0; i < 2 * n; i++) a[i] *= s;
    }
    memcpy(out, a, sizeof(double) * 2 * (size_t)n);
    free(tw); free(a); free(b);
}

void orc_dft_direct_f64(const double *in, double *out, int n, int inverse)
{
    for (int k = 0; k < n; k++) {
        double sr = 0, si = 0;
        for (int t = 0; t < n; t++) {
            long kt = ((long)k * t) % n;
            double ang = TWO_PI * (double)kt / (double)n;
            double wr = cos(ang), wi = inverse ? sin(ang) : -sin(ang);
            sr += in[2 * t] * wr - in[2 * t + 1] * wi;
            si += in[2 * t] * wi + in[2 * t + 1] * wr;
        }
        if (inverse) { sr /= n; si /= n; }
        out[2 * k] = sr; out[2 * k + 1] = si;
    }
}

/* float32 Stockham with the plan rebuilt per call (fft.java:194 builds a new
 * FloatFFT_1D every block) — used only as the timed CPU baseline. */
static void dft_f32_plan_per_call(float *x, int n)
{
    float *tw = (float *)malloc(sizeof(float) * 2 * (size_t)n);
    float *b = (float *)malloc(sizeof(float) * 2 * (size_t)n);
    float *a = x;
    for (int t = 0; t < n; t++) {
        double ang = TWO_PI * (double)t / (double)n;
        tw[2 * t] = (float)cos(ang);
        tw[2 * t + 1] = (float)-sin(ang);
    }
    int ns = 1, rem = n;
    while (rem > 1) {
        int R = next_factor(rem);
        int m = n / R;
        float v[2 * 64];
        float *vv = v;
        if (R > 64) vv = (float *)malloc(sizeof(float) * 2 * (size_t)R);
        for (int j = 0; j < m; j++) {
            int k = j % ns;
            long step = (long)k * (n / (ns * R));
            for (int r = 0; r < R; r++) {
                float xr = a[2 * (j + (long)r * m)], xi = a[2 * (j + (long)r * m) + 1];
                long ti = (step * r) % n;
                float wr = tw[2 * ti], wi = tw[2 * ti + 1];
                vv[2 * r] = xr * wr - xi * wi;
                vv[2 * r + 1] = xr * wi + xi * wr;
            }
            long j0 = (long)(j / ns) * ns * R + k;
            if (R == 4) {
                float a0r = vv[0] + vv[4], a0i = vv[1] + vv[5];
                float a1r = vv[0] - vv[4], a1i = vv[1] - vv[5];
                float a2r = vv[2] + vv[6], a2i = vv[3] + vv[7];
                float a3r = vv[2] - vv[6], a3i = vv[3] - vv[7];
                b[2 * j0] = a0r + a2r;                 b[2 * j0 + 1] = a0i + a2i;
                b[2 * (j0 + ns)] = a1r + a3i;          b[2 * (j0 + ns) + 1] = a1i - a3r;
                b[2 * (j0 + 2L * ns)] = a0r - a2r;     b[2 * (j0 + 2L * ns) + 1] = a0i - a2i;
                b[2 * (j0 + 3L * ns)] = a1r - a3i;     b[2 * (j0 + 3L * ns) + 1] = a1i + a3r;
            } else if (R == 2) {
                b[2 * j0] = vv[0] + vv[2];             b[2 * j0 + 1] = vv[1] + vv[3];
                b[2 * (j0 + ns)] = vv[0] - vv[2];      b[2 * (j0 + ns) + 1] = vv[1] - vv[3];
            } else {
                for (int q = 0; q < R; q++) {
                    float sr = 0, si = 0;
                    for (int r = 0; r < R; r++) {
                        long ti = ((long)r * q % R) * (n / R);
                        float wr = tw[2 * ti], wi = tw[2 * ti + 1];
                        sr += vv[2 * r] * wr - vv[2 * r + 1] * wi;
                        si += vv[2 * r] * wi + vv[2 * r + 1] * wr;
                    }
                    b[2 * (j0 + (long)q * ns)] = sr;
                    b[2 * (j0 + (long)q * ns) + 1] = si;
                }
            }
        }
        if (vv != v) free(vv);
        float *t = a; a = b; b = t;
        ns *= R;
        rem /= R;
    }
    if (a != x) { memcpy(x, a, sizeof(float) * 2 * (size_t)n); b = a; }
    free(tw);
    free(b);
}

/* ------------------------------------------------------------------ */
/* fft.java:190-224                                                    */
/* ------------------------------------------------------------------ */
static void psd_from_spectrum(const float *dat, int n, int rate, float *psd, int *peak_bin)
{
    int datlen = 2 * n;
    float cf = 2.0f / (float)n;            /* :199 */
    cf = cf * cf;                          /* :200 */
    float m = -3.4028234663852886e38f;     /* :201 -Float.MAX_VALUE */
    int p = -1;                            /* :202 */
    for (int s = 0; s < datlen - 1; s += 2) {
        float re2 = dat[s] * dat[s];
        float im2 = dat[s + 1] * dat[s + 1];
        float pw = (re2 + im2) * cf;       /* :207 float arithmetic */
        psd[s / 2] = 10.0f * (float)log10((double)pw);
        if (m < psd[s / 2]) {              /* :208 strict, first max wins */
            m = psd[s / 2];
            p = s;
        }
    }
    if (peak_bin) *peak_bin = (p < 0) ? -1 : p / 2;
    if (p < datlen / 2) {                  /* :214 */
        p = j_imul(p, rate) / datlen;      /* :216 int32 wrap, trunc division */
    } else {
        p -= datlen;                       /* :219 */
        p = j_imul(p, rate) / datlen;      /* :220 */
    }
    psd[n] = (float)p;                     /* :223 */
    psd[n + 1] = m;                        /* :224 */
}

void orc_fft_receive(const float *buf, int n, int rate, float *psd, int *peak_bin)
{
    double *x = (double *)malloc(sizeof(double) * 2 * (size_t)n);
    double *X = (double *)malloc(sizeof(double) * 2 * (size_t)n);
    float *dat = (float *)malloc(sizeof(float) * 2 * (size_t)n);
    for (int i = 0; i < 2 * n; i++) x[i] = (double)buf[i];   /* :192 copy */
    orc_dft_f64(x, X, n, 0);                                   /* :194-195 */
    for (int i = 0; i < 2 * n; i++) dat[i] = (float)X[i];
    psd_from_spectrum(dat, n, rate, psd, peak_bin);
    free(x); free(X); free(dat);
}

void orc_fft_power_f64(const float *buf, int n, double *pw)
{
    double *x = (double *)malloc(sizeof(double) * 2 * (size_t)n);
    double *X = (double *)malloc(sizeof(double) * 2 * (size_t)n);
    for (int i = 0; i < 2 * n; i++) x[i] = (double)buf[i];
    orc_dft_f64(x, X, n, 0);
    double cf = 2.0 / (double)n;
    cf *= cf;
    for (int k = 0; k < n; k++) pw[k] = (X[2 * k] * X[2 * k] + X[2 * k + 1] * X[2 * k + 1]) * cf;
    free(x); free(X);
}

/* The same transform with everything a careful CPU implementation would hoist: the twiddle
 * table is built once per (thread, length) instead of per block, the work buffers are kept, and
 * the index arithmetic has no modulo (the twiddle index k*r*(n/(ns*R)) never reaches n).  This
 * is MORE favourable to the CPU than the reference's own code, which constructs a new
 * FloatFFT_1D — plan and tables — for every block (fft.java:194); bench.py times the CPU arm
 * with it so that the GPU/CPU ratio is not inflated by a naive port.  Timing use only. */
static __thread float *tl_tw = NULL, *tl_b = NULL, *tl_dat = NULL;
static __thread int tl_n = 0;
static int g_fft_mode = 0;      /* 0: plan per block (fft.java:194), 1: cached plan (tight) */

void orc_baseline_set_fft_mode(int mode) { g_fft_mode = mode; }

static int largest_factor(int n)
{
    int big = 1;
    while (n > 1) { int f = next_factor(n); if (f > big) big = f; n /= f; }
    return big;
}

static void fft_cache_prepare(int n)
{
    if (tl_n != n) {
        free(tl_tw); free(tl_b); free(tl_dat);
        tl_tw = (float *)malloc(sizeof(float) * 2 * (size_t)n);
        tl_b = (float *)malloc(sizeof(float) * 2 * (size_t)n);
        tl_dat = (float *)malloc(sizeof(float) * 2 * (size_t)n);
        for (int t = 0; t < n; t++) {
            double ang = TWO_PI * (double)t / (double)n;
            tl_tw[2 * t] = (float)cos(ang);
            tl_tw[2 * t + 1] = (float)-sin(ang);
        }
        tl_n = n;
    }
}

static void dft_f32_cached(float *x, int n)
{
    fft_cache_prepare(n);
    const float *tw = tl_tw;
    float *a = x, *b = tl_b;
    int ns = 1, rem = n;
    while (rem > 1) {
        const int R = next_factor(rem);
        const int m = n / R;
        const int tstep = n / (ns * R);
        if (R == 4) {
            for (int jh = 0; jh < m; jh += ns) {
                float *o = b + 2 * ((size_t)jh * 4);
                for (int k = 0; k < ns; k++) {
                    const int j = jh + k;
                    const float *w1 = tw + 2 * (size_t)(k * tstep), *w2 = tw + 2 * (size_t)(2 * k * tstep),
                                *w3 = tw + 2 * (size_t)(3 * k * tstep);
                    const float x0r = a[2 * j], x0i = a[2 * j + 1];
                    const float *p1 = a + 2 * ((size_t)j + m), *p2 = a + 2 * ((size_t)j + 2 * (size_t)m),
                                *p3 = a + 2 * ((size_t)j + 3 * (size_t)m);
                    const float x1r = p1[0] * w1[0] - p1[1] * w1[1], x1i = p1[0] * w1[1] + p1[1] * w1[0];
                    const float x2r = p2[0] * w2[0] - p2[1] * w2[1], x2i = p2[0] * w2[1] + p2[1] * w2[0];
                    const float x3r = p3[0] * w3[0] - p3[1] * w3[1], x3i = p3[0] * w3[1] + p3[1] * w3[0];
                    const float a0r = x0r + x2r, a0i = x0i + x2i, a1r = x0r - x2r, a1i = x0i - x2i;
                    const float a2r = x1r + x3r, a2i = x1i + x3i, a3r = x1r - x3r, a3i = x1i - x3i;
                    o[2 * k] = a0r + a2r;                       o[2 * k + 1] = a0i + a2i;
                    o[2 * (k + ns)] = a1r + a3i;                o[2 * (k + ns) + 1] = a1i - a3r;
                    o[2 * (k + 2 * (size_t)ns)] = a0r - a2r;    o[2 * (k + 2 * (size_t)ns) + 1] = a0i - a2i;
                    o[2 * (k + 3 * (size_t)ns)] = a1r - a3i;    o[2 * (k + 3 * (size_t)ns) + 1] = a1i + a3r;
                }
            }
        } else {
            float v[2 * 64];
            for (int jh = 0; jh < m; jh += ns) {
                for (int k = 0; k < ns; k++) {
                    const int j = jh + k;
                    for (int r = 0; r < R; r++) {
                        const float xr = a[2 * ((size_t)j + (size_t)r * m)], xi = a[2 * ((size_t)j + (size_t)r * m) + 1];
                        const float *w = tw + 2 * (size_t)(k * tstep * r);
                        v[2 * r] = xr * w[0] - xi * w[1];
                        v[2 * r + 1] = xr * w[1] + xi * w[0];
                    }
                    float *o = b + 2 * ((size_t)jh * R + k);
                    if (R == 2) {
                        o[0] = v[0] + v[2];                     o[1] = v[1] + v[3];
                        o[2 * (size_t)ns] = v[0] - v[2];        o[2 * (size_t)ns + 1] = v[1] - v[3];
                    } else {
                        const int qs = n / R;
                        for (int q = 0; q < R; q++) {
                            float sr = 0, si = 0;
                            int ti = 0;
                            for (int r = 0; r < R; r++) {
                                const float *w = tw + 2 * (size_t)ti * qs;
                                sr += v[2 * r] * w[0] - v[2 * r + 1] * w[1];
                                si += v[2 * r] * w[1] + v[2 * r + 1] * w[0];
                                ti += q;
                                if (ti >= R) ti -= R;
                            }
                            o[2 * (size_t)q * ns] = sr;
                            o[2 * (size_t)q * ns + 1] = si;
                        }
                    }
                }
            }
        }
        float *t = a; a = b; b = t;
        ns *= R;
        rem /= R;
    }
    if (a != x) memcpy(x, a, sizeof(float) * 2 * (size_t)n);
}

void orc_fft_receive_f32plan(const float *buf, int n, int rate, float *psd, int *peak_bin)
{
    if (g_fft_mode == 1 && largest_factor(n) <= 64) {
        fft_cache_prepare(n);
        memcpy(tl_dat, buf, sizeof(float) * 2 * (size_t)n);
        dft_f32_cached(tl_dat, n);
        psd_from_spectrum(tl_dat, n, rate, psd, peak_bin);
        return;
    }
    float *dat = (float *)malloc(sizeof(float) * 2 * (size_t)n);
    memcpy(dat, buf, sizeof(float) * 2 * (size_t)n);
    dft_f32_plan_per_call(dat, n);
    psd_from_spectrum(dat, n, rate, psd, peak_bin);
    free(dat);
}

/* ------------------------------------------------------------------ */
/* fir.java:169-228                                                    */
/* ------------------------------------------------------------------ */
void orc_fir_init(orc_fir *s)
{
    memset(s, 0, sizeof(*s));
    s->fof = 20;                                   /* :32 */
}

void orc_fir_weights(orc_fir *s, int f1, int f2, float rate)
{
    if (f1 == INT_MIN && f2 == INT_MIN) {          /* :171 */
        for (int i = 0; i < 21; i++) s->wfir[i] = 0;
        s->wfir[10] = 1;
    } else {
        double df1 = (double)f1 / rate;            /* :177 double / float -> double */
        double df2 = (double)f2 / rate;
        int ord = 20;
        for (int n = 0; n < 21; n++) {
            if (n == ord / 2) {
                s->wfir[n] = 2 * (df2 - df1);      /* :182 */
            } else {
                int d = n - ord / 2;
                s->wfir[n] = (sin(2 * M_PI * df2 * d) / (M_PI * d))
                           - (sin(2 * M_PI * df1 * d) / (M_PI * d));      /* :185-186 */
            }
            s->wfir[n] = s->wfir[n] * (0.54 - 0.46 * cos(2 * M_PI * n / ord)); /* :188 */
        }
    }
    for (int i = 0; i < 21; i++) s->fir[i] = 0;    /* :192-193 */
    s->fof = 20;
}

int orc_fir_filter(orc_fir *s, int in)
{
    s->fir[s->fof] = in;                           /* :200 */
    double o = 0;
    for (int i = 0; i < 21; i++) {
        int ti = (s->fof + i) % 21;
        o = o + s->fir[ti] * s->wfir[i];           /* :205 int*double, separate add */
    }
    s->fof = s->fof - 1;
    if (s->fof < 0) s->fof = 20;
    return j_d2i(o);                               /* :210 (int)o */
}

void orc_fir_filter_block(orc_fir *s, const int *in, int *out, int n)
{
    for (int i = 0; i < n; i++) out[i] = orc_fir_filter(s, in[i]);
}

void orc_fir_complex_gen(int sig[2], int wav[2], float rate)
{
    /* :222 (2*Math.PI*wav[0]*wav[1])/fmt.getSampleRate(), left to right */
    double w = (((2 * M_PI) * wav[0]) * wav[1]) / rate;
    sig[0] = j_d2i(cos(w) * 4096);
    sig[1] = j_d2i(sin(w) * 4096);
    wav[1] += 1;
    if (wav[1] >= (int)rate) wav[1] = 0;
}

void orc_fir_complex_mod(const int a[2], const int b[2], int out[2])
{
    out[0] = (int)((uint32_t)j_imul(a[0], b[0]) - (uint32_t)j_imul(a[1], b[1]));  /* :216 */
    out[1] = (int)((uint32_t)j_imul(a[0], b[1]) + (uint32_t)j_imul(a[1], b[0]));  /* :217 */
}

/* ------------------------------------------------------------------ */
/* demod.java:341-434                                                  */
/* ------------------------------------------------------------------ */
void orc_demod_init(orc_demod *s, int rate)
{
    memset(s, 0, sizeof(*s));
    s->rate = rate;        /* taps all zero, fof = 0 until weights() runs (Q5) */
}

void orc_demod_weights(orc_demod *s, int flo, int fhi)
{
    if (flo == INT_MIN) {                           /* :343 */
        for (int i = 0; i < 21; i++) s->wfir[i] = 0;
        s->wfir[10] = 1;
    } else {
        float rate = (float)s->rate;                /* :350 */
        float nlo = (float)flo / rate;
        float nhi = (float)fhi / rate;
        int ord = 20;
        for (int n = 0; n < 21; n++) {
            if (n == ord / 2) {
                s->wfir[n] = 2.0f * (nhi - nlo);    /* :358 float */
            } else {
                s->wfir[n] = (float)(
                    (sin(2 * M_PI * nhi * (double)(n - ord / 2)) / (M_PI * (double)(n - ord / 2)))
                  - (sin(2 * M_PI * nlo * (double)(n - ord / 2)) / (M_PI * (double)(n - ord / 2))));
            }
            s->wfir[n] *= (float)(0.54 - 0.46 * cos(2 * M_PI * (double)n / (double)ord)); /* :365 */
        }
        s->phi = (float)(2 * M_PI * nlo);           /* :368 */
        s->car = 0.0f;
    }
    for (int i = 0; i < 42; i++) s->fir[i] = 0.0f;
    s->fof = 40;                                    /* :374 */
}

static int demod_filter(const float in[2], float out[2], float *buf, const float *w, int o)
{
    buf[o] = in[0];
    buf[o + 1] = in[1];
    float oi = 0, oq = 0;
    for (int i = 0; i < 42; i += 2) {
        int ti = (o + i) % 42;
        oi = oi + buf[ti] * w[i / 2];               /* :387 float mul, float add */
        oq = oq + buf[ti + 1] * w[i / 2];
    }
    out[0] = oi;
    out[1] = oq;
    o = o - 2;
    if (o < 0) o = 40;
    return o;
}

void orc_demod_receive(orc_demod *s, const float *buf, int nsamples, float *out)
{
    for (int k = 0; k < 2 * nsamples; k += 2) {
        float si = buf[k], sq = buf[k + 1];         /* :412-413 */
        if (s->dofir) {                             /* :415 */
            float fs[2] = { si, sq }, os[2] = { 0, 0 };
            s->fof = demod_filter(fs, os, s->fir, s->wfir, s->fof);
            si = os[0]; sq = os[1];
        }
        if (s->dodwn) {                             /* :423 */
            float ci = (float)cos((double)s->car);
            float cq = (float)sin((double)s->car);
            s->car -= s->phi;
            if (s->car < 0.0f) s->car += (float)(2 * M_PI);
            float a = si, b = sq;
            si = (a * ci - b * cq);                 /* :432 */
            sq = (a * cq + b * ci);                 /* :433 */
        }
        out[k] = si;
        out[k + 1] = sq;
    }
}

/* The value of car seen by each of n samples of orc_demod_receive (:425-426), from car0 on, and
 * the carried value after them in out[n]: the two lines of :427-429 on their own. */
void orc_demod_phases(float phi, float car0, int n, float *out)
{
    float car = car0;
    for (int k = 0; k < n; k++) {
        out[k] = car;
        car -= phi;
        if (car < 0.0f) car += (float)(2 * M_PI);
    }
    out[n] = car;
}

static int j_f2i(float f)                    /* Java (int)float */
{
    if (f != f) return 0;
    if (f >= 2147483648.0f) return INT_MAX;
    if (f <= -2147483648.0f) return INT_MIN;
    return (int)f;
}

void orc_demod_detect(const float *buf, int nsamples, int mode, int rate, int doagc,
                      float lilq[2], int16_t *audio, float max_avg[2])
{
    float *sam = (float *)malloc(sizeof(float) * 2 * (size_t)(nsamples > 0 ? nsamples : 1));
    float max = 0, avg = 0;                                             /* :405-406 */
    float li = lilq[0], lq = lilq[1];
    float fmgain = (float)rate / (mode == 3 ? 5000.0f : 75000.0f);      /* :409 */
    for (int s = 0; s < 2 * nsamples; s += 2) {
        sam[s] = buf[s];
        sam[s + 1] = buf[s + 1];
        if (mode == 0) {                                                /* :441-443 */
            sam[s] = sam[s + 1] = 0;
        } else if (mode == 1) {                                         /* :445-446 */
        } else if (mode == 2) {                                         /* :448-451 */
            float ss = sam[s] * sam[s] + sam[s + 1] * sam[s + 1];
            sam[s] = (float)sqrt((double)ss);
            avg = ((float)(s / 2) * avg + sam[s]) / (float)(s / 2 + 1);
        } else {                                                        /* :453-461 */
            float v = ((li * sam[s + 1]) - (lq * sam[s])) * fmgain;
            li = sam[s];
            lq = sam[s + 1];
            sam[s] = v;
        }
        float a = fabsf(sam[s]);                                        /* :463 Math.max keeps NaN */
        max = (max != max || a != a) ? NAN : (a > max ? a : max);
    }
    if (mode == 2) max -= avg;                                          /* :466-468 */
    for (int s = 0; s < 2 * nsamples; s += 2) {                         /* :471-473 */
        float x = (mode == 2 ? sam[s] - avg : sam[s]) * (doagc ? 1.0f / max : 1.0f);
        audio[s / 2] = (int16_t)(j_f2i(x * 32767.0f) & 0xffff);
    }
    lilq[0] = li;
    lilq[1] = lq;
    max_avg[0] = max;
    max_avg[1] = avg;
    free(sam);
}

void orc_waterfall_row(const float *psd, int n, int width, uint32_t peak_rgb, int32_t *pix)
{
    float h = -2.55f;                                                   /* :92 */
    float step = (float)n / (float)width;                               /* :61 */
    int off = width / 2;                                                /* :62 */
    int pr = (peak_rgb >> 16) & 255, pg = (peak_rgb >> 8) & 255, pb = peak_rgb & 255;
    for (int p = 0; p < width; p++) {
        int o = j_f2i((float)p * step), l = j_f2i(step);
        float r = psd[o];                                               /* getMax :109-116 */
        for (int i = o + 1; i < o + l; i++)
            if (psd[i] > r) r = psd[i];
        int f = 255 - j_f2i(r * h);
        f = f < 0 ? 0 : f;
        f = f > 255 ? 255 : f;
        uint32_t c = 0xff000000u | ((uint32_t)(pr * f / 256) << 16) | ((uint32_t)(pg * f / 256) << 8) | (uint32_t)(pb * f / 256);
        pix[(p + off) % width] = (int32_t)c;
    }
}

/* ------------------------------------------------------------------ */
/* FUNcubeBPSKDemod.java                                               */
/* ------------------------------------------------------------------ */
static const float DS_FILTER_F[27] = {             /* :27-55, F-suffixed literals */
    -6.103515625000e-004F, -1.220703125000e-004F, +2.380371093750e-003F, +6.164550781250e-003F,
    +7.324218750000e-003F, +7.629394531250e-004F, -1.464843750000e-002F, -3.112792968750e-002F,
    -3.225708007813e-002F, -1.617431640625e-003F, +6.463623046875e-002F, +1.502380371094e-001F,
    +2.231445312500e-001F, +2.518310546875e-001F, +2.231445312500e-001F, +1.502380371094e-001F,
    +6.463623046875e-002F, -1.617431640625e-003F, -3.225708007813e-002F, -3.112792968750e-002F,
    -1.464843750000e-002F, +7.629394531250e-004F, +7.324218750000e-003F, +6.164550781250e-003F,
    +2.380371093750e-003F, -1.220703125000e-004F, -6.103515625000e-004F
};
static const float DM_FILTER_F[65] = {             /* :58-67 (table is this, twice) */
    -0.0101130691F, -0.0086975143F, -0.0038246093F, +0.0033563764F, +0.0107237026F, +0.0157790936F, +0.0164594107F, +0.0119213911F,
    +0.0030315224F, -0.0076488191F, -0.0164594107F, -0.0197184277F, -0.0150109226F, -0.0023082460F, +0.0154712381F, +0.0327423589F,
    +0.0424493086F, +0.0379940454F, +0.0154712381F, -0.0243701991F, -0.0750320094F, -0.1244834076F, -0.1568500423F, -0.1553748911F,
    -0.1061032953F, -0.0015013786F, +0.1568500423F, +0.3572048240F, +0.5786381191F, +0.7940228249F, +0.9744923010F, +1.0945250059F,
    +1.1366117829F, +1.0945250059F, +0.9744923010F, +0.7940228249F, +0.5786381191F, +0.3572048240F, +0.1568500423F, -0.0015013786F,
    -0.1061032953F, -0.1553748911F, -0.1568500423F, -0.1244834076F, -0.0750320094F, -0.0243701991F, +0.0154712381F, +0.0379940454F,
    +0.0424493086F, +0.0327423589F, +0.0154712381F, -0.0023082460F, -0.0150109226F, -0.0197184277F, -0.0164594107F, -0.0076488191F,
    +0.0030315224F, +0.0119213911F, +0.0164594107F, +0.0157790936F, +0.0107237026F, +0.0033563764F, -0.0038246093F, -0.0086975143F,
    -0.0101130691F
};
static const int8_t SYNC_VECTOR[65] = {            /* :79-81 */
    1,1,1,1,1,1,1,-1,-1,-1,-1,1,1,1,-1,1,1,1,1,-1,-1,1,-1,1,1,-1,-1,1,-1,-1,1,-1,-1,-1,-1,-1,-1,1,-1,-1,-1,1,-1,-1,1,1,-1,-1,-1,1,-1,1,1,1,-1,1,-1,1,1,-1,1,1,-1,-1,-1
};
#define MATCHED_FILTER_SIZE 65
#define FEC_BITS_SIZE 5200
#define SAMPLES_PER_BIT 8
#define SINCOS_SIZE 256
static const int dmHalfTable[8] = { 4, 5, 6, 7, 0, 1, 2, 3 };   /* :500 */

void orc_sync_vector(int8_t out[65]) { memcpy(out, SYNC_VECTOR, 65); }

void orc_bpsk_default_taps(double *ds27, double *dm65)
{
    if (ds27) for (int i = 0; i < 27; i++) ds27[i] = (double)DS_FILTER_F[i];
    if (dm65) for (int i = 0; i < 65; i++) dm65[i] = (double)DM_FILTER_F[i];
}

int orc_bpsk_sizeof(void) { return (int)sizeof(orc_bpsk); }

void orc_bpsk_init(orc_bpsk *s, int rate, double tuning)
{
    memset(s, 0, sizeof(*s));
    s->rate = rate;
    s->D = rate / 9600;                             /* :476 adsc.rate/DOWN_SAMPLE_RATE */
    for (int n = 0; n < SINCOS_SIZE; n++) {         /* :159-162 */
        s->sinTab[n] = sin(n * 2.0 * M_PI / SINCOS_SIZE);
        s->cosTab[n] = cos(n * 2.0 * M_PI / SINCOS_SIZE);
    }
    s->ds_ntaps = 27;
    for (int i = 0; i < 27; i++) s->dsFilter[i] = (double)DS_FILTER_F[i];
    s->dsPos = s->ds_ntaps - 1;                     /* :468 */
    s->dmPos = MATCHED_FILTER_SIZE - 1;             /* :496 */
    s->dmEnergyOut = 1.0;                           /* :499 */
    s->stages = 3;
    orc_bpsk_set_tuning(s, tuning);
}

void orc_bpsk_set_ds_filter(orc_bpsk *s, const double *taps, int ntaps)
{
    s->ds_ntaps = ntaps;
    for (int i = 0; i < ntaps; i++) s->dsFilter[i] = taps[i];
    memset(s->dsBuf, 0, sizeof(s->dsBuf));
    s->dsPos = ntaps - 1;
    s->dsCnt = 0;
}

void orc_bpsk_set_tuning(orc_bpsk *s, double tuning)
{
    s->tuning = tuning;
    s->tuPhaseInc = 2.0 * M_PI * tuning / (double)s->rate;   /* :196 */
}

static void RxDemodulate(orc_bpsk *s, double i, double q)
{
    static const double VCO_PHASE_INC = 2.0 * M_PI * 1200.0 / (double)9600;   /* :88 */
    static const double BIT_SMOOTH1 = 1.0 / 200.0;
    static const double BIT_SMOOTH2 = 1.0 / 800.0;
    static const double BIT_PHASE_INC = 1.0 / (double)9600;
    static const double BIT_TIME = 1.0 / (double)1200;

    if (s->cap_ds && s->cap_ds_n < s->cap_ds_max) {
        s->cap_ds[2 * s->cap_ds_n] = i;
        s->cap_ds[2 * s->cap_ds_n + 1] = q;
        s->cap_ds_n++;
    }
    s->vcoPhase += VCO_PHASE_INC;                           /* :511 */
    if (s->vcoPhase > 2.0 * M_PI) s->vcoPhase -= 2.0 * M_PI;
    int ix = j_d2i(s->vcoPhase * (double)SINCOS_SIZE / (2.0 * M_PI)) % SINCOS_SIZE;
    s->dmBuf[s->dmPos][0] = i * s->cosTab[ix];              /* :515 */
    s->dmBuf[s->dmPos][1] = q * s->sinTab[ix];              /* :516 */
    double fi = 0.0, fq = 0.0;
    for (int n = 0; n < MATCHED_FILTER_SIZE; n++) {         /* :519-523 */
        int dmi = (MATCHED_FILTER_SIZE - s->dmPos + n);     /* index into the doubled table */
        double h = (double)DM_FILTER_F[dmi % MATCHED_FILTER_SIZE];
        fi += s->dmBuf[n][0] * h;
        fq += s->dmBuf[n][1] * h;
    }
    s->dmPos--;
    if (s->dmPos < 0) s->dmPos = MATCHED_FILTER_SIZE - 1;

    if (s->cap_dm && s->cap_dm_n < s->cap_dm_max) {
        s->cap_dm[2 * s->cap_dm_n] = fi;
        s->cap_dm[2 * s->cap_dm_n + 1] = fq;
        s->cap_dm_n++;
    }

    s->energy1 = fi * fi + fq * fq;                         /* :534 */
    s->dmEnergy[s->dmBitPos] = (s->dmEnergy[s->dmBitPos] * (1.0 - BIT_SMOOTH1)) + (s->energy1 * BIT_SMOOTH1);
    if (s->dmBitPos == s->dmPeakPos) {                      /* :537 */
        s->dmEnergyOut = (s->dmEnergyOut * (1.0 - BIT_SMOOTH2)) + (s->energy1 * BIT_SMOOTH2);
        double di = -(s->dmLastIQ[0] * fi + s->dmLastIQ[1] * fq);
        double dq = s->dmLastIQ[0] * fq - s->dmLastIQ[1] * fi;
        s->dmLastIQ[0] = fi;
        s->dmLastIQ[1] = fq;
        s->energy2 = sqrt(di * di + dq * dq);               /* :543 */
        if (s->energy2 > 100.0) {                           /* :544 */
            int bit = di < 0.0;                             /* :545 */
            if (s->cap_bits && s->cap_bits_n < s->cap_bits_max) {
                s->cap_bits[s->cap_bits_n] = (int8_t)(bit ? 1 : -1);
                if (s->cap_bit_at) s->cap_bit_at[s->cap_bits_n] = s->cntDS;
                s->cap_bits_n++;
            }
            if (s->do_fec) {
                memmove(s->dmFECCorr, s->dmFECCorr + 1, FEC_BITS_SIZE - 1);   /* :553 */
                s->dmFECCorr[FEC_BITS_SIZE - 1] = (int8_t)(bit ? 1 : -1);
                s->dmCorr = 0;
                for (int n = 0; n < 65; n++) s->dmCorr += s->dmFECCorr[n * 80] * SYNC_VECTOR[n];
                if (s->dmCorr >= 45) {                                        /* :560 */
                    uint8_t fecbits[FEC_BITS_SIZE];
                    for (int n = 0; n < FEC_BITS_SIZE; n++)
                        fecbits[n] = (uint8_t)(s->dmFECCorr[n] == 1 ? 0xc0 : 0x40);
                    s->dmErrBits = orc_fec_decode(fecbits, s->decoded);
                    s->cntFEC++;
                    s->dmMaxCorr = 0;
                    s->decodeOK = s->dmErrBits < 0 ? 0 : 1;
                    s->cntDec += s->decodeOK ? 1 : 0;
                    if (s->decodeOK && s->cap_frames && s->cap_frames_n < s->cap_frames_max) {
                        memcpy(s->cap_frames + 256 * s->cap_frames_n, s->decoded, 256);
                        s->cap_frames_n++;
                    }
                }
                if (s->dmCorr > s->dmMaxCorr) s->dmMaxCorr = s->dmCorr;
            }
            s->cntBit++;
        }
    }
    if (s->dmBitPos == dmHalfTable[s->dmPeakPos])           /* :577 */
        s->dmPeakPos = s->dmNewPeak;
    s->dmBitPos = (s->dmBitPos + 1) % SAMPLES_PER_BIT;
    s->dmBitPhase += BIT_PHASE_INC;                         /* :581 */
    if (s->dmBitPhase >= BIT_TIME) {
        s->dmBitPhase -= BIT_TIME;
        s->dmBitPos = 0;                                    /* :584 */
        double eMax = (double)-1.0e10F;
        for (int n = 0; n < SAMPLES_PER_BIT; n++) {
            if (s->dmEnergy[n] > eMax) {
                s->dmNewPeak = n;
                eMax = s->dmEnergy[n];
            }
        }
    }
    s->cntDS++;
}

static void RxDownSample(orc_bpsk *s, double i, double q)
{
    static const double HOWARD_FUDGE_FACTOR = 0.9 * 32768.0;  /* :469 */
    s->dsBuf[s->dsPos][0] = i;
    s->dsBuf[s->dsPos][1] = q;
    if (++s->dsCnt >= s->D) {                                 /* :476 */
        double fi = 0.0, fq = 0.0;
        for (int n = 0; n < s->ds_ntaps; n++) {               /* :479-483 */
            int dsi = (n + s->dsPos) % s->ds_ntaps;
            fi += s->dsBuf[dsi][0] * s->dsFilter[n];
            fq += s->dsBuf[dsi][1] * s->dsFilter[n];
        }
        s->dsCnt = 0;
        if (s->stages >= 2) {
            RxDemodulate(s, fi * HOWARD_FUDGE_FACTOR, fq * HOWARD_FUDGE_FACTOR);
        } else {
            if (s->cap_ds && s->cap_ds_n < s->cap_ds_max) {
                s->cap_ds[2 * s->cap_ds_n] = fi * HOWARD_FUDGE_FACTOR;
                s->cap_ds[2 * s->cap_ds_n + 1] = fq * HOWARD_FUDGE_FACTOR;
                s->cap_ds_n++;
            }
            s->cntDS++;
        }
    }
    s->dsPos--;
    if (s->dsPos < 0) s->dsPos = s->ds_ntaps - 1;
    s->cntRaw++;
}

static void RxMixTuner(orc_bpsk *s, double i, double q)
{
    s->tuPhase += s->tuPhaseInc;                              /* :384 */
    if (s->tuPhase > 2.0 * M_PI) s->tuPhase -= 2.0 * M_PI;
    if (s->tuPhase > 0.0) {                                   /* :388 */
        int ix = j_d2i(s->tuPhase * (double)SINCOS_SIZE / (2.0 * M_PI)) % SINCOS_SIZE;
        double mi = i * s->cosTab[ix];
        double mq = q * s->sinTab[ix];
        RxDownSample(s, mi, mq);
    } else {
        RxDownSample(s, i, q);
    }
}

void orc_bpsk_receive(orc_bpsk *s, const float *buf, int nsamples)
{
    for (int n = 0; n < nsamples; n++) {                      /* :371-376 */
        double i = (double)buf[n * 2];
        double q = (double)buf[n * 2 + 1];
        RxMixTuner(s, i, q);
    }
}

void orc_bpsk_receive_fft(orc_bpsk *s, const float *buf, int samples)
{
    /* :399-402 float expressions widened to double */
    static const double CFREQ_INV_AVERAGE_FACTOR = (double)(1.0F - (2.0F / (1 + 1)));
    static const double CFREQ_AVERAGE_FACTOR = (double)(2.0F / (1 + 1));
    static const double PSD_INV_AVERAGE_FACTOR = (double)(1.0F - (2.0F / (10 + 1)));
    static const double PSD_AVERAGE_FACTOR = (double)(2.0F / (10 + 1));
    double *fftFwd = (double *)malloc(sizeof(double) * 2 * (size_t)samples);
    double *fftRev = (double *)calloc(2 * (size_t)samples, sizeof(double));
    double *tmp = (double *)malloc(sizeof(double) * 2 * (size_t)samples);
    double *psd = (double *)calloc((size_t)samples, sizeof(double));
    double *avePsd = (double *)calloc((size_t)samples, sizeof(double));
    for (int n = 0; n < samples; n++) {
        fftFwd[2 * n] = (double)buf[n * 2];
        fftFwd[2 * n + 1] = (double)buf[n * 2 + 1];
    }
    orc_dft_f64(fftFwd, tmp, samples, 0);                     /* :422-423 */
    memcpy(fftFwd, tmp, sizeof(double) * 2 * (size_t)samples);
    for (int i = 0; i < samples / 2; i++)                     /* :425-427 */
        psd[i] = sqrt(fftFwd[2 * i] * fftFwd[2 * i] + fftFwd[2 * i + 1] * fftFwd[2 * i + 1]);
    double maxBin = 0.0;
    int binPos = -1;
    int beg = s->doUp ? samples / 4 : 0;
    int end = s->doUp ? samples / 2 : samples / 4;
    avePsd[0] = 0;
    for (int i = beg + 75; i < end - 75; i++) {               /* :433-443 */
        avePsd[i] = 0;
        for (int j = i - 50; j < i + 50; j++) avePsd[i] += psd[j];
        if (maxBin < avePsd[i]) {
            maxBin = avePsd[i];
            binPos = i;
        }
    }
    if (s->centreBin < 0) s->centreBin = 0;
    if (s->centreBin > end - 1) s->centreBin = end - 1;
    s->avePeakPower = (PSD_AVERAGE_FACTOR * avePsd[s->centreBin]) + (PSD_INV_AVERAGE_FACTOR * s->avePeakPower);
    if (maxBin > (s->avePeakPower / 4) * 5 && binPos > 0) {   /* :447 */
        s->aveCentreBin = (CFREQ_AVERAGE_FACTOR * (float)binPos) + (CFREQ_INV_AVERAGE_FACTOR * s->aveCentreBin);
        s->centreBin = j_d2i(s->aveCentreBin + 1.0F);
    }
    if (s->centreBin < 102) s->centreBin = 102;               /* :453 */
    memcpy(fftRev, fftFwd + 2 * (s->centreBin - 102), sizeof(double) * 2 * 204);   /* :458 */
    orc_dft_f64(fftRev, tmp, samples, 1);                     /* :459 complexInverse(.., true) */
    for (int i = 0; i < samples; i++)                         /* :461-463 */
        RxDownSample(s, tmp[2 * i], tmp[2 * i]);              /* yes, Q is dropped */
    free(fftFwd); free(fftRev); free(tmp); free(psd); free(avePsd);
}

/* ------------------------------------------------------------------ */
/* FECDecoder.java (AO-40 FEC)                                         */
/* ------------------------------------------------------------------ */
#define RS_NN 255
#define RS_KK 223
#define RS_NROOTS 32
#define RS_FCR 112
#define RS_PRIM 11
#define RS_IPRIM 116
#define RS_A0 RS_NN
#define RS_BLOCKS 2
#define RS_PAD 95
#define VK 7
#define CPOLYA 0x4f
#define CPOLYB 0x6d
#define NBITS ((256 + RS_NROOTS * RS_BLOCKS) * 8 + VK - 1)
#define IL_ROWS 80
#define IL_COLS 65
#define SYNC_POLY 0x48

/* The reference carries these as literal tables (:40-57, :105-181); here
 * they are generated from their defining polynomials and self-checked in
 * the tests against spot values read from the reference tables. */
static uint8_t Partab[256];
static int mettab[2][256];
static int Syms[128];
static uint8_t Scrambler[320];
static int ALPHA_TO[256], INDEX_OF[256];
static int RS_poly[16];
static int tables_ready = 0;

static int parity8(int x) { x ^= x >> 4; x ^= x >> 2; x ^= x >> 1; return x & 1; }

static int mod255(int x)
{
    while (x >= 255) { x -= 255; x = (x >> 8) + (x & 255); }
    return x;
}

/* literal metric table of FECDecoder.java:67-100 (it is not generated by a
 * closed form in the reference, so it is carried as data; mettab[1][i] ==
 * mettab[0][255-i] except the clipped ends, see init) */
static const short METTAB0[256] = {
     20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,
     20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,
     20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,
     20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,
     20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,
     20,   20,   20,   20,   20,   20,   20,   19,   19,   19,   19,   19,   19,   19,   19,   19,
     19,   19,   18,   18,   18,   18,   18,   18,   17,   17,   17,   16,   16,   16,   15,   15,
     14,   14,   13,   13,   12,   11,   10,   10,    9,    8,    7,    6,    5,    3,    2,    1,
     -1,   -2,   -4,   -5,   -7,   -9,  -11,  -13,  -15,  -17,  -19,  -21,  -23,  -25,  -28,  -30,
    -32,  -35,  -37,  -40,  -42,  -45,  -47,  -50,  -52,  -55,  -58,  -60,  -63,  -66,  -68,  -71,
    -74,  -77,  -79,  -82,  -85,  -88,  -90,  -93,  -96,  -99, -102, -104, -107, -110, -113, -116,
   -119, -121, -124, -127, -130, -133, -136, -138, -141, -144, -147, -150, -153, -155, -158, -161,
   -164, -167, -170, -172, -175, -178, -181, -184, -187, -190, -192, -195, -198, -201, -204, -207,
   -210, -212, -215, -218, -221, -224, -227, -229, -232, -235, -238, -241, -244, -247, -249, -252,
   -255, -258, -261, -264, -267, -269, -272, -275, -278, -281, -284, -286, -289, -292, -295, -298,
   -301, -304, -306, -309, -312, -315, -318, -320, -324, -326, -329, -332, -335, -337, -341, -372
};
static const short METTAB1[256] = {
   -372, -341, -338, -335, -332, -329, -326, -324, -321, -318, -315, -312, -309, -306, -304, -301,
   -298, -295, -292, -289, -286, -284, -281, -278, -275, -272, -269, -267, -264, -261, -258, -255,
   -252, -249, -247, -244, -241, -238, -235, -232, -229, -227, -224, -221, -218, -215, -212, -210,
   -207, -204, -201, -198, -195, -192, -190, -187, -184, -181, -178, -175, -172, -170, -167, -164,
   -161, -158, -155, -153, -150, -147, -144, -141, -138, -136, -133, -130, -127, -124, -121, -119,
   -116, -113, -110, -107, -104, -102,  -99,  -96,  -93,  -90,  -88,  -85,  -82,  -79,  -77,  -74,
    -71,  -68,  -66,  -63,  -60,  -58,  -55,  -52,  -50,  -47,  -45,  -42,  -40,  -37,  -35,  -32,
    -30,  -28,  -25,  -23,  -21,  -19,  -17,  -15,  -13,  -11,   -9,   -7,   -5,   -4,   -2,   -1,
      1,    2,    3,    5,    6,    7,    8,    9,   10,   10,   11,   12,   13,   13,   14,   14,
     15,   15,   16,   16,   16,   17,   17,   17,   18,   18,   18,   18,   18,   18,   19,   19,
     19,   19,   19,   19,   19,   19,   19,   19,   19,   20,   20,   20,   20,   20,   20,   20,
     20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,
     20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,
     20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,
     20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,
     20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20,   20
};

static void fec_tables(void)
{
    if (tables_ready) return;
    for (int i = 0; i < 256; i++) Partab[i] = (uint8_t)parity8(i);
    for (int i = 0; i < 256; i++) { mettab[0][i] = METTAB0[i]; mettab[1][i] = METTAB1[i]; }
    /* Syms[s] (:105-114): symbol pair for encoder state s; the second
     * encoder symbol is inverted (:564) */
    for (int s = 0; s < 128; s++)
        Syms[s] = (parity8(s & CPOLYA) << 1) | (1 - parity8(s & CPOLYB));
    /* GF(256), field polynomial x^8+x^7+x^2+x+1 (0x187) — ALPHA_TO[8]=0x87 (:146) */
    int sr = 1;
    for (int i = 0; i < 255; i++) {
        ALPHA_TO[i] = sr;
        INDEX_OF[sr] = i;
        sr <<= 1;
        if (sr & 0x100) sr ^= 0x187;
    }
    ALPHA_TO[255] = 0;
    INDEX_OF[0] = RS_A0;
    /* CCSDS pseudo-randomiser h(x)=x^8+x^7+x^5+x^3+1, all-ones start, MSB
     * first (:118-139; first bytes ff 48 0e c0 9a) */
    {
        int st = 0xff;
        for (int i = 0; i < 320; i++) {
            int byte = 0;
            for (int b = 0; b < 8; b++) {
                byte = (byte << 1) | ((st >> 7) & 1);
                int fb = ((st >> 7) ^ (st >> 4) ^ (st >> 2) ^ st) & 1;
                st = ((st << 1) | fb) & 0xff;
            }
            Scrambler[i] = (uint8_t)byte;
        }
    }
    /* RS generator polynomial, roots alpha^(PRIM*(FCR+i)), index form,
     * first 16 of the palindromic 33 coefficients (:544-546) */
    {
        int g[RS_NROOTS + 1];
        memset(g, 0, sizeof(g));
        g[0] = 1;
        int root = RS_FCR * RS_PRIM;
        for (int i = 0; i < RS_NROOTS; i++, root += RS_PRIM) {
            g[i + 1] = 1;
            for (int j = i; j > 0; j--) {
                if (g[j] != 0) g[j] = g[j - 1] ^ ALPHA_TO[mod255(INDEX_OF[g[j]] + root)];
                else g[j] = g[j - 1];
            }
            g[0] = ALPHA_TO[mod255(INDEX_OF[g[0]] + root)];
        }
        /* the encoder uses RS_poly[j] for taps j+1 and 31-j, and [15] for tap 16 */
        for (int j = 0; j < 16; j++) RS_poly[j] = INDEX_OF[g[j + 1]];
    }
    tables_ready = 1;
}

/* exposed for the table self-check test */
int orc_fec_table_probe(int which, int idx)
{
    fec_tables();
    switch (which) {
    case 0: return Partab[idx];
    case 1: return Syms[idx];
    case 2: return Scrambler[idx];
    case 3: return ALPHA_TO[idx];
    case 4: return INDEX_OF[idx];
    case 5: return RS_poly[idx];
    case 6: return mettab[0][idx];
    case 7: return mettab[1][idx];
    }
    return -1;
}

static int decode_rs_8(uint8_t *data);
int orc_rs_decode(uint8_t data[255])
{
    fec_tables();
    return decode_rs_8(data);
}

void orc_fec_sync_lfsr(uint8_t out[65])
{
    fec_tables();
    int sr = 0x7f;                                         /* :600 */
    for (int i = 0; i < 65; i++) {
        out[i] = (sr & 64) ? 1 : 0;
        sr = (sr << 1) | Partab[sr & SYNC_POLY];           /* :604 (only low 8 bits matter) */
    }
}

typedef struct {
    int Nbytes, Bindex, Conv_sr;
    int RS_block[RS_BLOCKS][RS_NROOTS];
    uint8_t *reencode;
} enc_t;

static void interleave_symbol(enc_t *e, int c)
{
    int col = e->Bindex / IL_COLS;                         /* :551 */
    int row = e->Bindex % IL_COLS;
    if (c) e->reencode[row * IL_ROWS + col] = 1;
    e->Bindex++;
}

static void encode_and_interleave(enc_t *e, int c, int cnt)
{
    while (cnt-- != 0) {
        /* :561-562.  Java keeps c in an int, so c>>7 carries already-shifted
         * bits as well; OR-ing them into Conv_sr is idempotent (they sit at
         * the positions they were shifted to), so one bit per step is the
         * same stream — as in Karn's unsigned-char original. */
        e->Conv_sr = ((e->Conv_sr << 1) | ((c >> 7) & 1)) & 0xff;
        c = (c << 1) & 0xff;
        interleave_symbol(e, Partab[e->Conv_sr & CPOLYA]);
        interleave_symbol(e, 1 - Partab[e->Conv_sr & CPOLYB]);
    }
}

static void scramble_and_encode(enc_t *e, int c)
{
    c ^= Scrambler[e->Nbytes];
    encode_and_interleave(e, c, 8);
}

void orc_fec_encode(const uint8_t data[256], uint8_t sym[5200])
{
    fec_tables();
    enc_t e;
    memset(&e, 0, sizeof(e));
    e.reencode = sym;
    e.Bindex = IL_COLS;                                    /* :589 */
    memset(sym, 0, 5200);
    int sr = 0x7f;
    for (int i = 0; i < 65; i++) {                         /* :600-605 */
        if (sr & 64) sym[IL_ROWS * i] = 1;
        sr = (sr << 1) | Partab[sr & SYNC_POLY];
        sr &= 0xff;
    }
    for (int i = 0; i < 256; i++) {                        /* :614-655 local_encode_byte */
        int c = data[i];
        int rsi = e.Nbytes & 1;
        int feedback = INDEX_OF[c ^ e.RS_block[rsi][0]];
        if (feedback != RS_A0) {
            for (int j = 0; j < 15; j++) {
                int t = ALPHA_TO[mod255(feedback + RS_poly[j])];
                e.RS_block[rsi][j + 1] ^= t;
                e.RS_block[rsi][31 - j] ^= t;
            }
            e.RS_block[rsi][16] ^= ALPHA_TO[mod255(feedback + RS_poly[15])];
        }
        for (int k = 0; k < 31; k++) e.RS_block[rsi][k] = e.RS_block[rsi][k + 1];
        e.RS_block[rsi][31] = (feedback != RS_A0) ? ALPHA_TO[feedback] : 0;
        scramble_and_encode(&e, c);
        e.Nbytes++;
    }
    for (int i = 0; i < 64; i++) {                         /* :662-671 local_encode_parity */
        int c = e.RS_block[e.Nbytes & 1][(e.Nbytes - 256) >> 1];
        scramble_and_encode(&e, c);
        if (++e.Nbytes == 320) encode_and_interleave(&e, 0, 6);
    }
}

static void viterbi27(uint8_t *data, const uint8_t *symbols, int nbits)
{
    /* :203-278 */
    int bitcnt = 0, beststate = 0, k = 0, l = 0;
    long long cmetric[64], nmetric[64];
    uint64_t *pp = (uint64_t *)calloc((size_t)nbits * 2, sizeof(uint64_t));
    int mets[4];
    cmetric[0] = 0;
    for (int i = 1; i < 64; i++) cmetric[i] = -999999;
    for (;;) {
        for (int i = 0; i < 4; i++) {
            mets[i] = 0;
            for (int j = 0; j < 2; j++) mets[i] += mettab[(i >> (1 - j)) & 1][symbols[j + k]];
        }
        k += 2;
        uint64_t mask = 1;
        for (int i = 0; i < 64; i += 2) {
            int b1 = mets[Syms[i]];
            long long m0, m1;
            nmetric[i] = m0 = cmetric[i / 2] + b1;
            int b2 = mets[Syms[i + 1]];
            b1 -= b2;
            m1 = cmetric[(i / 2) + (1 << (VK - 2))] + b2;
            if (m1 > m0) { nmetric[i] = m1; pp[l] |= mask; }
            m0 -= b1;
            nmetric[i + 1] = m0;
            m1 += b1;
            if (m1 > m0) { nmetric[i + 1] = m1; pp[l] |= mask << 1; }
            mask <<= 2;
            if ((mask & 0xffffffffULL) == 0) { mask = 1; l++; }
        }
        if (mask != 1) l++;
        if (++bitcnt == nbits) { beststate = 0; break; }
        memcpy(cmetric, nmetric, sizeof(cmetric));
    }
    l -= 2;
    for (int i = 0; i < nbits / 8; i++) data[i] = 0;
    for (int i = nbits - VK; i >= 0; i--) {
        if (pp[l + (beststate >> 5)] & (1ULL << (beststate & 31))) {
            beststate |= (1 << (VK - 1));
            data[i >> 3] |= (uint8_t)(0x80 >> (i & 7));
        }
        beststate >>= 1;
        l -= 2;
    }
    free(pp);
}

static int decode_rs_8(uint8_t *data)
{
    /* :325-519 with no_eras == 0 (the only way the reference calls it, :775) */
    int lambda[RS_NROOTS + 1] = {0}, s[RS_NROOTS];
    int b[RS_NROOTS + 1], t[RS_NROOTS + 1], omega[RS_NROOTS + 1];
    int root[RS_NROOTS], reg[RS_NROOTS + 1], loc[RS_NROOTS];
    int deg_lambda, el, deg_omega, count, r, syn_error;
    for (int i = 0; i < RS_NROOTS; i++) s[i] = data[0];
    for (int j = 1; j < RS_NN; j++)
        for (int i = 0; i < RS_NROOTS; i++) {
            if (s[i] == 0) s[i] = data[j];
            else s[i] = data[j] ^ ALPHA_TO[mod255(INDEX_OF[s[i]] + (RS_FCR + i) * RS_PRIM)];
        }
    syn_error = 0;
    for (int i = 0; i < RS_NROOTS; i++) { syn_error |= s[i]; s[i] = INDEX_OF[s[i]]; }
    if (!syn_error) return 0;
    lambda[0] = 1;
    for (int i = 0; i < RS_NROOTS + 1; i++) b[i] = INDEX_OF[lambda[i]];
    r = 0; el = 0;
    while (++r <= RS_NROOTS) {
        int discr_r = 0;
        for (int i = 0; i < r; i++)
            if (lambda[i] != 0 && s[r - i - 1] != RS_A0)
                discr_r ^= ALPHA_TO[mod255(INDEX_OF[lambda[i]] + s[r - i - 1])];
        discr_r = INDEX_OF[discr_r];
        if (discr_r == RS_A0) {
            memmove(&b[1], b, RS_NROOTS * sizeof(b[0]));
            b[0] = RS_A0;
        } else {
            t[0] = lambda[0];
            for (int i = 0; i < RS_NROOTS; i++) {
                if (b[i] != RS_A0) t[i + 1] = lambda[i + 1] ^ ALPHA_TO[mod255(discr_r + b[i])];
                else t[i + 1] = lambda[i + 1];
            }
            if (2 * el <= r - 1) {
                el = r - el;
                for (int i = 0; i <= RS_NROOTS; i++)
                    b[i] = (lambda[i] == 0) ? RS_A0 : mod255(INDEX_OF[lambda[i]] - discr_r + RS_NN);
            } else {
                memmove(&b[1], b, RS_NROOTS * sizeof(b[0]));
                b[0] = RS_A0;
            }
            memcpy(lambda, t, (RS_NROOTS + 1) * sizeof(t[0]));
        }
    }
    deg_lambda = 0;
    for (int i = 0; i < RS_NROOTS + 1; i++) {
        lambda[i] = INDEX_OF[lambda[i]];
        if (lambda[i] != RS_A0) deg_lambda = i;
    }
    memcpy(&reg[1], &lambda[1], RS_NROOTS * sizeof(reg[0]));
    count = 0;
    for (int i = 1, k = RS_IPRIM - 1; i <= RS_NN; i++, k = mod255(k + RS_IPRIM)) {
        int q = 1;
        for (int j = deg_lambda; j > 0; j--)
            if (reg[j] != RS_A0) { reg[j] = mod255(reg[j] + j); q ^= ALPHA_TO[reg[j]]; }
        if (q != 0) continue;
        root[count] = i;
        loc[count] = k;
        if (++count == deg_lambda) break;
    }
    if (deg_lambda != count) return -1;
    deg_omega = 0;
    for (int i = 0; i < RS_NROOTS; i++) {
        int tmp = 0;
        int j = (deg_lambda < i) ? deg_lambda : i;
        for (; j >= 0; j--)
            if (s[i - j] != RS_A0 && lambda[j] != RS_A0) tmp ^= ALPHA_TO[mod255(s[i - j] + lambda[j])];
        if (tmp != 0) deg_omega = i;
        omega[i] = INDEX_OF[tmp];
    }
    omega[RS_NROOTS] = RS_A0;
    for (int j = count - 1; j >= 0; j--) {
        int num1 = 0;
        for (int i = deg_omega; i >= 0; i--)
            if (omega[i] != RS_A0) num1 ^= ALPHA_TO[mod255(omega[i] + i * root[j])];
        int num2 = ALPHA_TO[mod255(root[j] * (RS_FCR - 1) + RS_NN)];
        int den = 0;
        int lim = deg_lambda < RS_NROOTS - 1 ? deg_lambda : RS_NROOTS - 1;
        for (int i = lim & ~1; i >= 0; i -= 2)
            if (lambda[i + 1] != RS_A0) den ^= ALPHA_TO[mod255(lambda[i + 1] + i * root[j])];
        if (den == 0) return -1;
        if (num1 != 0)
            data[loc[j]] ^= (uint8_t)ALPHA_TO[mod255(INDEX_OF[num1] + INDEX_OF[num2] + RS_NN - INDEX_OF[den])];
    }
    return count;
}

int orc_fec_decode(const uint8_t raw[5200], uint8_t RSdecdata[256])
{
    fec_tables();
    uint8_t symbols[NBITS * 2 + 65 + 3];
    uint8_t vitdecdata[(NBITS - 6) / 8];
    int nRC = 0;
    memset(symbols, 0, sizeof(symbols));
    {   /* :707-723 de-interleave, skipping the sync column */
        int coltop = 0;
        for (int col = 1; col < IL_ROWS; col++) {
            int rowstart = 0;
            for (int row = 0; row < IL_COLS; row++) {
                symbols[coltop + row] = raw[rowstart + col];
                rowstart += IL_ROWS;
            }
            coltop += IL_COLS;
        }
    }
    viterbi27(vitdecdata, symbols, NBITS);                 /* :731 */
    {
        uint8_t rsblocks[RS_BLOCKS][RS_NN];
        int rserrs[RS_BLOCKS];
        memset(rsblocks, 0, sizeof(rsblocks));
        int di = 0, si = 0;
        for (int col = RS_PAD; col < RS_NN; col++)
            for (int row = 0; row < RS_BLOCKS; row++)
                rsblocks[row][col] = (uint8_t)(vitdecdata[di++] ^ Scrambler[si++]);   /* :769 */
        int rs_failures = 0;
        for (int row = 0; row < RS_BLOCKS; row++) {
            rserrs[row] = decode_rs_8(rsblocks[row]);
            rs_failures += (rserrs[row] == -1) ? 1 : 0;
        }
        if (rs_failures == 0) {
            int j = 0;
            for (int col = RS_PAD; col < RS_KK; col++)
                for (int row = 0; row < RS_BLOCKS; row++) RSdecdata[j++] = rsblocks[row][col];
        }
        for (int row = 0; row < RS_BLOCKS; row++)
            if (rserrs[row] == -1) nRC = -1;
    }
    if (nRC >= 0) {                                        /* :831-847 re-encode and count */
        uint8_t reencode[5200];
        orc_fec_encode(RSdecdata, reencode);
        int errors = 0;
        for (int i = 0; i < 5200; i++)
            if (reencode[i] != (raw[i] >> 7)) errors++;
        nRC = errors;
    }
    return nRC;
}

/* ------------------------------------------------------------------ */
/* CPU baseline drivers (pthreads; libgomp is not in this image)       */
/* ------------------------------------------------------------------ */
#include <pthread.h>

typedef struct {
    int tid, nthreads;
    /* fft job */
    const int16_t *raw; int nblocks, n, rate; float *psd;
    /* mixdecim / pipeline job */
    int nchan, nsamples; const double *tuning, *taps; int ntaps; double *out;
    int stages;
} job_t;

static void *fft_worker(void *arg)
{
    job_t *j = (job_t *)arg;
    float *buf = (float *)malloc(sizeof(float) * 2 * (size_t)j->n);
    for (int b = j->tid; b < j->nblocks; b += j->nthreads) {
        orc_s16_to_float(j->raw + (size_t)b * 2 * j->n, j->n, 2, 0, 0, buf);
        orc_fft_receive_f32plan(buf, j->n, j->rate, j->psd + (size_t)b * (j->n + 2), NULL);
    }
    free(buf);
    return NULL;
}

static void *mixdecim_worker(void *arg)
{
    job_t *j = (job_t *)arg;
    int D = j->rate / 9600;
    int nout = j->nsamples / D;
    orc_bpsk *s = (orc_bpsk *)malloc(sizeof(orc_bpsk));
    float *buf = (float *)malloc(sizeof(float) * 2 * 4096);
    for (int c = j->tid; c < j->nchan; c += j->nthreads) {
        orc_bpsk_init(s, j->rate, j->tuning[c]);
        s->stages = j->stages;
        if (j->taps) orc_bpsk_set_ds_filter(s, j->taps, j->ntaps);
        s->cap_ds = j->out + (size_t)c * nout * 2;
        s->cap_ds_max = nout;
        s->cap_ds_n = 0;
        for (int off = 0; off < j->nsamples; off += 4096) {
            int cnt = j->nsamples - off < 4096 ? j->nsamples - off : 4096;
            orc_s16_to_float(j->raw + ((size_t)c * j->nsamples + off) * 2, cnt, 2, 0, 0, buf);
            orc_bpsk_receive(s, buf, cnt);
        }
    }
    free(s);
    free(buf);
    return NULL;
}

static int run_jobs(void *(*fn)(void *), job_t *proto, int nthreads)
{
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 256) nthreads = 256;
    pthread_t th[256];
    job_t jobs[256];
    for (int t = 0; t < nthreads; t++) {
        jobs[t] = *proto;
        jobs[t].tid = t;
        jobs[t].nthreads = nthreads;
        pthread_create(&th[t], NULL, fn, &jobs[t]);
    }
    for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
    return nthreads;
}

int orc_baseline_fft_s16(const int16_t *raw, int nblocks, int n, int rate, float *psd, int nthreads)
{
    job_t j;
    memset(&j, 0, sizeof(j));
    j.raw = raw; j.nblocks = nblocks; j.n = n; j.rate = rate; j.psd = psd;
    return run_jobs(fft_worker, &j, nthreads);
}

int orc_baseline_mixdecim_s16(const int16_t *raw, int nchan, int nsamples, int rate,
                              const double *tuning, const double *taps, int ntaps,
                              double *out, int nthreads)
{
    job_t j;
    memset(&j, 0, sizeof(j));
    j.raw = raw; j.nchan = nchan; j.nsamples = nsamples; j.rate = rate;
    j.tuning = tuning; j.taps = taps; j.ntaps = ntaps; j.out = out; j.stages = 1;
    return run_jobs(mixdecim_worker, &j, nthreads);
}

static void *pipeline_worker(void *arg)
{
    job_t *j = (job_t *)arg;
    const int n = j->n, D = j->rate / 9600;
    const int nout = (j->nblocks * n) / D;
    orc_bpsk *s = (orc_bpsk *)malloc(sizeof(orc_bpsk));
    float *buf = (float *)malloc(sizeof(float) * 2 * (size_t)n);
    for (int c = j->tid; c < j->nchan; c += j->nthreads) {
        orc_bpsk_init(s, j->rate, j->tuning[c]);
        s->stages = 1;
        if (j->taps) orc_bpsk_set_ds_filter(s, j->taps, j->ntaps);
        s->cap_ds = j->out + (size_t)c * nout * 2;
        s->cap_ds_max = nout;
        s->cap_ds_n = 0;
        for (int b = 0; b < j->nblocks; b++) {
            /* JavaAudio.run: convert once, then fan out to the handlers (:276-304) */
            orc_s16_to_float(j->raw + ((size_t)c * j->nblocks + b) * 2 * n, n, 2, 0, 0, buf);
            orc_fft_receive_f32plan(buf, n, j->rate, j->psd + ((size_t)c * j->nblocks + b) * (n + 2), NULL);
            orc_bpsk_receive(s, buf, n);
        }
    }
    free(s);
    free(buf);
    return NULL;
}

int orc_baseline_pipeline_s16(const int16_t *raw, int nchan, int nblocks, int n, int rate,
                              const double *tuning, const double *taps, int ntaps,
                              float *psd, double *ds, int nthreads)
{
    job_t j;
    memset(&j, 0, sizeof(j));
    j.raw = raw; j.nchan = nchan; j.nblocks = nblocks; j.n = n; j.rate = rate;
    j.tuning = tuning; j.taps = taps; j.ntaps = ntaps; j.psd = psd; j.out = ds;
    return run_jobs(pipeline_worker, &j, nthreads);
}
