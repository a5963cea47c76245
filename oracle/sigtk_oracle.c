/* sigtk_oracle.c -- TEST INFRASTRUCTURE ONLY (CPU restatement, never shipped
 * in the product path; the product fails loudly without its CUDA library).
 *
 * Restates, with every rounding step written as an explicit cast, the
 * arithmetic of the reference's per-read hot path.  Build with
 * -std=c99 -ffp-contract=off (no FMA contraction, FLT_EVAL_METHOD 0), the
 * same floating-point environment as the reference (Makefile:5).
 *
 * PARITY PINNED by tests/test_oracle.py against
 *   - /root/reference/test/event_dna.exp  (committed as tests/golden/event_dna.exp)
 *   - outputs of the compiled, unmodified reference (oracle/_ref) on
 *     test/sp1_dna.blow5 and on seeded synthetic DNA / RNA reads,
 *     committed under tests/golden/ with the generating script.
 */
#define _POSIX_C_SOURCE 200809L
#include "sigtk_oracle.h"

#include <float.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

/* events.c:43-54 */
void orc_params(int rna, orc_params_t *p) {
    if (rna) {
        p->w_short = 7;  p->w_long = 14;
        p->thr_short = 2.5f; p->thr_long = 9.0f; p->peak_height = 1.0f;
    } else {
        p->w_short = 3;  p->w_long = 6;
        p->thr_short = 1.4f; p->thr_long = 9.0f; p->peak_height = 0.2f;
    }
}

/* misc.c:15-32: the three per-read doubles are narrowed to float first
 * (17-19), raw_unit is a float division (26), then float add, float mul (28). */
void orc_pa(const int16_t *raw, uint64_t n, double digitisation, double offset,
            double range, float *pa) {
    const float range_f = (float)range;
    const float dig_f = (float)digitisation;
    const float off_f = (float)offset;
    const float unit = range_f / dig_f;
    for (uint64_t j = 0; j < n; j++) {
        const float shifted = (float)raw[j] + off_f;
        pa[j] = shifted * unit;
    }
}

/* events.c:293-303: sequential double accumulation; the square is a FLOAT
 * product widened afterwards. */
void orc_prefix(const float *pa, uint64_t n, double *S, double *Q) {
    double s = 0.0, q = 0.0;
    S[0] = 0.0;
    Q[0] = 0.0;
    for (uint64_t i = 0; i < n; i++) {
        const float sq = pa[i] * pa[i];
        s = s + (double)pa[i];
        q = q + (double)sq;
        S[i + 1] = s;
        Q[i + 1] = q;
    }
}

/* events.c:315-364 */
void orc_tstat(const double *S, const double *Q, uint64_t n, uint32_t w, float *t) {
    memset(t, 0, n * sizeof(float));
    if (n < 2ull * w || w < 2) return;           /* 328-330 */
    const float wf = (float)w;
    const double wd = (double)wf;
    for (uint64_t i = w; i + w <= n; i++) {      /* 338: w <= i <= n-w */
        /* left window [i-w, i): kept in double (339-344; i==w subtracts S[0]==0) */
        const double sum1 = (i > w) ? S[i] - S[i - w] : S[i];
        const double ssq1 = (i > w) ? Q[i] - Q[i - w] : Q[i];
        /* right window [i, i+w): narrowed to float at once (345-346) */
        const float sum2 = (float)(S[i + w] - S[i]);
        const float ssq2 = (float)(Q[i + w] - Q[i]);
        const float mean1 = (float)(sum1 / wd);  /* double division, then narrow */
        const float mean2 = sum2 / wf;           /* float division */
        const float m1sq = mean1 * mean1;        /* float products */
        const float m2sq = mean2 * mean2;
        const float v2 = ssq2 / wf;              /* float division */
        double acc = ssq1 / wd;                  /* 349-350, left to right in double */
        acc = acc - (double)m1sq;
        acc = acc + (double)v2;
        acc = acc - (double)m2sq;
        float cv = (float)acc;
        cv = fmaxf(cv, FLT_MIN);                 /* 353 */
        const float delta = mean2 - mean1;
        const float scaled = cv / wf;            /* float division inside sqrt() */
        const double num = fabs((double)delta);
        const double den = sqrt((double)scaled);
        t[i] = (float)(num / den);               /* 360 */
    }
}

/* events.c:516-536 */
void orc_det_init(orc_det_t *s, orc_det_t *l) {
    s->masked_to = 0; s->peak_pos = -1; s->peak_value = FLT_MAX; s->valid = 0;
    *l = *s;
}

/* cold start with `at` the first index that is processed (SURVEY 7.3(2)) */
void orc_det_cold(orc_det_t *s, orc_det_t *l, uint64_t at) {
    orc_det_init(s, l);
    if (at > 0) { s->masked_to = at - 1; l->masked_to = at - 1; }
}

/* CASE 1 (391-404): no maximum recorded yet. Track the running minimum until
 * the signal has risen by more than `height` above it. */
static void seek_rise(orc_det_t *d, uint64_t i, float cur, float height) {
    if (cur < d->peak_value) {
        d->peak_value = cur;
    } else if (cur - d->peak_value > height) {
        d->peak_value = cur;
        d->peak_pos = (int64_t)i;
    }
}

uint64_t orc_detect(const float *t1, const float *t2, uint64_t from, uint64_t to,
                    const orc_params_t *p, orc_det_t *s, orc_det_t *l,
                    uint64_t *peaks, uint64_t cap) {
    uint64_t np = 0;
    orc_det_t *det[2] = {s, l};
    const float *sig[2] = {t1, t2};
    const float thr[2] = {p->thr_short, p->thr_long};
    const uint32_t win[2] = {p->w_short, p->w_long};
    for (uint64_t i = from; i < to; i++) {
        for (int k = 0; k < 2; k++) {            /* short first, then long (385-386) */
            orc_det_t *d = det[k];
            if (d->masked_to >= i) continue;     /* 387 */
            const float cur = sig[k][i];
            if (d->peak_pos < 0) {
                seek_rise(d, i, cur, p->peak_height);
                continue;                        /* a 1->2 transition acts from the next i */
            }
            /* CASE 2, 405-437 */
            if (cur > d->peak_value) {
                d->peak_value = cur;
                d->peak_pos = (int64_t)i;
            }
            if (k == 0 && d->peak_value > thr[0]) {   /* 414-422: dominate the long detector */
                l->masked_to = (uint64_t)d->peak_pos + win[0];
                l->peak_pos = -1;
                l->peak_value = FLT_MAX;
                l->valid = 0;
            }
            if (d->peak_value - cur > p->peak_height && d->peak_value > thr[k]) d->valid = 1;
            if (d->valid && (i - (uint64_t)d->peak_pos) > win[k] / 2) {
                if (np < cap) peaks[np] = (uint64_t)d->peak_pos;
                np++;
                d->peak_pos = -1;
                d->peak_value = cur;
                d->valid = 0;
            }
        }
    }
    return np;
}

/* events.c:457-473 */
static void make_event(uint64_t a, uint64_t b, const double *S, const double *Q,
                       uint64_t *start, float *length, float *mean, float *stdv) {
    const float len = (float)(b - a);
    const float dsum = (float)(S[b] - S[a]);     /* narrowed BEFORE the float division */
    const float m = dsum / len;
    const float dsq = (float)(Q[b] - Q[a]);
    const float ex2 = dsq / len;
    const float mm = m * m;
    const float var = ex2 - mm;
    *start = a;
    *length = len;
    *mean = m;
    *stdv = sqrtf(fmaxf(var, 0.0f));
}

/* events.c:475-504 */
uint64_t orc_events(const uint64_t *peaks, uint64_t n_peaks, const double *S,
                    const double *Q, uint64_t n, uint64_t *start, float *length,
                    float *mean, float *stdv) {
    uint64_t ne = 0, a = 0;
    for (uint64_t k = 0; k < n_peaks; k++) {
        const uint64_t p = peaks[k];
        if (!(p > 0 && p < n)) continue;         /* 481-485 */
        make_event(a, p, S, Q, &start[ne], &length[ne], &mean[ne], &stdv[ne]);
        ne++;
        a = p;
    }
    make_event(a, n, S, Q, &start[ne], &length[ne], &mean[ne], &stdv[ne]);
    return ne + 1;
}

int64_t orc_getevents(uint64_t n, const float *pa, int rna, uint64_t cap,
                      uint64_t *start, float *length, float *mean, float *stdv) {
    orc_params_t p;
    orc_params(rna, &p);
    double *S = (double *)malloc((n + 1) * sizeof(double));
    double *Q = (double *)malloc((n + 1) * sizeof(double));
    float *t1 = (float *)malloc((n ? n : 1) * sizeof(float));
    float *t2 = (float *)malloc((n ? n : 1) * sizeof(float));
    uint64_t *peaks = (uint64_t *)malloc((n ? n : 1) * sizeof(uint64_t));
    orc_prefix(pa, n, S, Q);
    orc_tstat(S, Q, n, p.w_short, t1);
    orc_tstat(S, Q, n, p.w_long, t2);
    orc_det_t s, l;
    orc_det_init(&s, &l);
    const uint64_t np = orc_detect(t1, t2, 0, n, &p, &s, &l, peaks, n);
    int64_t ne;
    if (np + 1 > cap) {
        ne = -(int64_t)(np + 1);
    } else {
        ne = (int64_t)orc_events(peaks, np, S, Q, n, start, length, mean, stdv);
    }
    free(peaks); free(t2); free(t1); free(Q); free(S);
    return ne;
}

int64_t orc_event_read(const int16_t *raw, uint64_t n, double digitisation,
                       double offset, double range, int rna, uint64_t cap,
                       uint64_t *start, float *length, float *mean, float *stdv) {
    float *pa = (float *)malloc((n ? n : 1) * sizeof(float));
    orc_pa(raw, n, digitisation, offset, range, pa);
    const int64_t ne = orc_getevents(n, pa, rna, cap, start, length, mean, stdv);
    free(pa);
    return ne;
}

static int cmp_float(const void *a, const void *b) {
    const float x = *(const float *)a, y = *(const float *)b;
    return (x > y) - (x < y);
}

/* cfunc.c:126-159 + stat.h:17-73 (sequential float accumulators; the median
 * is the element of rank n/2, ksort.h:233-259) */
/* jnn.c:176-266 for the raw-sample entry point (jnn.c:269-282, 58-75). The thresholds are mean -/+ 0.75 standard
 * deviations of the clamped signal, both accumulated in float in sample order (stat.h:17-24, 36-44). The segmenter is
 * a counter machine over one bit per sample ("inside the band or not"); it is written here as a switch on that bit
 * and on whether a stretch is open, with the reference's counters:
 *   run   : samples in the open stretch, tolerated outliers included        (c)
 *   grow  : 50 + every inside sample of the record so far                   (w; never reset)
 *   bad   : tolerated outliers of the stretch (< 5)                         (err)
 *   tail  : outliers at the very end of the stretch                         (prev_err)            */
int64_t orc_jnn(const int16_t *raw, uint64_t n, int rna, uint64_t cap, int64_t *xy) {
    if (n == 0) return 0;
    const int ni = (int)n;
    const int window = rna ? 1000 : 150;                 /* jnn.h:24-45 */
    const float stall = rna ? 1.0f : 0.25f;
    const float scale = 0.75f;
    const int tolerated = 5, merge_dist = 50;
    float *sig = (float *)malloc((size_t)ni * sizeof(float));
    float acc = 0.0f;
    for (int i = 0; i < ni; i++) {
        const int v = raw[i];
        sig[i] = v > 1200 ? 1200.0f : v < 0 ? 0.0f : (float)v;
        acc = acc + sig[i];
    }
    const float mean = acc / (float)ni;
    float dev = 0.0f;
    for (int i = 0; i < ni; i++) {
        const float d = sig[i] - mean;
        dev = dev + d * d;
    }
    const float sd = sqrtf(dev / (float)ni);
    const float band = sd * scale;
    const float hi = mean + band, lo = mean - band;

    int open = 0, run = 0, grow = 50, bad = 0, tail = 0, first = 0;
    int64_t n_seg = 0, last_y = 0;
    for (int i = 0; i < ni; i++) {
        const int inside = sig[i] < hi && sig[i] > lo;
        if (inside) {
            if (!open) { open = 1; first = i; }
            run++; grow++; tail = 0;
            if (run >= window && run >= grow && run % grow == 0) bad--;
        } else if (open) {
            if (bad < tolerated) {
                run++; bad++; tail++;
                if (run >= window && run >= grow && run % grow == 0) bad--;
            } else {
                if (run >= window || (n_seg == 0 && (float)run >= (float)window * stall)) {
                    const int stop = i - tail;
                    if (n_seg && first - last_y < merge_dist) {
                        if ((uint64_t)n_seg <= cap) xy[2 * (n_seg - 1) + 1] = stop;
                    } else {
                        if ((uint64_t)n_seg < cap) { xy[2 * n_seg] = first; xy[2 * n_seg + 1] = stop; }
                        n_seg++;
                    }
                    last_y = stop;
                }
                open = 0; run = 0; bad = 0; tail = 0;
            }
        }
    }
    free(sig);
    return (uint64_t)n_seg > cap ? -n_seg : n_seg;
}

/* float mean / stdv in sample order (stat.h:17-24, 36-44) and the n/2-th smallest (stat.h:55-63) of x[0..n) */
static float seq_meanf(const float *x, int n) {
    float acc = 0.0f;
    for (int i = 0; i < n; i++) acc = acc + x[i];
    return acc / (float)n;
}
static float seq_stdvf(const float *x, int n) {
    const float m = seq_meanf(x, n);
    float acc = 0.0f;
    for (int i = 0; i < n; i++) {
        const float d = x[i] - m;
        acc = acc + d * d;
    }
    return sqrtf(acc / (float)n);
}
static float rank_half(const float *x, int n) {
    float *tmp = (float *)malloc((size_t)(n > 0 ? n : 1) * sizeof(float));
    memcpy(tmp, x, (size_t)n * sizeof(float));
    qsort(tmp, (size_t)n, sizeof(float), cmp_float);
    const float v = n > 0 ? tmp[n / 2] : 0.0f;
    free(tmp);
    return v;
}

/* jnn.c:103-175 (jnnv2): the band's lower edge (mean - std_scale * stdv) over a 2000-sample rolling mean of the
 * clamped signal, runs below it, first run of a plausible length. The two adaptor parameter sets of jnn.h:88-102
 * differ only in std_scale and the shortest run: JNNV2_RNA_R9_ADAPTOR 0.5f / 2000, JNNV2_RNA_RNA004_ADAPTOR 0.7f / 500
 * (window 2000, merge distance 1500 and longest run 200000 are common). The RNA004 set is restated from jnn.h as
 * prefix.cu passes it to prefix_walk_kernel; no stored reference output covers it. */
static void adaptor_jnnv2(const int16_t *raw, int64_t n, float std_scale, int shortest, int64_t *x, int64_t *y) {
    const int w = 2000, merge = 1500, longest = 200000;
    if (n <= w) { *x = -1; *y = -1; return; }
    const int nt = (int)n - w;
    float *t = (float *)malloc((size_t)nt * sizeof(float));
    #define CLAMPED(i) (raw[i] > 1200 ? 1200.0f : raw[i] < 0 ? 0.0f : (float)raw[i])
    float run = 0.0f;
    for (int i = 0; i < w; i++) run = run + CLAMPED(i);
    t[0] = run / (float)w;
    for (int i = 1; i < nt; i++) {
        run = run - CLAMPED(i - 1);
        run = run + CLAMPED(i + w - 1);
        t[i] = run / (float)w;
    }
    #undef CLAMPED
    const float mn = seq_meanf(t, nt), sd = seq_stdvf(t, nt);
    const float floor_ = mn - sd * std_scale;
    int below = 0, first = 0, last = 0;
    int64_t n_seg = 0, cap = 64;
    int64_t *sx = (int64_t *)malloc((size_t)cap * 2 * sizeof(int64_t));
    for (int j = 0; j < nt; j++) {
        const float v = t[j];
        if (v < floor_) {
            if (!below) { first = j; below = 1; } else last = j;
        } else if (v > floor_ && below) {
            if (n_seg && first - sx[2 * (n_seg - 1) + 1] < merge) {
                sx[2 * (n_seg - 1) + 1] = last;
            } else {
                if (n_seg == cap) { cap *= 2; sx = (int64_t *)realloc(sx, (size_t)cap * 2 * sizeof(int64_t)); }
                sx[2 * n_seg] = first; sx[2 * n_seg + 1] = last;
                n_seg++;
            }
            first = 0; last = 0; below = 0;
        }
    }
    *x = 0; *y = 0;
    for (int64_t k = 0; k < n_seg; k++) {
        const int64_t len = sx[2 * k + 1] - sx[2 * k];
        if (len > longest || len < shortest) continue;
        *x = sx[2 * k] + w / 2 - 1;
        *y = sx[2 * k + 1] + w / 2 - 1;
        break;
    }
    free(sx); free(t);
}

/* jnn.c:176-266 on pA clamped to [0,1200] (jnn_pa, jnn.c:284-297) with a given band and JNNV1_R9_POLYA
 * (window 250, 30 tolerated outliers, merge distance 200, stall_len 1): only the FIRST segment is wanted (jnn.c:360) */
static void polya_r9(const float *pa, int64_t n, float top, float bot, int64_t *x, int64_t *y) {
    const int window = 250, tolerated = 30, merge = 200;
    const float stall = 1.0f;
    *x = -1; *y = -1;
    int open = 0, run = 0, grow = 50, bad = 0, tail = 0, first = 0;
    int64_t n_seg = 0, sx0 = 0, sy0 = 0, last_y = 0;
    for (int i = 0; i < (int)n; i++) {
        const float v = pa[i] > 1200.0f ? 1200.0f : pa[i] < 0.0f ? 0.0f : pa[i];
        if (v < top && v > bot) {
            if (!open) { open = 1; first = i; }
            run++; grow++; tail = 0;
            if (run >= window && run >= grow && run % grow == 0) bad--;
        } else if (open) {
            if (bad < tolerated) {
                run++; bad++; tail++;
                if (run >= window && run >= grow && run % grow == 0) bad--;
            } else {
                if (run >= window || (n_seg == 0 && (float)run >= (float)window * stall)) {
                    const int stop = i - tail;
                    if (n_seg && first - last_y < merge) {
                        if (n_seg == 1) sy0 = stop;
                    } else {
                        if (n_seg == 0) { sx0 = first; sy0 = stop; }
                        n_seg++;
                    }
                    last_y = stop;
                }
                open = 0; run = 0; bad = 0; tail = 0;
            }
        }
    }
    if (n_seg > 0) { *x = sx0; *y = sy0; }
}

void orc_adaptor_polya_pore(const int16_t *raw, uint64_t n, double digitisation, double offset, double range, int rna,
                int pore, int64_t *pos4, float *st6) {
    for (int k = 0; k < 6; k++) st6[k] = 0.0f;
    pos4[2] = -1; pos4[3] = -1;
    if (pore) adaptor_jnnv2(raw, (int64_t)n, 0.7f, 500, &pos4[0], &pos4[1]);   /* JNNV2_RNA_RNA004_ADAPTOR */
    else adaptor_jnnv2(raw, (int64_t)n, 0.5f, 2000, &pos4[0], &pos4[1]);       /* JNNV2_RNA_R9_ADAPTOR */
    if (pos4[1] <= 0) return;                                  /* cfunc.c:173 */
    float *pa = (float *)malloc((n ? n : 1) * sizeof(float));
    orc_pa(raw, n, digitisation, offset, range, pa);
    const int64_t ax = pos4[0], ay = pos4[1];
    st6[0] = seq_meanf(pa + ax, (int)(ay - ax));
    st6[1] = seq_stdvf(pa + ax, (int)(ay - ax));
    st6[2] = rank_half(pa + ax, (int)(ay - ax));
    if (rna) {                                                  /* cfunc.c:189-190: m_a+30+20, m_a+30-20 in float */
        const float top = (st6[0] + 30) + 20, bot = (st6[0] + 30) - 20;
        polya_r9(pa + ay, (int64_t)n - ay, top, bot, &pos4[2], &pos4[3]);
        if (pos4[3] > 0) {
            const int64_t px = pos4[2] + ay, len = pos4[3] - pos4[2];
            st6[3] = seq_meanf(pa + px, (int)len);
            st6[4] = seq_stdvf(pa + px, (int)len);
            st6[5] = rank_half(pa + px, (int)len);
        }
    }
    free(pa);
}

void orc_adaptor_polya(const int16_t *raw, uint64_t n, double digitisation, double offset, double range, int rna,
                int64_t *pos4, float *st6) {
    orc_adaptor_polya_pore(raw, n, digitisation, offset, range, rna, 0, pos4, st6);
}

/* Shannon entropy in bits of a table of bin counts taken over `total` symbols; terms are subtracted in
 * ascending bin order like ent.c:38-46 (the order matters in the last bits). */
static double bits_of_counts(const uint64_t *cnt, uint32_t bins, uint64_t total) {
    double h = 0.0;
    for (uint32_t k = 0; k < bins; k++) {
        if (cnt[k] == 0) continue;
        const double p = (double)cnt[k] / (double)total;
        h -= p * log2(p);
    }
    return h;
}

/* ent.c:108-151. The reference materialises four arrays per record (int32 copy, zig-zag deltas, the deltas
 * narrowed to int16, two byte planes) and calls entropy() on each; the same four count tables are filled
 * here in one pass. Keys: (uint16)raw[i] for i < n; for i < n-1 the low 16 bits of zigzag32(raw[i]-raw[i-1])
 * with raw[-1] = 0 (ent.c:62,124,128), and that key's high / low byte (ent.c:144-145). */
void orc_ent(const int16_t *raw, uint64_t n, double *out3) {
    out3[0] = out3[1] = out3[2] = 0.0;
    if (n == 0) return;
    uint64_t *tab = (uint64_t *)calloc(65536 * 2 + 512, sizeof(uint64_t));
    uint64_t *c_raw = tab, *c_dlt = tab + 65536, *c_hi = tab + 131072, *c_lo = tab + 131072 + 256;
    int32_t before = 0;
    for (uint64_t i = 0; i < n; i++) {
        const int32_t cur = raw[i];
        c_raw[(uint16_t)raw[i]]++;
        if (i + 1 < n) {
            const int32_t d = cur - before;
            const uint16_t key = (uint16_t)(((uint32_t)d << 1) ^ (uint32_t)(d >> 31));
            c_dlt[key]++;
            c_hi[key >> 8]++;
            c_lo[key & 0xff]++;
        }
        before = cur;
    }
    out3[0] = bits_of_counts(c_raw, 65536, n);
    if (n > 1) {
        out3[1] = bits_of_counts(c_dlt, 65536, n - 1);
        out3[2] = bits_of_counts(c_hi, 256, n - 1) + bits_of_counts(c_lo, 256, n - 1);
    }
    free(tab);
}

void orc_stat(const int16_t *raw, uint64_t n, double digitisation, double offset,
              double range, float *out6) {
    const int ni = (int)n;
    const float nf = (float)ni;
    float *pa = (float *)malloc((n ? n : 1) * sizeof(float));
    orc_pa(raw, n, digitisation, offset, range, pa);

    float acc_r = 0.0f, acc_p = 0.0f;
    for (int i = 0; i < ni; i++) {
        acc_r = acc_r + (float)raw[i];
        acc_p = acc_p + pa[i];
    }
    const float mean_r = acc_r / nf, mean_p = acc_p / nf;

    float dev_r = 0.0f, dev_p = 0.0f;
    for (int i = 0; i < ni; i++) {
        const float dr = (float)raw[i] - mean_r;
        const float dp = pa[i] - mean_p;
        dev_r = dev_r + dr * dr;
        dev_p = dev_p + dp * dp;
    }
    const float std_r = sqrtf(dev_r / nf), std_p = sqrtf(dev_p / nf);

    /* rank n/2 of the raw values by counting */
    uint32_t *hist = (uint32_t *)calloc(65536, sizeof(uint32_t));
    for (int i = 0; i < ni; i++) hist[(uint16_t)(raw[i] + 32768)]++;
    uint64_t rank = (uint64_t)(ni / 2), seen = 0;
    int med_r = 0;
    for (int v = 0; v < 65536; v++) {
        seen += hist[v];
        if (seen > rank) { med_r = v - 32768; break; }
    }
    free(hist);
    qsort(pa, n, sizeof(float), cmp_float);
    const float med_p = ni > 0 ? pa[ni / 2] : 0.0f;
    free(pa);

    out6[0] = mean_r; out6[1] = mean_p; out6[2] = std_r; out6[3] = std_p;
    out6[4] = (float)med_r; out6[5] = med_p;
}

double orc_time_events(const int16_t *samples, const uint64_t *read_off,
                       uint64_t n_reads, const double *digitisation,
                       const double *offset, const double *range, int rna,
                       uint64_t *total_events) {
    uint64_t maxn = 1, nev = 0;
    for (uint64_t r = 0; r < n_reads; r++) {
        const uint64_t n = read_off[r + 1] - read_off[r];
        if (n > maxn) maxn = n;
    }
    uint64_t *st = (uint64_t *)malloc(maxn * sizeof(uint64_t));
    float *ln = (float *)malloc(maxn * sizeof(float));
    float *mn = (float *)malloc(maxn * sizeof(float));
    float *sd = (float *)malloc(maxn * sizeof(float));
    struct timespec a, b;
    clock_gettime(CLOCK_MONOTONIC, &a);
    for (uint64_t r = 0; r < n_reads; r++) {
        const uint64_t n = read_off[r + 1] - read_off[r];
        const int64_t ne = orc_event_read(samples + read_off[r], n, digitisation[r],
                                          offset[r], range[r], rna, maxn, st, ln, mn, sd);
        if (ne > 0) nev += (uint64_t)ne;
    }
    clock_gettime(CLOCK_MONOTONIC, &b);
    free(sd); free(mn); free(ln); free(st);
    if (total_events) *total_events = nev;
    return (double)(b.tv_sec - a.tv_sec) + 1e-9 * (double)(b.tv_nsec - a.tv_nsec);
}

/* ---- svb-zd signal compression (SURVEY 8f rank 1) ---------------------------------------------------------
 * slow5lib stores the raw signal of a BLOW5 record as
 *   uint32 count | ceil(count/4) key bytes (2 bits per value, low bits first) | data bytes
 * where value i = zigzag(raw[i] - raw[i-1]) (raw[-1] = 0, 32-bit arithmetic) takes code+1 little-endian bytes
 * (/root/reference/slow5lib/src/slow5_press.c:1055-1150; thirdparty/streamvbyte/src/streamvbyte_encode.c,
 * streamvbyte_decode.c:30-83; streamvbyte_zigzag.c:5-47). */
uint64_t orc_svbzd_bound(uint64_t n) { return 4u + (n + 3u) / 4u + 4u * n; }

int64_t orc_svbzd_encode(const int16_t *raw, uint64_t n, uint8_t *out, uint64_t cap) {
    if (n > 0xffffffffull || cap < orc_svbzd_bound(n)) return -1;
    const uint32_t count = (uint32_t)n;
    memcpy(out, &count, 4);
    uint8_t *keys = out + 4, *data = keys + (n + 3u) / 4u;
    memset(keys, 0, (size_t)((n + 3u) / 4u));
    int32_t prev = 0;
    for (uint64_t i = 0; i < n; i++) {
        const int32_t cur = raw[i];
        const int32_t d = (int32_t)((uint32_t)cur - (uint32_t)prev);           /* streamvbyte_zigzag.c:21-24 */
        const uint32_t z = ((uint32_t)d + (uint32_t)d) ^ (uint32_t)(d >> 31);  /* streamvbyte_zigzag.c:6-8 */
        prev = cur;
        uint32_t code = z < (1u << 8) ? 0u : z < (1u << 16) ? 1u : z < (1u << 24) ? 2u : 3u;
        for (uint32_t b = 0; b <= code; b++) *data++ = (uint8_t)(z >> (8u * b));
        keys[i >> 2] |= (uint8_t)(code << (2u * (i & 3u)));
    }
    return (int64_t)(data - out);
}

/* returns the number of samples, or -1 when the stream is malformed (length mismatch: slow5_press.c:1103) */
int64_t orc_svbzd_decode(const uint8_t *in, uint64_t n_bytes, int16_t *out, uint64_t cap) {
    if (n_bytes < 4) return -1;
    uint32_t count;
    memcpy(&count, in, 4);
    const uint64_t key_len = ((uint64_t)count + 3u) / 4u;
    if (count > cap || 4u + key_len > n_bytes) return -1;
    const uint8_t *keys = in + 4, *data = keys + key_len, *end = in + n_bytes;
    int32_t prev = 0;
    for (uint64_t i = 0; i < count; i++) {
        const uint32_t code = (keys[i >> 2] >> (2u * (i & 3u))) & 3u;           /* streamvbyte_decode.c:62-75 */
        if (data + code + 1u > end) return -1;
        uint32_t z = 0;
        for (uint32_t b = 0; b <= code; b++) z |= (uint32_t)data[b] << (8u * b);
        data += code + 1u;
        const int32_t d = (int32_t)((z >> 1) ^ (0u - (z & 1u)));                 /* streamvbyte_zigzag.c:27-29 */
        out[i] = (int16_t)((uint32_t)d + (uint32_t)prev);                         /* streamvbyte_zigzag.c:41-46 */
        prev = (int32_t)((uint32_t)prev + (uint32_t)d);
    }
    return data == end ? (int64_t)count : -1;
}
