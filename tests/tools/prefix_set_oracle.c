/* prefix_set_oracle.c -- TEST INFRASTRUCTURE ONLY: the reference's `sigtk prefix` (prefix_func, cfunc.c:169-234) with
 * every field of its two parameter sets general: jnnv2's adaptor set (jnn.h:88-102) and jnn_core's poly-A set as
 * find_polya uses it (jnn.h:47-56). It is oracle/sigtk_oracle.c's orc_adaptor_polya_pore with the sets as arguments:
 * tests/test_prefix_sets.py checks that it equals orc_adaptor_polya_pore and the compiled reference's stored stdout for
 * the reference's sets, and the GPU tests compare sgpu_set_prefix's results with it. Build with -std=c99
 * -ffp-contract=off, like the oracle.
 *
 * Poly-A counters (jnn.c:192-245):
 *   run   : samples in the open stretch, tolerated outliers included        (c)
 *   grow  : corrector + every in-band sample of the record so far          (w; never reset; kept in 64 bits)
 *   bad   : tolerated outliers of the stretch (< error)                    (err)
 *   tail  : outliers at the very end of the stretch                        (prev_err)                             */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct {
    int32_t window;
    float std_scale;
    int32_t seg_dist, lo_thresh, hi_thresh;
} orc_adaptor_t;
typedef struct {
    int32_t window;
    float stall_len;
    int32_t error, seg_dist, corrector;
} orc_polya_t;

static int cmp_float(const void *a, const void *b) {
    const float x = *(const float *)a, y = *(const float *)b;
    return (x > y) - (x < y);
}
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
    if (n > 0) memcpy(tmp, x, (size_t)n * sizeof(float));
    if (n > 0) qsort(tmp, (size_t)n, sizeof(float), cmp_float);
    const float v = n > 0 ? tmp[n / 2] : 0.0f;
    free(tmp);
    return v;
}

/* jnnv2 (jnn.c:103-175): rolling mean of the clamped signal over a->window samples (a running FLOAT sum), the floor
 * mean - std_scale * stdv of the rolling means, runs below it merged when closer than seg_dist, the first run of a
 * plausible length mapped back by window/2 - 1 */
static void adaptor_jnnv2(const int16_t *raw, int64_t n, const orc_adaptor_t *a, int64_t *x, int64_t *y) {
    const int w = a->window;
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
    const float floor_ = mn - sd * a->std_scale;
    int below = 0, first = 0, last = 0;
    int64_t n_seg = 0, cap = 64;
    int64_t *sx = (int64_t *)malloc((size_t)cap * 2 * sizeof(int64_t));
    for (int j = 0; j < nt; j++) {
        const float v = t[j];
        if (v < floor_) {
            if (!below) { first = j; below = 1; } else last = j;
        } else if (v > floor_ && below) {
            if (n_seg && first - sx[2 * (n_seg - 1) + 1] < a->seg_dist) {
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
        if (len > a->hi_thresh || len < a->lo_thresh) continue;
        *x = sx[2 * k] + w / 2 - 1;
        *y = sx[2 * k + 1] + w / 2 - 1;
        break;
    }
    free(sx); free(t);
}

/* find_polya (jnn.c:352-374): jnn_core (jnn.c:176-266) on pA clamped to [0,1200] (jnn_pa) with the given band; only
 * the FIRST segment is wanted (jnn.c:360). *n_dec: how often the corrector decremented err */
static void polya_set(const float *pa, int64_t n, float top, float bot, const orc_polya_t *p, int64_t *x, int64_t *y,
                      int64_t *n_dec) {
    *x = -1; *y = -1;
    int open = 0, run = 0, bad = 0, tail = 0, first = 0;
    int64_t grow = p->corrector, n_seg = 0, sx0 = 0, sy0 = 0, last_y = 0;
#define CORRECT() \
    if (run >= p->window && run >= grow && run % grow == 0) { bad--; (*n_dec)++; }
    for (int i = 0; i < (int)n; i++) {
        const float v = pa[i] > 1200.0f ? 1200.0f : pa[i] < 0.0f ? 0.0f : pa[i];
        if (v < top && v > bot) {
            if (!open) { open = 1; first = i; }
            run++; grow++; tail = 0;
            CORRECT()
        } else if (open) {
            if (bad < p->error) {
                run++; bad++; tail++;
                CORRECT()
            } else {
                if (run >= p->window || (n_seg == 0 && (float)run >= (float)p->window * p->stall_len)) {
                    const int stop = i - tail;
                    if (n_seg && first - last_y < p->seg_dist) {
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
#undef CORRECT
    if (n_seg > 0) { *x = sx0; *y = sy0; }
}

/* misc.c:15-32 */
static void to_pa(const int16_t *raw, uint64_t n, double digitisation, double offset, double range, float *pa) {
    const float range_f = (float)range, dig_f = (float)digitisation, off_f = (float)offset;
    const float unit = range_f / dig_f;
    for (uint64_t j = 0; j < n; j++) pa[j] = ((float)raw[j] + off_f) * unit;
}

/* prefix_func's numbers of one record: pos4 = adaptor (x, y), poly-A (x, y) relative to the adaptor's end; st6 = mean,
 * stdv, median of the adaptor's pA, then of the poly-A's (valid when the respective y > 0). -> corrector decrements */
int64_t orc_prefix_set(const int16_t *raw, uint64_t n, double digitisation, double offset, double range, int rna,
                       const orc_adaptor_t *a, const orc_polya_t *p, int64_t *pos4, float *st6) {
    int64_t n_dec = 0;
    for (int k = 0; k < 6; k++) st6[k] = 0.0f;
    pos4[2] = -1; pos4[3] = -1;
    adaptor_jnnv2(raw, (int64_t)n, a, &pos4[0], &pos4[1]);
    if (pos4[1] <= 0) return 0;                                /* cfunc.c:173 */
    float *pa = (float *)malloc((n ? n : 1) * sizeof(float));
    to_pa(raw, n, digitisation, offset, range, pa);
    const int64_t ax = pos4[0], ay = pos4[1];
    st6[0] = seq_meanf(pa + ax, (int)(ay - ax));
    st6[1] = seq_stdvf(pa + ax, (int)(ay - ax));
    st6[2] = rank_half(pa + ax, (int)(ay - ax));
    if (rna) {                                                  /* cfunc.c:189-190: m_a+30+20, m_a+30-20 in float */
        const float top = (st6[0] + 30) + 20, bot = (st6[0] + 30) - 20;
        polya_set(pa + ay, (int64_t)n - ay, top, bot, p, &pos4[2], &pos4[3], &n_dec);
        if (pos4[3] > 0) {
            const int64_t px = pos4[2] + ay, len = pos4[3] - pos4[2];
            st6[3] = seq_meanf(pa + px, (int)len);
            st6[4] = seq_stdvf(pa + px, (int)len);
            st6[5] = rank_half(pa + px, (int)len);
        }
    }
    free(pa);
    return n_dec;
}
