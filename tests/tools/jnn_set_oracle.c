/* jnn_set_oracle.c -- TEST INFRASTRUCTURE ONLY: the reference's jnn segmenter (jnn.c:176-282, jnn_raw) with every
 * field of jnn_param_t (jnn.h:24-45) general, restated on the CPU sample by sample with the reference's counters.
 * It is oracle/sigtk_oracle.c's orc_jnn with the parameters as arguments: tests/test_jnn_sets.py checks that it
 * equals orc_jnn and the compiled reference's stored stdout for jnn_print's two sets, and the GPU tests compare
 * sgpu_set_jnn's results with it. Build with -std=c99 -ffp-contract=off, like the oracle.
 *
 *   run   : samples in the open stretch, tolerated outliers included        (c)
 *   grow  : corrector + every in-band sample of the record so far          (w; never reset; kept in 64 bits)
 *   bad   : tolerated outliers of the stretch (< error)                    (err)
 *   tail  : outliers at the very end of the stretch                        (prev_err)                             */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

typedef struct {
    int32_t window;
    float stall_len;
    int32_t error, seg_dist, corrector;
    float std_scale;
} orc_jnn_param_t;

/* -> segments (negative: more than cap; xy holds the first cap), *n_dec: how often the corrector decremented err */
static int64_t jnn_core(const int16_t *raw, uint64_t n, const orc_jnn_param_t *p, uint64_t cap, int64_t *xy,
                        int64_t *n_dec) {
    *n_dec = 0;
    if (n == 0) return 0;
    const int ni = (int)n;
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
    const float band = sd * p->std_scale;
    const float hi = mean + band, lo = mean - band;

    int open = 0, run = 0, bad = 0, tail = 0, first = 0;
    int64_t grow = p->corrector, n_seg = 0, last_y = 0;
#define CORRECT() \
    if (run >= p->window && run >= grow && run % grow == 0) { bad--; (*n_dec)++; }
    for (int i = 0; i < ni; i++) {
        const int inside = sig[i] < hi && sig[i] > lo;
        if (inside) {
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
#undef CORRECT
    free(sig);
    return (uint64_t)n_seg > cap ? -n_seg : n_seg;
}

int64_t orc_jnn_set(const int16_t *raw, uint64_t n, const orc_jnn_param_t *p, uint64_t cap, int64_t *xy) {
    int64_t n_dec;
    return jnn_core(raw, n, p, cap, xy, &n_dec);
}

/* orc_jnn_set, counting the corrector's decrements of err */
int64_t orc_jnn_set_counted(const int16_t *raw, uint64_t n, const orc_jnn_param_t *p, uint64_t cap, int64_t *xy,
                            int64_t *n_dec) {
    return jnn_core(raw, n, p, cap, xy, n_dec);
}
