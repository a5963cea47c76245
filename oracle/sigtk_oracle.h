/* sigtk_oracle.h -- TEST INFRASTRUCTURE ONLY.
 *
 * CPU restatement (plain C99) of the reference's per-read raw-signal hot path.
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
 * reference legs may load this library; the product path never does.
 * Parity is PINNED: see tests/test_oracle.py (reference golden files
 * test/event_dna.exp, test/event_rna.exp-style fixtures, and the compiled
 * reference in oracle/_ref on every seeded input).
 */
#ifndef SIGTK_ORACLE_H
#define SIGTK_ORACLE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* detector parameter sets, /root/reference/src/events.c:35-54 */
typedef struct {
    uint32_t w_short, w_long;
    float thr_short, thr_long;
    float peak_height;
} orc_params_t;

/* state of one peak detector between samples, events.c:269-281 */
typedef struct {
    uint64_t masked_to;
    int64_t peak_pos; /* -1 = none */
    float peak_value;
    int32_t valid;
} orc_det_t;

void orc_params(int rna, orc_params_t *p);

/* misc.c:15-32 */
void orc_pa(const int16_t *raw, uint64_t n, double digitisation, double offset,
            double range, float *pa);

/* events.c:293-303: S,Q have n+1 entries */
void orc_prefix(const float *pa, uint64_t n, double *S, double *Q);

/* events.c:315-364 */
void orc_tstat(const double *S, const double *Q, uint64_t n, uint32_t w, float *t);

/* events.c:371-443. Runs samples [from, to) starting from the given states
 * (use orc_det_init for the reference's initial state); appends emitted peak
 * positions to peaks[] (capacity cap) in emission order; returns the number
 * emitted. States are updated in place. */
void orc_det_init(orc_det_t *s, orc_det_t *l);
void orc_det_cold(orc_det_t *s, orc_det_t *l, uint64_t at); /* cold start so that `at` is the first processed index */
uint64_t orc_detect(const float *t1, const float *t2, uint64_t from, uint64_t to,
                    const orc_params_t *p, orc_det_t *s, orc_det_t *l,
                    uint64_t *peaks, uint64_t cap);

/* events.c:457-504. Returns number of events (1 + peaks in (0,n)); zero peaks
 * gives the single event [0,n) (documented divergence: the reference aborts). */
uint64_t orc_events(const uint64_t *peaks, uint64_t n_peaks, const double *S,
                    const double *Q, uint64_t n, uint64_t *start, float *length,
                    float *mean, float *stdv);

/* events.c:553-573 without the dead trimming call. Returns number of events,
 * or -(needed) when cap is too small. */
int64_t orc_getevents(uint64_t n, const float *pa, int rna, uint64_t cap,
                      uint64_t *start, float *length, float *mean, float *stdv);

/* raw -> pA -> events (event_func, cfunc.c:72-83, minus printing) */
int64_t orc_event_read(const int16_t *raw, uint64_t n, double digitisation,
                       double offset, double range, int rna, uint64_t cap,
                       uint64_t *start, float *length, float *mean, float *stdv);

/* stat_func numbers (cfunc.c:126-159, stat.h:17-73) in print order:
 * raw_mean, pa_mean, raw_std, pa_std, raw_median, pa_median */
void orc_stat(const int16_t *raw, uint64_t n, double digitisation, double offset,
              double range, float *out6);

/* `sigtk ent` numbers for one record (ent.c:25-51 entropy, 56-65 zig-zag delta, 108-151 the loop of entmain) in
 * print order: raw_ent, delta_ent, byte_ent. n == 0 gives zeros (the reference crashes there: len-1 wraps). */
void orc_ent(const int16_t *raw, uint64_t n, double *out3);

/* `sigtk jnn` segments of one record: jnn_raw (jnn.c:269-282) = rm_outlier (58-75: clamp to [0,1200]) + jnn_core
 * (176-266) with the parameters jnn_print picks (305-312: JNNV1_DRNA_R9_PARAM for rna, JNNV1_CDNA_R9_PARAM
 * otherwise, jnn.h:24-45). Writes up to cap pairs (x,y) to xy[2k], xy[2k+1]; returns the number of segments
 * (or -(needed) when cap is too small). */
int64_t orc_jnn(const int16_t *raw, uint64_t n, int rna, uint64_t cap, int64_t *xy);

/* `sigtk prefix` numbers of one record (prefix_func cfunc.c:169-234; find_adaptor / jnnv2 jnn.c:103-175 with
 * JNNV2_RNA_R9_ADAPTOR (pore 0) or JNNV2_RNA_RNA004_ADAPTOR (pore 1), jnn.h:88-102; find_polya jnn.c:345-370 = jnn_pa +
 * jnn_core with JNNV1_R9_POLYA jnn.h:47-56). `pore` is what SGPU_PARAM_PORE holds; orc_adaptor_polya is the R9 call
 * (pore 0) with the argument list it has always had.
 * pos[0..1] = adaptor (x, y) as jnnv2 returns them ((0,0): none found, (-1,-1): record not longer than the window),
 * pos[2..3] = poly-A (x, y) relative to the adaptor end ((-1,-1): none / DNA); st[0..2] = mean, stdv, median of the
 * adaptor's pA, st[3..5] of the poly-A's (valid when the respective y > 0). */
void orc_adaptor_polya_pore(const int16_t *raw, uint64_t n, double digitisation, double offset, double range, int rna,
                int pore, int64_t *pos4, float *st6);
void orc_adaptor_polya(const int16_t *raw, uint64_t n, double digitisation, double offset, double range, int rna,
                int64_t *pos4, float *st6);

/* svb-zd signal stream of a BLOW5 record (slow5_press.c:1055-1150, streamvbyte_decode.c:30-83,
 * streamvbyte_zigzag.c): encode returns the stream length in bytes (cap >= orc_svbzd_bound(n)), decode the
 * number of samples; -1 on a malformed stream. */
uint64_t orc_svbzd_bound(uint64_t n);
int64_t orc_svbzd_encode(const int16_t *raw, uint64_t n, uint8_t *out, uint64_t cap);
int64_t orc_svbzd_decode(const uint8_t *in, uint64_t n_bytes, int16_t *out, uint64_t cap);

/* single-thread timing of orc_event_read over a flat batch; returns seconds */
double orc_time_events(const int16_t *samples, const uint64_t *read_off,
                       uint64_t n_reads, const double *digitisation,
                       const double *offset, const double *range, int rna,
                       uint64_t *total_events);

#ifdef __cplusplus
}
#endif
#endif
