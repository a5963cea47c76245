/* sigtk_main.c -- drop-in `sigtk event | pa | stat | ent | jnn | prefix` on top of the B200 hot path (C99 host).
 * SLOW5 / BLOW5 files are read by blow5.c.
 *
 * Same command line, stdout bytes, stderr information lines and exit codes as the reference tool for the three
 * sub-commands of the raw-signal path:
 *     reference src/main.c:76-123   (command switch, footer)
 *     reference src/cmain.c:40-156  (options -h -n -c -V --version --help --print-stat -o, record iteration,
 *                                    read-id random access)
 *     reference src/cfunc.c:16-159  (output formats of event / pa / stat)
 *     reference src/misc.c:34-101   (DNA/RNA and pore detection from the BLOW5 header)
 *     reference src/cfunc.c:108-120, src/jnn.c:303-343 (`jnn`: line format, long and -c compact)
 *     reference src/ent.c:67-177    (`ent`: its own option set, usage text, header and "%f" line per record)
 * What changes is the execution model: instead of one record -> compute -> printf, decoded records are batched
 * into pinned slots of the CUDA library (include/sigtk_b200.h), several batches are in flight on one or more
 * GPUs, and the per-read results are printed in input order.  There is no CPU implementation of the path in
 * here: without a usable GPU the tool exits with an error.
 * The batch loader and the output path are parallel: records are read serially (blow5_next_bytes); for BLOW5
 * files with svb-zd signal compression the pool only inflates the records (zlib) and the svb-zd streams are decoded
 * on the GPU (--cpu-decode: blow5_decode on the pool, as for every other format); every finished batch is formatted by the same pool with
 * exact re-implementations of the reference's printf conversions (fastfmt.h) and written in input order.
 * Additive options (default off / 1): --gpus N, --batch-samples S, --threads T.
 */
#define _POSIX_C_SOURCE 200809L
#include <getopt.h>
#include <inttypes.h>
#include <pthread.h>
#include <stdint.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/resource.h>
#include <sys/stat.h>
#include <sys/time.h>
#include <unistd.h>

#include "blow5.h"
#include "fastfmt.h"
#include "sigtk_b200.h"

#define SIGTK_VERSION "0.2.0" /* reference src/sigtk.h:11 */

#define INFO(msg, ...) fprintf(stderr, "[%s::INFO]\033[1;34m " msg "\033[0m\n", __func__, __VA_ARGS__)
#define WARNING(msg, ...) \
    fprintf(stderr, "[%s::WARNING]\033[1;33m " msg "\033[0m At %s:%d\n", __func__, __VA_ARGS__, __FILE__, __LINE__ - 1)
#define ERROR(msg, ...) \
    fprintf(stderr, "[%s::ERROR]\033[1;31m " msg "\033[0m At %s:%d\n", __func__, __VA_ARGS__, __FILE__, __LINE__ - 1)

enum { MODE_EVENT, MODE_PA, MODE_STAT, MODE_ENT, MODE_JNN, MODE_PREFIX };

typedef struct {
    int mode;
    int compact;
    int rna;
    int p_stat; /* --print-stat (prefix) */
    int rna004; /* the pore picks jnnv2's parameters for `prefix` (jnn.c:181-188) */
} opt_t;

/* ---- timing footer (reference src/misc.h:19-43) ------------------------------------------------------------- */
static double realtime(void) {
    struct timeval tp;
    gettimeofday(&tp, NULL);
    return (double)tp.tv_sec + (double)tp.tv_usec * 1e-6;
}
static double cputime(void) {
    struct rusage r;
    getrusage(RUSAGE_SELF, &r);
    return (double)r.ru_utime.tv_sec + (double)r.ru_stime.tv_sec + 1e-6 * (double)(r.ru_utime.tv_usec + r.ru_stime.tv_usec);
}
static long peakrss(void) {
    struct rusage r;
    getrusage(RUSAGE_SELF, &r);
    return r.ru_maxrss * 1024;
}

/* ---- header inspection (reference src/misc.c:34-101) ----------------------------------------------------------
 * Both questions the reference asks of the BLOW5 header -- DNA or RNA, which pore -- have the same shape: one
 * attribute of read group 0 decides, a list of substrings maps its value to an answer and an INFO line, the other
 * read groups are only compared with it. The stderr lines are the reference's. */
typedef struct {
    const char *needle; /* substring (pore) or whole value (experiment type) looked for in the attribute */
    int value;
    const char *info;   /* INFO line printed on a match */
} hdr_rule_t;
typedef struct {
    const char *attr;
    const char *missing;      /* WARNING when read group 0 has no such attribute */
    int whole;                /* rules must match the whole value */
    const hdr_rule_t *rules;
    int n_rules;
    int fallback;             /* answer when no rule matches */
    const char *fallback_info;    /* INFO line for the fallback, or NULL: */
    const char *fallback_warning; /* WARNING format taking the value */
    const char *mismatch;     /* WARNING format: other value, first value, group, first value */
} hdr_query_t;

/* the reference's WARNING line (error.h:60-66) for a format that is not a string literal */
static void warn_fmt(const char *func, int line, const char *fmt, ...) {
    va_list ap;
    fprintf(stderr, "[%s::WARNING]\033[1;33m ", func);
    va_start(ap, fmt);
    vfprintf(stderr, fmt, ap);
    va_end(ap);
    fprintf(stderr, "\033[0m At %s:%d\n", __FILE__, line);
}

static int hdr_ask(const blow5_file_t *sp, const hdr_query_t *q) {
    const char *first = blow5_hdr_get(sp, q->attr, 0);
    if (first == NULL) {
        warn_fmt(__func__, __LINE__, "%s", q->missing);
        return 0;
    }
    int answer = q->fallback, hit = 0;
    for (int k = 0; k < q->n_rules && !hit; k++) {
        const hdr_rule_t *r = &q->rules[k];
        if (q->whole ? strcmp(first, r->needle) == 0 : strstr(first, r->needle) != NULL) {
            answer = r->value;
            INFO("%s", r->info);
            hit = 1;
        }
    }
    if (!hit) {
        if (q->fallback_info) INFO("%s", q->fallback_info);
        else warn_fmt(__func__, __LINE__, q->fallback_warning, first);
    }
    for (uint32_t g = 1; g < sp->num_read_groups; g++) {
        const char *other = blow5_hdr_get(sp, q->attr, g);
        if (other && strcmp(other, first)) warn_fmt(__func__, __LINE__, q->mismatch, other, first, (int)g, first);
    }
    return answer;
}

enum { PORE_R9 = 0, PORE_R10 = 1, PORE_RNA004 = 2 }; /* sigtk.h:107-109 */
static int drna_detect(const blow5_file_t *sp) { /* misc.c:34-60 */
    static const hdr_rule_t rules[] = {{"genomic_dna", 0, "DNA data detected."}, {"rna", 1, "RNA data detected."}};
    static const hdr_query_t q = {"experiment_type", "experiment_type not found in SLOW5 header. Assuming genomic_dna", 1,
                                  rules, 2, 0, NULL, "Unknown experiment type: %s. Assuming genomic_dna",
                                  "Experiment type mismatch: %s != %s in read group %d. Defaulted to %s"};
    return hdr_ask(sp, &q);
}
static int pore_detect(const blow5_file_t *sp) { /* misc.c:74-101; only `prefix` uses the answer */
    static const hdr_rule_t rules[] = {{"114", PORE_R10, "R10 data detected."}, {"rna004", PORE_RNA004, "RNA004 data detected."}};
    static const hdr_query_t q = {"sequencing_kit", "sequencing_kit not found in SLOW5 header. Assuming R9.4.1", 0,
                                  rules, 2, PORE_R9, "R9 data detected.", NULL,
                                  "sequencing_kit type mismatch: %s != %s in read group %d. Defaulted to %s"};
    return hdr_ask(sp, &q);
}

/* optional wall-clock breakdown of the host side (SIGTK_PROFILE=1): read, decode, add, wait, format, write */
static double g_prof[10];

/* ---- fork-join thread pool ---------------------------------------------------------------------------------------- */
typedef void (*task_fn)(void *arg, int item);
typedef struct {
    pthread_t *th;
    int n_threads; /* workers besides the caller */
    pthread_mutex_t mu;
    pthread_cond_t go, done;
    task_fn fn;
    void *arg;
    int n_items;
    volatile int next;
    unsigned gen;
    int busy, stop;
} pool_t;

static void pool_work(pool_t *p) {
    for (;;) {
        const int i = __sync_fetch_and_add(&p->next, 1);
        if (i >= p->n_items) break;
        p->fn(p->arg, i);
    }
}
static void *pool_main(void *vp) {
    pool_t *p = (pool_t *)vp;
    unsigned seen = 0;
    pthread_mutex_lock(&p->mu);
    for (;;) {
        while (!p->stop && p->gen == seen) pthread_cond_wait(&p->go, &p->mu);
        if (p->stop) break;
        seen = p->gen;
        pthread_mutex_unlock(&p->mu);
        pool_work(p);
        pthread_mutex_lock(&p->mu);
        if (--p->busy == 0) pthread_cond_signal(&p->done);
    }
    pthread_mutex_unlock(&p->mu);
    return NULL;
}
static void pool_open(pool_t *p, int n_threads) {
    memset(p, 0, sizeof *p);
    pthread_mutex_init(&p->mu, NULL);
    pthread_cond_init(&p->go, NULL);
    pthread_cond_init(&p->done, NULL);
    p->n_threads = n_threads > 1 ? n_threads - 1 : 0;
    p->th = (pthread_t *)calloc((size_t)p->n_threads + 1, sizeof(pthread_t));
    for (int k = 0; k < p->n_threads; k++)
        if (pthread_create(&p->th[k], NULL, pool_main, p) != 0) { p->n_threads = k; break; }
}
/* runs fn(arg, 0..n_items-1) on the pool and the calling thread; returns when all items are done */
static void pool_run(pool_t *p, task_fn fn, void *arg, int n_items) {
    if (n_items <= 0) return;
    p->fn = fn; p->arg = arg; p->n_items = n_items; p->next = 0;
    if (p->n_threads > 0 && n_items > 1) {
        pthread_mutex_lock(&p->mu);
        p->busy = p->n_threads;
        p->gen++;
        pthread_cond_broadcast(&p->go);
        pthread_mutex_unlock(&p->mu);
        pool_work(p);
        pthread_mutex_lock(&p->mu);
        while (p->busy) pthread_cond_wait(&p->done, &p->mu);
        pthread_mutex_unlock(&p->mu);
    } else {
        pool_work(p);
    }
}
static void pool_close(pool_t *p) {
    pthread_mutex_lock(&p->mu);
    p->stop = 1;
    pthread_cond_broadcast(&p->go);
    pthread_mutex_unlock(&p->mu);
    for (int k = 0; k < p->n_threads; k++) pthread_join(p->th[k], NULL);
    free(p->th);
}

/* ---- growable output buffer ------------------------------------------------------------------------------------------- */
typedef struct { char *p; size_t len, cap; } obuf_t;
static inline char *obuf_reserve(obuf_t *o, size_t need) {
    if (o->cap - o->len < need) {
        size_t cap = o->cap * 2 + need + (1u << 16);
        char *np = (char *)realloc(o->p, cap);
        if (!np) { fprintf(stderr, "[sigtk] out of memory\n"); exit(EXIT_FAILURE); }
        o->p = np; o->cap = cap;
    }
    return o->p + o->len;
}

/* ---- batches in flight ------------------------------------------------------------------------------------------ */
typedef struct {
    sgpu_ctx_t *ctx;
    uint32_t slot;
    int busy;          /* submitted, not yet printed */
    uint32_t n_reads;
    char *ids;         /* read ids, NUL separated */
    size_t ids_len, ids_cap;
    size_t *id_off;    /* [n_reads] */
    size_t id_off_cap;
} lane_t;

typedef struct {
    lane_t *lanes;
    int n_lanes;
    int cur;       /* lane being filled */
    int oldest;    /* oldest busy lane (print order) */
    int n_busy;
    int n_gpus;
    uint64_t cap_samples;
    uint32_t cap_reads;
    opt_t opt;
    uint32_t want;
    uint32_t ctx_flags; /* SGPU_F_* of the contexts */
    uint64_t n_seq_order, n_fixups, n_reads_total;
    pool_t pool;
    obuf_t *obufs;   /* one per formatting chunk */
    int n_obufs;
} engine_t;

static void die_sgpu(sgpu_ctx_t *ctx, int rc, const char *what) {
    ERROR("%s failed: %s (%s)", what, sgpu_strerror(rc), ctx ? sgpu_last_error(ctx) : "-");
    exit(EXIT_FAILURE);
}

/* one context (CUDA context on first use + pinned slots) per GPU, created concurrently: on a cold box this is the
 * largest single cost of the whole command (seconds), and it does not depend on the input */
typedef struct {
    int device;
    uint64_t cap_samples;
    uint32_t cap_reads, flags;
    int rna004;
    sgpu_ctx_t *ctx;
    int rc;
} ctx_job_t;
static void *ctx_create_thread(void *arg) {
    ctx_job_t *j = (ctx_job_t *)arg;
    j->rc = sgpu_create(&j->ctx, j->device, j->cap_samples, j->cap_reads, 2, j->flags);
    if (j->rc == 0 && j->rna004) sgpu_set_param(j->ctx, SGPU_PARAM_PORE, 1.0);
    return NULL;
}

static void engine_open(engine_t *e, int n_gpus, uint64_t cap_samples) {
    const int avail = sgpu_device_count();
    if (avail <= 0) {
        ERROR("%s", "no CUDA device found: the B200 hot path has no CPU fallback");
        exit(EXIT_FAILURE);
    }
    if (n_gpus > avail) n_gpus = avail;
    e->n_gpus = n_gpus;
    e->cap_samples = cap_samples;
    e->cap_reads = (uint32_t)(cap_samples / 256 + 1024);
    e->n_lanes = 2 * n_gpus;
    e->lanes = (lane_t *)calloc((size_t)e->n_lanes, sizeof(lane_t));
    ctx_job_t *jobs = (ctx_job_t *)calloc((size_t)n_gpus, sizeof(ctx_job_t));
    pthread_t *th = (pthread_t *)calloc((size_t)n_gpus, sizeof(pthread_t));
    for (int g = 0; g < n_gpus; g++) {
        jobs[g].device = g; jobs[g].cap_samples = cap_samples; jobs[g].cap_reads = e->cap_reads;
        jobs[g].flags = e->ctx_flags; jobs[g].rna004 = e->opt.rna004;
        if (g == 0 || pthread_create(&th[g], NULL, ctx_create_thread, &jobs[g]) != 0) {
            if (g) { ctx_create_thread(&jobs[g]); th[g] = 0; }
        }
    }
    ctx_create_thread(&jobs[0]); /* the caller creates the first one itself */
    for (int g = 0; g < n_gpus; g++) {
        if (g && th[g]) pthread_join(th[g], NULL);
        if (jobs[g].rc) die_sgpu(NULL, jobs[g].rc, "sgpu_create");
        for (uint32_t s = 0; s < 2; s++) {
            lane_t *l = &e->lanes[s * n_gpus + g]; /* consecutive lanes alternate between the GPUs */
            l->ctx = jobs[g].ctx;
            l->slot = s;
        }
    }
    free(jobs);
    free(th);
    e->cur = 0;
    e->oldest = 0;
    e->n_busy = 0;
    int rc = sgpu_slot_reset(e->lanes[0].ctx, e->lanes[0].slot, (uint32_t)e->opt.rna);
    if (rc) die_sgpu(e->lanes[0].ctx, rc, "sgpu_slot_reset");
}

/* engine_open on a helper thread while the caller opens the file, reads and inflates the first records */
typedef struct { engine_t *e; int n_gpus; uint64_t cap; double seconds; } open_job_t;
static open_job_t g_open_job;
static pthread_t g_open_thread;
static int g_open_pending;
static void *engine_open_thread(void *arg) {
    open_job_t *j = (open_job_t *)arg;
    const double t0 = realtime();
    engine_open(j->e, j->n_gpus, j->cap);
    j->seconds = realtime() - t0;
    return NULL;
}
static void engine_open_async(engine_t *e, int n_gpus, uint64_t cap_samples) {
    g_open_job.e = e; g_open_job.n_gpus = n_gpus; g_open_job.cap = cap_samples; g_open_job.seconds = 0.0;
    if (pthread_create(&g_open_thread, NULL, engine_open_thread, &g_open_job) == 0) g_open_pending = 1;
    else engine_open_thread(&g_open_job);
}
static void engine_ready(void) { /* before the first use of the engine */
    if (g_open_pending) {
        const double t0 = realtime();
        pthread_join(g_open_thread, NULL);
        g_open_pending = 0;
        g_prof[6] = g_open_job.seconds;   /* the open itself ... */
        g_prof[8] = realtime() - t0;      /* ... and how long the main thread still had to wait for it */
    }
}

static void engine_close(engine_t *e) {
    for (int g = 0; g < e->n_gpus; g++) sgpu_destroy(e->lanes[g].ctx);
    for (int k = 0; k < e->n_lanes; k++) {
        free(e->lanes[k].ids);
        free(e->lanes[k].id_off);
    }
    free(e->lanes);
    e->lanes = NULL;
}

/* ---- output (reference src/cfunc.c) -------------------------------------------------------------------------------- */
static void print_header(const opt_t *opt) {
    if (opt->mode == MODE_EVENT) {
        if (opt->compact) printf("read_id\tlen_raw_signal\traw_start\traw_end\tnum_event\tevents\n");
        else printf("read_id\tevent_idx\traw_start\traw_end\tevent_mean\tevent_std\n");
    } else if (opt->mode == MODE_STAT) {
        printf("read_id\tlen_raw_signal\traw_mean\tpa_mean\traw_std\tpa_std\traw_median\tpa_median\n");
    } else if (opt->mode == MODE_JNN) { /* cfunc.c:118-120 */
        printf("read_id\tlen_raw_signal\tnum_seg\tseg\n");
    } else if (opt->mode == MODE_ENT) { /* ent.c:106 */
        printf("read_id\traw_ent\tdelta_ent\tbyte_ent\n");
    } else if (opt->mode == MODE_PREFIX) { /* cfunc.c:161-167 */
        printf("read_id\tlen_raw_signal\tadapt_start\tadapt_end\tpolya_start\tpolya_end");
        if (opt->p_stat) printf("\tadapt_mean\tadapt_std\tadapt_median\tpolya_mean\tpolya_std\tpolya_median");
        printf("\n");
    } else {
        printf("read_id\tlen_raw_signal\tpa\n");
    }
}

/* one read, formatted exactly as the reference's printf calls do (fastfmt.h), appended to `o` */
static void format_read(const opt_t *opt, const sgpu_result_t *res, const sgpu_batch_t *b, uint32_t r, const char *rid,
                        obuf_t *o) {
    const long n = (long)b->read_len[r];
    const size_t idl = strlen(rid);
    char *p;
    if (opt->mode == MODE_EVENT) {
        const uint64_t k0 = res->ev_off[r], k1 = res->ev_off[r + 1];
        if (opt->compact) { /* cfunc.c:19-49 */
            p = obuf_reserve(o, idl + 128 + (size_t)(k1 - k0) * 12);
            memcpy(p, rid, idl); p += idl; *p++ = '\t';
            p = fmt_i64(p, n); *p++ = '\t';
            if (k1 > k0) {
                p = fmt_i64(p, (long)res->ev_start[k0]); *p++ = '\t';
                p = fmt_i64(p, n); *p++ = '\t';
                p = fmt_i64(p, (long)(k1 - k0)); *p++ = '\t';
                for (uint64_t k = k0; k < k1; k++) {
                    const long end = (k + 1 < k1) ? (long)res->ev_start[k + 1] : n;
                    const int len = (int)(float)(end - (long)res->ev_start[k]);
                    if (len) {
                        p = fmt_i64(p, len);
                        if (k + 1 < k1) *p++ = ',';
                    }
                }
            } else {
                memcpy(p, ".\t.\t.\t.", 7); p += 7;
            }
            *p++ = '\n';
            o->len = (size_t)(p - o->p);
        } else { /* cfunc.c:51-58 */
            for (uint64_t k = k0; k < k1; k++) {
                p = obuf_reserve(o, idl + 192);
                const long start = (long)res->ev_start[k];
                const long end = (k + 1 < k1) ? (long)res->ev_start[k + 1] : n;
                const float length = (float)(end - start);
                memcpy(p, rid, idl); p += idl; *p++ = '\t';
                p = fmt_i64(p, (int)(k - k0)); *p++ = '\t';
                p = fmt_i64(p, start); *p++ = '\t';
                p = fmt_i64(p, start + (int)length); *p++ = '\t';
                p = fmt_f6(p, res->ev_mean[k]); *p++ = '\t';
                p = fmt_f6(p, res->ev_stdv[k]); *p++ = '\n';
                o->len = (size_t)(p - o->p);
            }
            p = obuf_reserve(o, 1);
            *p++ = '\n';
            o->len = (size_t)(p - o->p);
        }
    } else if (opt->mode == MODE_PA) { /* cfunc.c:85-102 */
        const float *pa = res->pa + b->read_off[r];
        p = obuf_reserve(o, idl + 64);
        memcpy(p, rid, idl); p += idl; *p++ = '\t';
        p = fmt_i64(p, n); *p++ = '\t';
        o->len = (size_t)(p - o->p);
        for (long i = 0; i < n; i += 64) {
            const long m = n - i < 64 ? n - i : 64;
            p = obuf_reserve(o, 64 * 49 + 2);
            for (long q = 0; q < m; q++) {
                p = fmt_f6(p, pa[i + q]);
                if (i + q != n - 1) *p++ = ',';
            }
            o->len = (size_t)(p - o->p);
        }
        p = obuf_reserve(o, 1);
        *p++ = '\n';
        o->len = (size_t)(p - o->p);
    } else if (opt->mode == MODE_JNN) { /* cfunc.c:108-117 + jnn_print, jnn.c:303-343 */
        const uint32_t ns = res->jnn_cnt[r];
        const int32_t *sg = res->jnn_seg + 2 * SGPU_JNN_BASE(b->read_off[r], r);
        p = obuf_reserve(o, idl + 96 + (size_t)ns * 44);
        memcpy(p, rid, idl); p += idl; *p++ = '\t';
        p = fmt_i64(p, n); *p++ = '\t';
        if (n > 0) { /* jnn_raw returns NULL for an empty record and jnn_print then prints nothing */
            p = fmt_i64(p, (long)ns); *p++ = '\t';
            if (opt->compact) {
                uint64_t ci = 0, mi = 0;
                for (uint32_t k = 0; k < ns; k++) {
                    ci += (mi = (uint64_t)(int64_t)sg[2 * k] - ci);
                    if (mi) { p = fmt_i64(p, (int)mi); *p++ = 'H'; }
                    ci += (mi = (uint64_t)(int64_t)sg[2 * k + 1] - ci);
                    if (mi) { p = fmt_i64(p, (int)mi); *p++ = ','; }
                }
            } else {
                for (uint32_t k = 0; k < ns; k++) {
                    p = fmt_i64(p, (long)sg[2 * k]); *p++ = ',';
                    p = fmt_i64(p, (long)sg[2 * k + 1]); *p++ = ';';
                }
            }
            if (ns == 0) *p++ = '.';
        }
        *p++ = '\n';
        o->len = (size_t)(p - o->p);
    } else if (opt->mode == MODE_PREFIX) { /* prefix_func, cfunc.c:169-234 */
        const int32_t *q = res->prefix_pos + (size_t)r * 4;
        const float *st = res->prefix_stat + (size_t)r * 6;
        p = obuf_reserve(o, idl + 640);
        memcpy(p, rid, idl); p += idl; *p++ = '\t';
        p = fmt_i64(p, n); *p++ = '\t';
        if (q[1] > 0) {
            p = fmt_i64(p, (long)q[0]); *p++ = '\t';
            p = fmt_i64(p, (long)q[1]); *p++ = '\t';
            if (q[3] > 0) {
                p = fmt_i64(p, (long)q[2] + q[1]); *p++ = '\t';
                p = fmt_i64(p, (long)q[3] + q[1]);
            } else {
                memcpy(p, ".\t.", 3); p += 3;
            }
            if (opt->p_stat) {
                *p++ = '\t';
                for (int k = 0; k < 3; k++) { p = fmt_f6(p, st[k]); *p++ = '\t'; }
                if (q[3] > 0) {
                    *p++ = '\t';
                    for (int k = 3; k < 6; k++) { p = fmt_f6(p, st[k]); *p++ = '\t'; }
                } else {
                    memcpy(p, "\t.\t.\t.", 6); p += 6;
                }
            }
        } else {
            if (q[1] < 0) WARNING("%s", "Not enough data to trim\n"); /* jnnv2, jnn.c:173 */
            memcpy(p, ".\t.\t.\t.", 7); p += 7;
        }
        *p++ = '\n';
        o->len = (size_t)(p - o->p);
    } else if (opt->mode == MODE_ENT) { /* ent.c:109,113,132,148,163: "%s\t" "%f" "\t%f" "\t%f" "\n" with doubles */
        const double *h = res->ent + (size_t)r * 3;
        p = obuf_reserve(o, idl + 256);
        memcpy(p, rid, idl); p += idl;
        p += snprintf(p, 200, "\t%f\t%f\t%f\n", h[0], h[1], h[2]);
        o->len = (size_t)(p - o->p);
    } else { /* cfunc.c:126-159: note the tab before the newline */
        const float *s = res->stat + (size_t)r * 6;
        p = obuf_reserve(o, idl + 400);
        memcpy(p, rid, idl); p += idl; *p++ = '\t';
        p = fmt_i64(p, n); *p++ = '\t';
        p = fmt_f6(p, s[0]); *p++ = '\t';
        p = fmt_f6(p, s[1]); *p++ = '\t';
        p = fmt_f6(p, s[2]); *p++ = '\t';
        p = fmt_f6(p, s[3]); *p++ = '\t';
        p = fmt_i64(p, (int)(int16_t)s[4]); *p++ = '\t';
        p = fmt_f6(p, s[5]); *p++ = '\t';
        *p++ = '\n';
        o->len = (size_t)(p - o->p);
    }
}

typedef struct {
    engine_t *e;
    lane_t *l;
    const sgpu_result_t *res;
    const sgpu_batch_t *b;
    const uint32_t *first; /* [n_chunks + 1] read ranges of the formatting chunks */
} fmt_job_t;

static void format_chunk(void *arg, int c) {
    fmt_job_t *j = (fmt_job_t *)arg;
    obuf_t *o = &j->e->obufs[c];
    o->len = 0;
    for (uint32_t r = j->first[c]; r < j->first[c + 1]; r++)
        format_read(&j->e->opt, j->res, j->b, r, j->l->ids + j->l->id_off[r], o);
}

static void print_lane(engine_t *e, lane_t *l) {
    sgpu_result_t res;
    double t0 = realtime();
    int rc = sgpu_wait(l->ctx, l->slot, &res);
    if (rc) die_sgpu(l->ctx, rc, "sgpu_wait");
    g_prof[3] += realtime() - t0;
    sgpu_batch_t *b = NULL;
    rc = sgpu_slot_batch(l->ctx, l->slot, &b);
    if (rc) die_sgpu(l->ctx, rc, "sgpu_slot_batch");
    if (e->opt.mode == MODE_EVENT)
        for (uint32_t r = 0; r < l->n_reads; r++) {
            e->n_seq_order += res.seq_order[r];
            e->n_fixups += res.fixups[r];
        }
    /* formatting chunks: contiguous read ranges of about equal sample counts, a few per thread */
    int n_chunks = 4 * (e->pool.n_threads + 1);
    if ((uint32_t)n_chunks > l->n_reads) n_chunks = (int)l->n_reads;
    if (n_chunks > e->n_obufs) {
        e->obufs = (obuf_t *)realloc(e->obufs, (size_t)n_chunks * sizeof(obuf_t));
        memset(e->obufs + e->n_obufs, 0, (size_t)(n_chunks - e->n_obufs) * sizeof(obuf_t));
        e->n_obufs = n_chunks;
    }
    uint32_t *first = (uint32_t *)malloc(((size_t)n_chunks + 1) * sizeof(uint32_t));
    if (!first || (n_chunks && !e->obufs)) { ERROR("%s", "out of memory"); exit(EXIT_FAILURE); }
    const uint64_t total = l->n_reads ? b->read_off[l->n_reads] : 0;
    uint32_t r = 0;
    for (int c = 0; c < n_chunks; c++) {
        first[c] = r;
        const uint64_t upto = total / (uint64_t)n_chunks * (uint64_t)(c + 1);
        while (r < l->n_reads && (c == n_chunks - 1 || b->read_off[r + 1] <= upto || r == first[c])) r++;
    }
    first[n_chunks] = l->n_reads;
    fmt_job_t job = {e, l, &res, b, first};
    t0 = realtime();
    pool_run(&e->pool, format_chunk, &job, n_chunks);
    g_prof[4] += realtime() - t0;
    t0 = realtime();
    for (int c = 0; c < n_chunks; c++)
        if (e->obufs[c].len && fwrite(e->obufs[c].p, 1, e->obufs[c].len, stdout) != e->obufs[c].len) {
            ERROR("%s", "write to stdout failed");
            exit(EXIT_FAILURE);
        }
    g_prof[5] += realtime() - t0;
    free(first);
    e->n_reads_total += l->n_reads;
    l->busy = 0;
    l->n_reads = 0;
    l->ids_len = 0;
}

static void engine_submit_current(engine_t *e) {
    engine_ready();
    lane_t *l = &e->lanes[e->cur];
    if (l->n_reads == 0) return;
    int rc = sgpu_submit(l->ctx, l->slot, e->want);
    if (rc) die_sgpu(l->ctx, rc, "sgpu_submit");
    l->busy = 1;
    e->n_busy++;
    /* next lane; if it still holds an unprinted batch, that one is the oldest: print it first */
    e->cur = (e->cur + 1) % e->n_lanes;
    lane_t *nx = &e->lanes[e->cur];
    if (nx->busy) {
        print_lane(e, nx);
        e->n_busy--;
        e->oldest = (e->cur + 1) % e->n_lanes;
    }
    rc = sgpu_slot_reset(nx->ctx, nx->slot, (uint32_t)e->opt.rna);
    if (rc) die_sgpu(nx->ctx, rc, "sgpu_slot_reset");
}

static void engine_drain(engine_t *e) {
    engine_submit_current(e);
    /* print what is still in flight, oldest first: lanes are used round-robin */
    for (int k = 0; k < e->n_lanes; k++) {
        lane_t *l = &e->lanes[(e->cur + k) % e->n_lanes];
        if (l->busy) {
            print_lane(e, l);
            e->n_busy--;
        }
    }
}

/* one record on its way into a batch: decoded samples (raw != NULL) or the still compressed svb-zd stream */
typedef struct {
    const char *read_id;
    size_t read_id_len;       /* without the NUL */
    double digitisation, offset, range;
    const int16_t *raw;       /* decoded samples ... */
    uint64_t len_raw_signal;
    const uint8_t *svb;       /* ... or the record's raw_signal field as stored (svb-zd) */
    uint64_t svb_bytes;
} rec_view_t;

static void engine_add_view(engine_t *e, const rec_view_t *v) {
    engine_ready();
    for (int attempt = 0; attempt < 3; attempt++) {
        lane_t *l = &e->lanes[e->cur];
        int64_t rc = v->raw || !v->svb
            ? sgpu_slot_add_read(l->ctx, l->slot, v->raw, v->len_raw_signal, v->digitisation, v->offset, v->range)
            : sgpu_slot_add_read_svbzd(l->ctx, l->slot, v->svb, v->svb_bytes, v->digitisation, v->offset, v->range);
        if (rc >= 0) {
            const size_t idl = v->read_id_len + 1;
            if (l->ids_len + idl > l->ids_cap) {
                l->ids_cap = (l->ids_len + idl) * 2 + 4096;
                l->ids = (char *)realloc(l->ids, l->ids_cap);
            }
            if (l->n_reads + 1 > l->id_off_cap) {
                l->id_off_cap = l->id_off_cap * 2 + 1024;
                l->id_off = (size_t *)realloc(l->id_off, l->id_off_cap * sizeof(size_t));
            }
            if (!l->ids || !l->id_off) {
                ERROR("%s", "out of memory");
                exit(EXIT_FAILURE);
            }
            memcpy(l->ids + l->ids_len, v->read_id, v->read_id_len);
            l->ids[l->ids_len + v->read_id_len] = '\0';
            l->id_off[l->n_reads++] = l->ids_len;
            l->ids_len += idl;
            return;
        }
        if (rc == SGPU_E_FULL) {
            engine_submit_current(e);
            continue;
        }
        if (rc == SGPU_E_TOOBIG && v->len_raw_signal < (1ull << 31)) {
            /* one read larger than a whole slot: finish what is in flight and reopen with bigger slots */
            engine_drain(e);
            const int n_gpus = e->n_gpus;
            uint64_t cap = e->cap_samples;
            while (cap < v->len_raw_signal + 64 || 2 * cap < v->svb_bytes + 64) cap *= 2;
            engine_close(e);
            e->ctx_flags |= SGPU_F_FULL_SEQ_SCRATCH; /* a read this long must be able to take the sequential-order kernels */
            engine_open(e, n_gpus, cap);
            continue;
        }
        die_sgpu(l->ctx, (int)rc, "sgpu_slot_add_read");
    }
    ERROR("%s", "could not place a read into a batch");
    exit(EXIT_FAILURE);
}

static void engine_add(engine_t *e, const blow5_rec_t *rec) {
    rec_view_t v;
    memset(&v, 0, sizeof v);
    v.read_id = rec->read_id;
    v.read_id_len = strlen(rec->read_id);
    v.digitisation = rec->digitisation;
    v.offset = rec->offset;
    v.range = rec->range;
    v.raw = rec->raw_signal;
    v.len_raw_signal = rec->len_raw_signal;
    engine_add_view(e, &v);
}

/* ---- batch loader: parallel decode of one group of records ------------------------------------------------------------ */
typedef struct {
    const blow5_file_t *sp;
    char **mem;         /* the records' bytes as read from the file (blow5_next_bytes) */
    size_t *bytes;
    blow5_rec_t **rec;  /* decoded records, reused from group to group */
    int *err;
} load_job_t;

static void decode_item(void *arg, int i) { /* blow5_decode: zlib inflate + svb-zd; frees the record's bytes */
    load_job_t *j = (load_job_t *)arg;
    j->err[i] = blow5_decode(j->sp, &j->mem[i], &j->bytes[i], &j->rec[i]);
}

/* GPU signal decode: the pool only undoes the RECORD compression (zlib) and finds the main columns of the binary
 * record (blow5_view); the svb-zd stream itself goes to the GPU as it is. */
typedef struct {
    const blow5_file_t *sp;
    char **mem;
    size_t *bytes;
    rec_view_t *view;
    int *err;
} inflate_job_t;

static void inflate_item(void *arg, int i) {
    inflate_job_t *j = (inflate_job_t *)arg;
    blow5_view_t b;
    rec_view_t *v = &j->view[i];
    memset(v, 0, sizeof *v);
    if ((j->err[i] = blow5_inflate(j->sp, &j->mem[i], &j->bytes[i])) < 0) return;
    if ((j->err[i] = blow5_view(j->sp, j->mem[i], j->bytes[i], &b)) < 0) return;
    v->read_id = b.read_id;
    v->read_id_len = b.read_id_len;
    v->digitisation = b.digitisation;
    v->offset = b.offset;
    v->range = b.range;
    v->svb = b.signal;
    v->svb_bytes = b.signal_bytes;
    v->len_raw_signal = b.len_raw_signal;
}

/* ---- sub-command driver (reference src/cmain.c) ----------------------------------------------------------------------- */
static struct option long_options[] = {{"verbose", required_argument, 0, 'v'},
                                       {"help", no_argument, 0, 'h'},
                                       {"version", no_argument, 0, 'V'},
                                       {"output", required_argument, 0, 'o'},
                                       {"print-stat", no_argument, 0, 0},
                                       {"no-header", no_argument, 0, 'n'},
                                       {"compact", no_argument, 0, 'c'},
                                       {"gpus", required_argument, 0, 0},          /* 7 (additive) */
                                       {"batch-samples", required_argument, 0, 0}, /* 8 (additive) */
                                       {"threads", required_argument, 0, 0},       /* 9 (additive) */
                                       {"cpu-decode", no_argument, 0, 0},          /* 10 (additive) */
                                       {0, 0, 0, 0}};

static int cmain(int argc, char *argv[], const char *mode) {
    const int is_ent = strcmp(mode, "ent") == 0;
    const char *optstring = is_ent ? "hV" : "o:hVnc"; /* ent.c:70: `ent` only has -h, -V and --no-header */
    int longindex = 0, c = -1;
    FILE *fp_help = stderr;
    int hdr = 1, n_gpus = 1, n_threads = 0, cpu_decode = 0;
    uint64_t batch_samples = 0;
    engine_t eng;
    memset(&eng, 0, sizeof eng);

    while ((c = getopt_long(argc, argv, optstring, long_options, &longindex)) >= 0) {
        if (c == 'V') {
            fprintf(stdout, "sigtk %s\n", SIGTK_VERSION);
            exit(EXIT_SUCCESS);
        } else if (c == 'h') {
            fp_help = stdout;
        } else if (c == 'n') {
            hdr = 0;
        } else if (c == 'c') {
            eng.opt.compact = 1;
        } else if (c == 0 && longindex == 4) { /* cmain.c:63-64 */
            eng.opt.p_stat = 1;
        } else if (c == 0 && longindex == 7) {
            n_gpus = atoi(optarg);
            if (n_gpus < 1) n_gpus = 1;
        } else if (c == 0 && longindex == 8) {
            batch_samples = strtoull(optarg, NULL, 10);
        } else if (c == 0 && longindex == 9) {
            n_threads = atoi(optarg);
        } else if (c == 0 && longindex == 10) {
            cpu_decode = 1;
        }
    }
    if (is_ent && (argc - optind != 1 || fp_help == stdout)) { /* ent.c:90-100 */
        fprintf(fp_help, "Usage: sigtk ent a.blow5\n");
        fprintf(fp_help, "\nbasic options:\n");
        fprintf(fp_help, "   -h                         help\n");
        fprintf(fp_help, "   -n                         suppress header\n");
        fprintf(fp_help, "   --version                  print version\n");
        if (fp_help == stdout) exit(EXIT_SUCCESS);
        exit(EXIT_FAILURE);
    }
    if (argc - optind < 1 || fp_help == stdout) {
        fprintf(fp_help, "Usage: sigtk %s reads.blow5 read_id1 read_id2 .. \n", mode);
        fprintf(fp_help, "       sigtk %s reads.blow5\n", mode);
        fprintf(fp_help, "\nbasic options:\n");
        fprintf(fp_help, "   -h                         help\n");
        fprintf(fp_help, "   -n                         suppress header\n");
        fprintf(fp_help, "   -c                         compact output\n");
        fprintf(fp_help, "   --version                  print version\n");
        if (fp_help == stdout) exit(EXIT_SUCCESS);
        exit(EXIT_FAILURE);
    }
    blow5_file_t *sp = blow5_open(argv[optind]);
    if (!sp) {
        if (is_ent) fprintf(stderr, "Error in opening file\n"); /* ent.c:104 */
        else ERROR("cannot open %s. \n", argv[optind]);
        exit(EXIT_FAILURE);
    }
    if (!is_ent) { /* entmain does not look at the header (ent.c:102-107) */
        eng.opt.rna = drna_detect(sp);
        eng.opt.rna004 = pore_detect(sp) == PORE_RNA004;
    }
    if (is_ent) {
        eng.opt.mode = MODE_ENT;
        eng.want = SGPU_WANT_ENT;
    } else if (strcmp(mode, "jnn") == 0) {
        eng.opt.mode = MODE_JNN;
        eng.want = SGPU_WANT_JNN;
    } else if (strcmp(mode, "prefix") == 0) {
        eng.opt.mode = MODE_PREFIX;
        eng.want = SGPU_WANT_PREFIX;
    } else if (strcmp(mode, "event") == 0) {
        eng.opt.mode = MODE_EVENT;
        eng.want = SGPU_WANT_EVENTS;
    } else if (strcmp(mode, "stat") == 0) {
        eng.opt.mode = MODE_STAT;
        eng.want = SGPU_WANT_STAT;
    } else {
        eng.opt.mode = MODE_PA;
        eng.want = SGPU_WANT_PA;
    }
    if (hdr) print_header(&eng.opt);

    if (batch_samples == 0) { /* slots sized from the file: small files must not pay for large pinned buffers */
        struct stat st;
        uint64_t bytes = (stat(argv[optind], &st) == 0) ? (uint64_t)st.st_size : (64ull << 20);
        batch_samples = bytes * 8;
        if (batch_samples < (1ull << 20)) batch_samples = 1ull << 20;
        if (batch_samples > (1ull << 24)) batch_samples = 1ull << 24; /* pinned memory is slow to allocate; the GPU
                                                                          is far from the limit of this pipeline */
    }
    if (n_threads <= 0) { /* decode and formatting threads: the host's cores, at most 32 */
        const long nc = sysconf(_SC_NPROCESSORS_ONLN);
        n_threads = nc < 1 ? 1 : nc > 32 ? 32 : (int)nc;
    }
    pool_open(&eng.pool, n_threads);
    if (eng.opt.mode == MODE_PA && batch_samples > (1ull << 23)) batch_samples = 1ull << 23; /* 13 text bytes per sample */
    engine_open_async(&eng, n_gpus, batch_samples); /* joined by the first engine_add / engine_drain */

    blow5_rec_t *rec = NULL;
    int ret = 0;
    /* BLOW5 with svb-zd signal compression (the default of slow5tools): the signal is decoded on the GPU */
    const int gpu_decode = !cpu_decode && argc - optind == 1 && !sp->ascii && sp->signal_press == BLOW5_SIGNAL_SVB_ZD;
    if (gpu_decode) {
        enum { GROUP = 512 };
        inflate_job_t job;
        memset(&job, 0, sizeof job);
        job.sp = sp;
        job.mem = (char **)calloc(GROUP, sizeof(char *));
        job.bytes = (size_t *)calloc(GROUP, sizeof(size_t));
        job.view = (rec_view_t *)calloc(GROUP, sizeof(rec_view_t));
        job.err = (int *)calloc(GROUP, sizeof(int));
        if (!job.mem || !job.bytes || !job.view || !job.err) { ERROR("%s", "out of memory"); exit(EXIT_FAILURE); }
        int eof = 0;
        while (!eof) {
            int n = 0;
            size_t group_bytes = 0;
            double t0 = realtime();
            while (n < GROUP && group_bytes < (64u << 20)) {
                if ((ret = blow5_next_bytes(sp, &job.mem[n], &job.bytes[n])) < 0) {
                    eof = 1;
                    break;
                }
                group_bytes += job.bytes[n++];
            }
            g_prof[0] += realtime() - t0;
            t0 = realtime();
            pool_run(&eng.pool, inflate_item, &job, n);
            g_prof[1] += realtime() - t0;
            t0 = realtime();
            for (int i = 0; i < n; i++) {
                if (job.err[i] < 0) {
                    engine_drain(&eng); /* the reference has printed every record before this one */
                    fflush(stdout);
                    fprintf(stderr, "Error in slow5_get_next. Error code %d\n", job.err[i]);
                    exit(EXIT_FAILURE);
                }
                engine_add_view(&eng, &job.view[i]);
                free(job.mem[i]);
                job.mem[i] = NULL;
            }
            g_prof[2] += realtime() - t0;
        }
        if (ret != BLOW5_EOF) {
            engine_drain(&eng);
            fflush(stdout);
            fprintf(stderr, "Error in slow5_get_next. Error code %d\n", ret);
            exit(EXIT_FAILURE);
        }
        free(job.mem); free(job.bytes); free(job.view); free(job.err);
    } else if (argc - optind == 1) {
        /* batch loader: the records' bytes are read serially, a group at a time, and decoded by the pool */
        enum { GROUP = 512 };
        load_job_t job;
        memset(&job, 0, sizeof job);
        job.sp = sp;
        job.mem = (char **)calloc(GROUP, sizeof(char *));
        job.bytes = (size_t *)calloc(GROUP, sizeof(size_t));
        job.rec = (blow5_rec_t **)calloc(GROUP, sizeof(blow5_rec_t *));
        job.err = (int *)calloc(GROUP, sizeof(int));
        if (!job.mem || !job.bytes || !job.rec || !job.err) { ERROR("%s", "out of memory"); exit(EXIT_FAILURE); }
        int eof = 0;
        while (!eof) {
            int n = 0;
            size_t group_bytes = 0;
            double t0 = realtime();
            while (n < GROUP && group_bytes < (64u << 20)) {
                if ((ret = blow5_next_bytes(sp, &job.mem[n], &job.bytes[n])) < 0) {
                    eof = 1;
                    break;
                }
                group_bytes += job.bytes[n++];
            }
            g_prof[0] += realtime() - t0;
            t0 = realtime();
            pool_run(&eng.pool, decode_item, &job, n);
            g_prof[1] += realtime() - t0;
            t0 = realtime();
            for (int i = 0; i < n; i++) {
                if (job.err[i] < 0) {
                    engine_drain(&eng);
                    fflush(stdout);
                    fprintf(stderr, "Error in slow5_get_next. Error code %d\n", job.err[i]);
                    exit(EXIT_FAILURE);
                }
                engine_add(&eng, job.rec[i]);
            }
            g_prof[2] += realtime() - t0; /* includes the submits and prints that engine_add triggers */
        }
        if (ret != BLOW5_EOF) {
            engine_drain(&eng);
            fflush(stdout);
            fprintf(stderr, "Error in slow5_get_next. Error code %d\n", ret);
            exit(EXIT_FAILURE);
        }
        for (int i = 0; i < GROUP; i++) blow5_rec_free(job.rec[i]);
        free(job.mem); free(job.bytes); free(job.rec); free(job.err);
    } else {
        if (blow5_idx_load(sp) < 0) {
            ERROR("Error loading index file for %s\n", argv[optind]);
            exit(EXIT_FAILURE);
        }
        for (int i = optind + 1; i < argc; i++) {
            fprintf(stderr, "Read ID %s\n", argv[i]);
            if (blow5_get(sp, argv[i], &rec) < 0) {
                ERROR("%s", "Error when fetching the read\n");
                exit(EXIT_FAILURE);
            }
            engine_add(&eng, rec);
        }
        blow5_idx_unload(sp);
    }
    engine_drain(&eng);
    fflush(stdout);
    if (eng.opt.mode == MODE_EVENT && (eng.n_seq_order || eng.n_fixups))
        fprintf(stderr, "[%s] %" PRIu64 " of %" PRIu64 " reads took the sequential-order kernels (%" PRIu64
                        " detector boundary mismatches); results are bit-identical either way\n",
                __func__, eng.n_seq_order, eng.n_reads_total, eng.n_fixups);
    {
        const double t0 = realtime();
        engine_close(&eng);
        g_prof[7] = realtime() - t0;
    }
    if (getenv("SIGTK_PROFILE"))
        fprintf(stderr, "[%s] signal decode: %s\n", __func__, gpu_decode ? "GPU (svb-zd)" : "host threads (blow5_decode)");
    if (getenv("SIGTK_PROFILE"))
        fprintf(stderr, "[%s] host wall clock: open (CUDA context, pinned slots) %.3f s on a helper thread, of which the main "
                        "thread waited %.3f s, read %.3f s, decode %.3f s (%d threads), "
                        "add+submit+print %.3f s of which wait %.3f s, format %.3f s, write %.3f s, close %.3f s\n", __func__,
                g_prof[6], g_prof[8], g_prof[0], g_prof[1], eng.pool.n_threads + 1, g_prof[2], g_prof[3], g_prof[4], g_prof[5], g_prof[7]);
    pool_close(&eng.pool);
    for (int c = 0; c < eng.n_obufs; c++) free(eng.obufs[c].p);
    free(eng.obufs);
    blow5_rec_free(rec);
    blow5_close(sp);
    return 0;
}

static int print_usage(FILE *fp_help) {
    fprintf(fp_help, "Usage: sigtk <command> [options]\n\n");
    fprintf(fp_help, "command:\n");
    fprintf(fp_help, "         pa        print raw signal in pico-amperes\n");
    fprintf(fp_help, "         event     segment raw signal into events\n");
    fprintf(fp_help, "         stat      print statistics of the raw signal\n");
    fprintf(fp_help, "         ent       entropy of the raw signal, its zig-zag deltas and their byte planes\n");
    fprintf(fp_help, "         jnn       stall / homopolymer-stretch segments of the raw signal\n");
    fprintf(fp_help, "         prefix    adaptor and poly-A stretch at the start of a read\n");
    fprintf(fp_help, "(B200 build: the raw-signal hot path only; sref, ss and qts are served by the\n");
    fprintf(fp_help, " reference sigtk)\n");
    exit(fp_help == stderr ? EXIT_FAILURE : EXIT_SUCCESS);
}

int main(int argc, char *argv[]) {
    const double realtime0 = realtime();
    int ret = 1;
    static char outbuf[1 << 22];
    setvbuf(stdout, outbuf, _IOFBF, sizeof outbuf);
    if (argc < 2) {
        return print_usage(stderr);
    } else if (strcmp(argv[1], "event") == 0 || strcmp(argv[1], "stat") == 0 || strcmp(argv[1], "pa") == 0 ||
               strcmp(argv[1], "ent") == 0 || strcmp(argv[1], "jnn") == 0 || strcmp(argv[1], "prefix") == 0) {
        ret = cmain(argc - 1, argv + 1, argv[1]);
    } else if (strcmp(argv[1], "--version") == 0 || strcmp(argv[1], "-V") == 0) {
        fprintf(stdout, "sigtk %s\n", SIGTK_VERSION);
        exit(EXIT_SUCCESS);
    } else if (strcmp(argv[1], "--help") == 0 || strcmp(argv[1], "-h") == 0) {
        print_usage(stdout);
    } else if (strcmp(argv[1], "sref") == 0 || strcmp(argv[1], "ss") == 0 || strcmp(argv[1], "qts") == 0) {
        fprintf(stderr, "[sigtk] command %s is outside the B200 raw-signal hot path; use the reference sigtk for it\n",
                argv[1]);
        exit(EXIT_FAILURE);
    } else {
        fprintf(stderr, "[sigtk] Unrecognised command %s\n", argv[1]);
        print_usage(stderr);
    }
    fprintf(stderr, "[%s] Version: %s\n", __func__, SIGTK_VERSION);
    fprintf(stderr, "[%s] CMD:", __func__);
    for (int i = 0; i < argc; ++i) fprintf(stderr, " %s", argv[i]);
    fprintf(stderr, "\n[%s] Real time: %.3f sec; CPU time: %.3f sec; Peak RAM: %.3f GB\n\n", __func__,
            realtime() - realtime0, cputime(), (double)peakrss() / 1024.0 / 1024.0 / 1024.0);
    return ret;
}
