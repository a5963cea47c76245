/* sigtk_b200.h -- C-ABI of the B200-native sigtk raw-signal hot path.
 *
 * Plain C99, no CUDA or torch types in any signature.  Built for sm_100a only;
 * there is NO CPU fallback: every entry point returns SGPU_E_CUDA (or the
 * library fails to load) when no CUDA device is usable.
 *
 * What it replaces in the reference (file:line under hasindu2008/sigtk):
 *   - float *signal_in_picoamps(slow5_rec_t*)            src/sigtk.h:124, src/misc.c:15-32
 *   - event_table getevents(size_t, float*, int8_t rna)  src/sigtk.h:134, src/events.c:553-573: fused with the
 *                                                        pA conversion on int16 records, or on the caller's own
 *                                                        pA floats (sgpu_slot_add_read_pa, sgpu_run_device_pa)
 *   - meanf/stdvf/medianf/meani16/stdvi16/mediani16      src/stat.h:17-73 (as used by stat_func,
 *                                                        src/cfunc.c:126-159)
 *   - jnn_pair_t *jnn_raw(const int16_t*, int64_t, jnn_param_t, int *n)   src/jnn.h:105, src/jnn.c:176-282
 *   - double entropy(int16_t*, uint64_t) and the zig-zag-delta / byte-plane loop of entmain
 *                                                        src/ent.c:25-51, 56-65, 108-151
 * The reference calls those once per record from a callback
 * `void (*func)(slow5_rec_t*, opt_t)` (src/cmain.c:95-126).  Here the unit of
 * work is a BATCH of records: the host appends decoded records to a pinned
 * slot, submits it, and reads per-read results back in record order.
 *
 * Ownership: the library owns all device and pinned memory for the lifetime
 * of the context; the host fills / reads slot buffers in place.  Nothing is
 * malloc'd per read.  A context is used by one host thread at a time.
 *
 * Errors: every function returns 0 or a negative SGPU_E_* code and never
 * calls exit(); sgpu_strerror() gives text, sgpu_last_error(ctx) the CUDA
 * detail.
 */
#ifndef SIGTK_B200_H
#define SIGTK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SGPU_ABI_VERSION 5

/* ---- error codes ------------------------------------------------------- */
#define SGPU_OK            0
#define SGPU_E_INVAL      -1  /* bad argument */
#define SGPU_E_CUDA       -2  /* CUDA runtime / driver / kernel error (see sgpu_last_error) */
#define SGPU_E_NOMEM      -3  /* host or device allocation failed */
#define SGPU_E_FULL       -4  /* slot cannot take this read: submit it and retry */
#define SGPU_E_TOOBIG     -5  /* a single read exceeds the context's max_samples */
#define SGPU_E_STATE      -6  /* call out of order (e.g. wait on a slot that was not submitted) */
#define SGPU_E_EVCAP      -7  /* event capacity exceeded (never for n/3+2 sizing; reported, not truncated) */
#define SGPU_E_SCRATCH    -8  /* sequential-order scratch too small for the reads that need it */
#define SGPU_E_STREAM     -9  /* malformed svb-zd stream (slow5lib: "Expected streamvbyte_decode to read ...", slow5_press.c:1103) */

/* ---- what to compute (bitmask) ------------------------------------------ */
#define SGPU_WANT_EVENTS   1u /* event table: getevents(), events.c:553-573 */
#define SGPU_WANT_PA       2u /* materialise pA floats: signal_in_picoamps(), misc.c:15-32 */
#define SGPU_WANT_STAT     4u /* the six numbers of stat_func, cfunc.c:126-159 */
#define SGPU_WANT_ENT      8u /* the three entropies of `sigtk ent`, ent.c:108-151 */
#define SGPU_WANT_JNN     16u /* the segments of `sigtk jnn`: jnn_raw(), jnn.c:269-282 with the parameters of
                                 jnn_print (jnn.c:305-312: JNNV1_DRNA_R9_PARAM when rna, else JNNV1_CDNA_R9_PARAM) */

#define SGPU_WANT_PREFIX  32u /* `sigtk prefix` (prefix_func, cfunc.c:169-234): find_adaptor (jnnv2, jnn.c:99-188), the
                                 adaptor's pA statistics, find_polya (jnn.c:352-374) when rna, its statistics */

/* ---- context flags ------------------------------------------------------ */
#define SGPU_F_DEFAULT       0u
#define SGPU_F_FORCE_GENERIC 1u /* run every read through the sequential-order (reference-order) kernels */
#define SGPU_F_NO_HOST_SLOTS 2u /* device-resident use only: do not allocate pinned slots */
#define SGPU_F_STAGE_TIMERS  4u /* record CUDA events between the kernel groups of a run (sgpu_stage_times) */
#define SGPU_F_FULL_SEQ_SCRATCH 8u /* size the sequential-order scratch for the whole batch (a context opened for one
                                      huge read: the reference handles any read < 2^31 samples, misc.c:20) */

typedef struct sgpu_ctx sgpu_ctx_t;

/* Reads are laid out back to back in one flat int16 array; read r occupies
 * samples[read_off[r] .. read_off[r]+read_len[r]) and every read_off[r] is a
 * multiple of SGPU_ALIGN samples (16 bytes) so that 128-bit / bulk loads are
 * aligned.  The per-read scalars are the reference's narrowed floats:
 *   offset_f   = (float)rec->offset                        (misc.c:19)
 *   raw_unit_f = (float)rec->range / (float)rec->digitisation  (misc.c:17-18,26)
 * computed on the host in C exactly as the reference does. */
#define SGPU_ALIGN 8

typedef struct {
    int16_t  *samples;     /* [capacity max_samples] */
    uint64_t *read_off;    /* [n_reads+1]; read_off[n_reads] = end of used span (aligned) */
    uint32_t *read_len;    /* [n_reads] */
    float    *offset_f;    /* [n_reads] */
    float    *raw_unit_f;  /* [n_reads] */
    uint32_t  n_reads;
    uint32_t  rna;         /* 0: DNA detector parameters (events.c:43-47), 1: RNA (50-54) */
} sgpu_batch_t;

/* Per-batch results.  Host pointers (pinned) from sgpu_wait(), device
 * pointers from sgpu_run_device().  Event k of read r is
 *   k in [ev_off[r], ev_off[r+1]),  start = ev_start[k] (sample index in the read),
 *   end = next event's start, or read_len[r] for the read's last event
 *   (event_t, sigtk.h:55-62: length = (float)(end-start)). */
typedef struct {
    uint64_t *ev_off;      /* [n_reads+1] */
    uint32_t *ev_start;    /* [n_events] */
    float    *ev_mean;     /* [n_events] */
    float    *ev_stdv;     /* [n_events] */
    float    *pa;          /* same layout as samples; NULL unless SGPU_WANT_PA */
    float    *stat;        /* [n_reads][6]: raw_mean, pa_mean, raw_std, pa_std, raw_median, pa_median */
    uint32_t *seq_order;   /* [n_reads] 1 if the read went through the sequential-order kernels
                              (exact-sum witness failed, or forced); such reads are still bit-exact */
    uint32_t *fixups;      /* [n_reads] number of detector chunks whose warm-up state did not match (the read is then redone
                              by the sequential-order kernels) */
    uint64_t  n_events;    /* total events in the batch (host result only; 0 from sgpu_run_device) */
    double   *ent;         /* [n_reads][3]: raw_ent, delta_ent, byte_ent in bits (ent.c:108-151); NULL unless
                              SGPU_WANT_ENT. Histogram counts are exact and the terms are summed in the reference's
                              order; log2 is CUDA's (<= 1 ulp), so the doubles agree to ~1e-15 and "%f" prints alike.
                              An empty record (where the reference crashes) gives zeros. */
    uint32_t *jnn_cnt;     /* [n_reads] number of segments (jnn_raw's *n); NULL unless SGPU_WANT_JNN */
    int32_t  *jnn_seg;     /* segment k of read r = (x, y) = jnn_seg[2*(SGPU_JNN_BASE(read_off[r], r) + k) + {0,1}]
                              (jnn_pair_t, jnn.h:13-16; sample indices in the read). Bit-exact. */
    int32_t  *prefix_pos;  /* [n_reads][4]: adaptor x, y as find_adaptor returns them ((0,0): none found, (-1,-1): record not
                              longer than the 2,000-sample window), poly-A x, y as find_polya returns them, i.e. relative
                              to the adaptor's end ((-1,-1): none / DNA); NULL unless SGPU_WANT_PREFIX. Bit-exact. */
    float    *prefix_stat; /* [n_reads][6]: meanf, stdvf, medianf of the adaptor's pA (valid when its y > 0), then of the
                              poly-A's (valid when its y > 0): cfunc.c:178-180, 202-204. Bit-exact. */
} sgpu_result_t;
/* first segment slot of read r (a read of n samples has at most n/38 + 1 segments, jnn.c:232) */
#define SGPU_JNN_BASE(read_off_r, r) (((uint64_t)(read_off_r) >> 5) + (uint64_t)(r))

/* ---- lifecycle ----------------------------------------------------------- */
int  sgpu_device_count(void);
int  sgpu_create(sgpu_ctx_t **out, int device, uint64_t max_samples, uint32_t max_reads,
                 uint32_t n_slots, uint32_t flags);
void sgpu_destroy(sgpu_ctx_t *ctx);
const char *sgpu_strerror(int code);
const char *sgpu_last_error(const sgpu_ctx_t *ctx);
int  sgpu_abi_version(void);

/* ---- host path: pinned slots, async H2D -> kernels -> D2H ---------------- */
/* Pinned input buffers of a slot (valid until destroy). */
int  sgpu_slot_batch(sgpu_ctx_t *ctx, uint32_t slot, sgpu_batch_t **out);
/* Start a new batch in the slot. */
int  sgpu_slot_reset(sgpu_ctx_t *ctx, uint32_t slot, uint32_t rna);
/* Append one decoded record (the fields of slow5_rec_t the path uses,
 * slow5.h:274-286).  Returns the read's index in the batch, SGPU_E_FULL when
 * it does not fit (submit and retry), SGPU_E_TOOBIG when it can never fit. */
int64_t sgpu_slot_add_read(sgpu_ctx_t *ctx, uint32_t slot, const int16_t *raw, uint64_t len_raw_signal,
                           double digitisation, double offset, double range);
/* Append one record whose raw signal is STILL svb-zd compressed: `stream` is the record's raw_signal field as
 * slow5lib stores it with SLOW5_COMPRESS_SVB_ZD (uint32 count | ceil(count/4) key bytes | data bytes), i.e. what
 * ptr_depress_svb_zd() (slow5lib/src/slow5_press.c:1116-1150; streamvbyte_decode.c:30-83,
 * streamvbyte_zigzag.c:27-47) would expand on the CPU. Only these bytes cross PCIe; the int16 samples are
 * produced in HBM (svbzd.cu). A batch holds either decoded records or svb-zd streams (SGPU_E_STATE when mixed).
 * A stream whose length contradicts its header is refused here (SGPU_E_STREAM); one whose length contradicts its
 * keys is reported by sgpu_wait (SGPU_E_STREAM), like slow5lib's error at slow5_press.c:1103. */
int64_t sgpu_slot_add_read_svbzd(sgpu_ctx_t *ctx, uint32_t slot, const uint8_t *stream, uint64_t n_bytes,
                                 double digitisation, double offset, double range);
/* Append one record given as pA floats: getevents(n, pa, rna) (events.c:553-573) on the caller's own signal
 * (calibrated, normalised, simulated or filtered), where the other entry points take int16 raw samples. Such a slot
 * holds pA records only (SGPU_E_STATE when mixed with decoded records or svb-zd streams) and computes
 * SGPU_WANT_EVENTS only (sgpu_submit returns SGPU_E_INVAL for any other bit). The floats are kept in the slot's
 * sample buffers: a slot holds max_samples / 2 pA samples, every read padded to SGPU_ALIGN of them (SGPU_E_FULL when
 * the next read does not fit, SGPU_E_TOOBIG when align_up(n, SGPU_ALIGN) > max_samples / 2). Results are bit-identical
 * to the reference's for every finite input; with NaN or Inf in the input the event boundaries are identical and the
 * NaN statistics are NaN in the same places. The read's offset_f / raw_unit_f in sgpu_batch_t read 0 and 1. */
int64_t sgpu_slot_add_read_pa(sgpu_ctx_t *ctx, uint32_t slot, const float *pa, uint64_t n);
/* Asynchronous: copies the slot to the device, runs the kernels, copies the
 * results back, all on the slot's stream. */
int  sgpu_submit(sgpu_ctx_t *ctx, uint32_t slot, uint32_t want);
/* Blocks until the slot's work is done; fills *out with pinned host pointers. */
int  sgpu_wait(sgpu_ctx_t *ctx, uint32_t slot, sgpu_result_t *out);

/* ---- device-resident path (benchmarks, callers that already hold the data in HBM) ---- */
typedef struct {
    const int16_t  *samples;    /* device */
    const uint64_t *read_off;   /* device [n_reads+1] */
    const uint32_t *read_len;   /* device [n_reads] */
    const float    *offset_f;   /* device [n_reads] */
    const float    *raw_unit_f; /* device [n_reads] */
    uint32_t n_reads;
    uint32_t rna;
    uint64_t span;              /* = read_off[n_reads] (known to the host) */
} sgpu_dev_batch_t;

/* Runs the kernels on `stream` (a cudaStream_t passed as void*, NULL = the
 * legacy default stream) without any host<->device copies or synchronisation.
 * *out receives DEVICE pointers owned by the context (valid until the next
 * run on this context). */
int  sgpu_run_device(sgpu_ctx_t *ctx, const sgpu_dev_batch_t *batch, uint32_t want,
                     void *stream, sgpu_result_t *out);

/* Device-resident event detection on the caller's pA floats (see sgpu_slot_add_read_pa): read r occupies
 * pa[read_off[r] .. read_off[r]+read_len[r]), every read_off[r] a multiple of SGPU_ALIGN -- the layout of the `pa`
 * output, so the pA of an int16 run can be fed straight back in. span <= max_samples. want must be SGPU_WANT_EVENTS.
 * Runs on `stream` without copies or synchronisation, like sgpu_run_device; *out receives the event table, seq_order
 * (1: the read's prefix sums were formed in the reference's order because a parallel scan could round) and fixups
 * (detector chunks whose warm-up state did not match), the other pointers NULL. The first batch whose span exceeds the
 * context's sequential-order scratch (an eighth of max_samples above 64 Mi samples) grows it to max_samples, which
 * allocates and synchronises the device once. */
typedef struct {
    const float    *pa;         /* device */
    const uint64_t *read_off;   /* device [n_reads+1] */
    const uint32_t *read_len;   /* device [n_reads] */
    uint32_t n_reads;
    uint32_t rna;
    uint64_t span;              /* = read_off[n_reads] (known to the host) */
} sgpu_dev_pa_batch_t;
int  sgpu_run_device_pa(sgpu_ctx_t *ctx, const sgpu_dev_pa_batch_t *batch, uint32_t want, void *stream,
                        sgpu_result_t *out);

/* Device-resident svb-zd decode (benchmarks / callers that hold the compressed records in HBM). All pointers are
 * DEVICE pointers; `bytes` holds the streams back to back, each starting on a 16-byte boundary, and its
 * allocation extends at least 8 bytes past n_bytes. n_blocks = sum over reads of ceil(read_len / 1024).
 * Writes read r's samples to samples_out[read_off[r] ..]. No synchronisation; a malformed stream shows as
 * status SGPU_E_STREAM in sgpu_counters(). */
typedef struct {
    const uint8_t  *bytes;
    uint64_t        n_bytes;
    const uint64_t *comp_off;   /* [n_reads] */
    const uint32_t *comp_len;   /* [n_reads] */
    const uint64_t *read_off;   /* [n_reads+1] multiples of SGPU_ALIGN */
    const uint32_t *read_len;   /* [n_reads] = the count in each stream's header */
    uint32_t n_reads;
    uint64_t n_blocks;
} sgpu_svb_dev_batch_t;
int  sgpu_decode_svbzd_device(sgpu_ctx_t *ctx, const sgpu_svb_dev_batch_t *batch, int16_t *samples_out, void *stream);

/* ---- live event detection: signal that arrives in chunks, channel by channel ----------------------------------
 * For tools that segment signal while the read is still in the pore (adaptive sampling, Read Until): per channel, a
 * read is opened by a START entry, grows by entries of samples and is closed by an END entry; one entry may carry
 * START, samples and END together. The context keeps every channel's detector state in HBM between entries.
 *   - Two forms of entry: int16 samples with a calibration (sgpu_slot_add_live, sgpu_run_device_live), or pA floats
 *     taken as they are (sgpu_slot_add_live_pa, sgpu_run_device_live_pa: calibrated, filtered, normalised or simulated
 *     signal). A read keeps the form of the entry that carries its START: an entry without START on a channel whose
 *     read is open must have that form, whatever its length and flags (an empty entry too), else it is refused with
 *     SGPU_E_STATE like the other violations below. A START entry of either form discards an open read of either form.
 *   - pA of every int16 sample is misc.c:28 with the calibration given at START (offset_f = (float)offset, raw_unit_f =
 *     (float)range / (float)digitisation, as sgpu_slot_add_read computes them); the DNA or RNA parameters also come
 *     from START (SGPU_LIVE_RNA, ignored without START). The long threshold follows SGPU_PARAM_THR_LONG. With a
 *     detector set (sgpu_set_detector) the read runs the set in force for its START entry instead.
 *   - When events are reported: let a read hold n samples after an entry that does not end it. The detector has then
 *     been stepped, in the reference's order (short, then long; events.c:385-437), over every position
 *     i <= n - max(w1, w2) (n - w2 for the reference's sets): the positions whose t-statistics can no longer change
 *     (both right windows [i, i+w) are complete). Every peak
 *     emitted during those steps closes one event [a, p), and the entry reports those events. END steps the remaining
 *     positions (their long t-statistic is 0, events.c:328-338) and reports the last event [a, n). A read with no peak
 *     ends with the single event [0, n); a read of 0 samples reports no event. A peak may be emitted long after its
 *     position, in a later entry.
 *   - Exactness: for every read, the events of all its entries taken in order are bit-identical to the event table of
 *     the whole read (getevents, events.c:553-573, and sgpu_slot_add_read), for any split into chunks. For a read of
 *     pA entries this holds for every finite input, against getevents(n, pa, rna) and sgpu_slot_add_read_pa (the
 *     prefix sums are formed one sample after another in the reference's order, so no exactness witness is needed);
 *     with NaN or Inf in the input the event boundaries are identical and the NaN statistics are NaN in the same
 *     places.
 *   - Ordering: live runs of a context update channel state in the order they are submitted (host slots run their
 *     kernels on one stream of the context). A device-resident live run is ordered by the caller's stream and must not
 *     overlap a submitted live slot.
 *   - START on a channel whose read is still open discards that read: its open event is never reported.
 * A live slot holds live entries of one form only (SGPU_E_STATE when mixed with other records or with entries of the
 * other form) in its int16 sample buffers, and computes SGPU_WANT_EVENTS only (sgpu_submit returns SGPU_E_INVAL for any
 * other want). sgpu_wait on a live slot and sgpu_wait_live on any other slot return SGPU_E_STATE. sgpu_slot_add_live
 * returns the entry's index, SGPU_E_FULL / SGPU_E_TOOBIG as sgpu_slot_add_read does (sgpu_slot_add_live_pa: as
 * sgpu_slot_add_read_pa does, max_samples / 2 floats a slot, and never a read of 2^31 samples), SGPU_E_INVAL for
 * channel >= n_channels, unknown flag bits or a second entry for the channel in the slot, SGPU_E_STATE before
 * sgpu_live_open. sgpu_submit checks the rules that depend on channel state against a host mirror updated in
 * submission order: samples or END for a channel without an open read, or an entry that continues a read of the other
 * form, give SGPU_E_STATE, a read that would exceed 2^31 - 1 samples (misc.c:20) SGPU_E_TOOBIG; then nothing is queued
 * and no channel changes. sgpu_run_device_live reports the same violations as `status` in sgpu_counters, and the offending
 * entries leave their channels unchanged. The event capacity covers every possible push (SGPU_E_EVCAP cannot occur). */
#define SGPU_LIVE_START 1u /* begin a new read on the channel: calibration (and SGPU_LIVE_RNA) taken from this entry */
#define SGPU_LIVE_END   2u /* the read ends after this entry's samples */
#define SGPU_LIVE_RNA   4u /* with START: the RNA detector parameters (events.c:50-54) */

/* Once per context: a table of n_channels channels in HBM (about 550 bytes each), all without a read.
 * SGPU_E_STATE the second time. */
int  sgpu_live_open(sgpu_ctx_t *ctx, uint32_t n_channels);
/* Append one entry to a live slot (digitisation, offset, range are read with SGPU_LIVE_START only). */
int64_t sgpu_slot_add_live(sgpu_ctx_t *ctx, uint32_t slot, uint32_t channel, uint32_t flags, const int16_t *raw,
                           uint64_t n, double digitisation, double offset, double range);
/* Append one live entry given as pA floats (channel, SGPU_LIVE_* flags as for sgpu_slot_add_live; no calibration). */
int64_t sgpu_slot_add_live_pa(sgpu_ctx_t *ctx, uint32_t slot, uint32_t channel, uint32_t flags, const float *pa,
                              uint64_t n);
/* Events of a live run, entry by entry: host pointers (pinned) from sgpu_wait_live, device pointers from
 * sgpu_run_device_live (n_events 0 there: see sgpu_counters). */
typedef struct {
    uint64_t *ev_off;      /* [n_entries+1]: the events of entry e are [ev_off[e], ev_off[e+1]) */
    uint32_t *ev_start;    /* sample index in the channel's read */
    uint32_t *ev_len;      /* end - start */
    float    *ev_mean;
    float    *ev_stdv;
    uint64_t  n_events;
} sgpu_live_result_t;
/* Blocks until a live slot submitted with SGPU_WANT_EVENTS is done. */
int  sgpu_wait_live(sgpu_ctx_t *ctx, uint32_t slot, sgpu_live_result_t *out);
/* Device-resident live entries: entry e is samples[read_off[e] .. +read_len[e]) of channel[e] with flags[e], and the
 * calibration offset_f[e], raw_unit_f[e] (read with SGPU_LIVE_START only). read_off[e] + read_len[e] <= read_off[e+1],
 * read_off[n_entries] = span <= max_samples, n_entries <= max_reads. Runs on `stream` without copies or
 * synchronisation; *out receives device pointers owned by the context (valid until the next run). */
typedef struct {
    const int16_t  *samples;
    const uint64_t *read_off;   /* [n_entries+1] */
    const uint32_t *read_len;
    const uint32_t *channel;
    const uint32_t *flags;
    const float    *offset_f;
    const float    *raw_unit_f;
    uint32_t n_entries;
    uint64_t span;
} sgpu_dev_live_batch_t;
int  sgpu_run_device_live(sgpu_ctx_t *ctx, const sgpu_dev_live_batch_t *batch, void *stream, sgpu_live_result_t *out);
/* Device-resident live entries of pA floats: as sgpu_run_device_live, entry e is pa[read_off[e] .. +read_len[e]). */
typedef struct {
    const float    *pa;         /* device; entry e is pa[read_off[e] .. +read_len[e]) */
    const uint64_t *read_off;   /* [n_entries+1] */
    const uint32_t *read_len;
    const uint32_t *channel;
    const uint32_t *flags;
    uint32_t n_entries;
    uint64_t span;              /* = read_off[n_entries] <= max_samples */
} sgpu_dev_live_pa_batch_t;
int  sgpu_run_device_live_pa(sgpu_ctx_t *ctx, const sgpu_dev_live_pa_batch_t *batch, void *stream,
                             sgpu_live_result_t *out);

/* Counters of the last completed run (host path: after sgpu_wait; device path:
 * after the caller synchronised the stream). Synchronises the device. */
typedef struct {
    uint64_t n_events;
    uint64_t n_seq_order_reads;   /* reads routed to the sequential-order kernels */
    uint64_t n_fixups;            /* detector chunks with a boundary-state mismatch */
    uint64_t n_kernel_launches;   /* kernels launched by the last run */
    int32_t  status;              /* 0 or SGPU_E_EVCAP / SGPU_E_SCRATCH reported by the device; after a live run also
                                     SGPU_E_INVAL / SGPU_E_STATE / SGPU_E_TOOBIG for refused entries */
    uint64_t n_long_jobs;         /* stretches of the long peak detector (events.c:414-437) that were replayed with the
                                     reference's own operations because their t-statistic may exceed its threshold */
} sgpu_counters_t;
int  sgpu_counters(sgpu_ctx_t *ctx, sgpu_counters_t *out);

/* Development / test parameters of a context (take effect from the next run; nothing reads the environment).
 * They never change results -- except SGPU_PARAM_THR_LONG, which replaces the reference's constant 9.0
 * (events.c:46,53) so that tests can make the long detector emit. */
#define SGPU_PARAM_CHUNK_LEN 1 /* samples per detector chunk (multiple of 32, >= 128 DNA / 512 RNA); 0 = automatic */
#define SGPU_PARAM_WARMUP    2 /* detector warm-up in samples (multiple of 8 DNA / 16 RNA, <= default); 0 = default */
#define SGPU_PARAM_THR_LONG  3 /* threshold of the long detector */
#define SGPU_PARAM_PORE      4 /* 0: R9 (JNNV2_RNA_R9_ADAPTOR), 1: RNA004 (JNNV2_RNA_RNA004_ADAPTOR), jnn.h:88-102: the
                                  host picks it from the BLOW5 header like pore_detect (misc.c:74-101); used by
                                  SGPU_WANT_PREFIX only (not a test parameter) */
#define SGPU_PARAM_STAT_CTA_MIN 5 /* stat / jnn moments: reads of at least this many samples are added up by a CTA
                                  (several warps per read), shorter ones by one warp; 0 = every read by a CTA */
int  sgpu_set_param(sgpu_ctx_t *ctx, int key, double value);

/* ---- the caller's own detector parameters -------------------------------------------------------------------
 * The reference's detector takes a detector_param (events.c:35-41); getevents uses one of two constant sets chosen by
 * rna (events.c:43-54: DNA {3, 6, 1.4, 9.0, 0.2}, RNA {7, 14, 2.5, 9.0, 1.0}). sgpu_set_detector makes every event
 * detection of the context use the caller's set instead, as short_long_peak_detector(..., &set) would:
 *   - Scope: int16 records, svb-zd streams and pA records, on host slots and in device-resident runs, and live
 *     entries of both forms. rna and SGPU_LIVE_RNA then no longer choose the event parameters (they still choose those
 *     of SGPU_WANT_JNN and SGPU_WANT_PREFIX), and SGPU_PARAM_THR_LONG is ignored. The other products of a batch (PA,
 *     STAT, ENT, JNN, PREFIX) do not depend on it.
 *   - When it takes effect: a host slot runs the set in force at its sgpu_submit (two slots in flight may carry
 *     different sets); a device-resident run the set in force when it is called; a live read the set in force for its
 *     START entry, until its END, whatever is set in between (like the form of its START entry).
 *   - Results: for every finite input the events are bit-identical to the reference's getevents with short_long_peak_
 *     detector called with the set (the event table of the detector's peaks, events.c:457-504); with NaN or Inf in pA
 *     input the boundaries are identical and the NaN statistics are NaN in the same places. Batches with a set run on
 *     the route of pA records whatever their input (seq_order and fixups have the meaning given at
 *     sgpu_run_device_pa; no long-detector job runs), so a set equal to a reference set gives the default path's events
 *     bit for bit on another route. The batch event capacity (max_samples / 3 + 2 max_reads + 16) is not proved for
 *     every set: a batch that exceeds it returns SGPU_E_EVCAP, never a truncated table. Live runs cannot exceed theirs:
 *     the first live run under a set whose detectors may emit more often than the DNA set's grows the live staging
 *     and event outputs by a quarter, which allocates and synchronises the device once.
 *   - Live finality: after an entry that does not end its read (n samples so far), the positions stepped are
 *     i <= n - max(w_short, w_long) (for the reference sets, w_long > w_short: i <= n - w_long).
 * NULL restores the reference's sets (chosen by rna). Returns SGPU_E_INVAL, leaving the setting as it was, for a window
 * outside [2, 14] (a window below 2 has no t-statistic, events.c:328-330; 14 is the reference's largest) or a threshold
 * or peak_height that is not finite. w_short > w_long is allowed, as in the reference. */
typedef struct {                  /* detector_param, events.c:35-41 */
    uint32_t w_short, w_long;     /* window_length1, window_length2 */
    float    thr_short, thr_long; /* threshold1, threshold2 */
    float    peak_height;
} sgpu_detector_t;
int  sgpu_set_detector(sgpu_ctx_t *ctx, const sgpu_detector_t *p);

/* Device time of every kernel group of the last run, measured with CUDA events on the stream the kernels were
 * launched on (needs SGPU_F_STAGE_TIMERS). Returns the number of entries written, or a negative code. */
typedef struct {
    const char *name;     /* e.g. "walk_chunks", "emit_events" */
    float       ms;
    uint32_t    launches; /* kernels in the group */
} sgpu_stage_time_t;
int  sgpu_stage_times(sgpu_ctx_t *ctx, sgpu_stage_time_t *out, uint32_t cap);

/* Copies `bytes` from a device pointer returned by sgpu_run_device() to host memory (synchronous;
 * for callers of the device-resident path that have no CUDA runtime of their own). */
int  sgpu_memcpy_d2h(sgpu_ctx_t *ctx, void *dst_host, const void *src_device, uint64_t bytes);

#ifdef __cplusplus
}
#endif
#endif /* SIGTK_B200_H */
