// capi.cu -- the C-ABI of the sigtk B200 hot path (include/sigtk_b200.h).
//
// Context = one device, its workspace in HBM, and n_slots pinned host slots.
// Host path per slot:  H2D (slot stream) -> kernels (context compute stream) -> D2H (slot stream),
// chained with events so that copies of one slot overlap the kernels of another while the
// kernels themselves are serialised (they share one scratch area).
#include "../../include/sigtk_b200.h"

#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <new>
#include <utility>

#include "kernels.cuh"

using namespace sgpu;

namespace {

// The output arrays. OUTS describes each per-batch output once, LIVE_OUTS each output of a live run; every place that
// allocates, clears, copies back or returns outputs loops over one of them. Device and pinned host copies are arrays of
// byte buffers indexed by Out (or Live).
enum Out { EV_OFF, EV_START, EV_MEAN, EV_STDV, SEQ_ORDER, FIXUPS, STAT, ENT, JNN_CNT, JNN_SEG, PREFIX_POS, PREFIX_STAT,
           PA, N_OUT };
enum Live { LIVE_EV_OFF, LIVE_EV_START, LIVE_EV_LEN, LIVE_EV_MEAN, LIVE_EV_STDV, N_LIVE_OUT };
static_assert(EV_OFF == 0 && LIVE_EV_OFF == 0, "row 0 of both tables: ev_off, which sizes the event outputs");

// what an output's element count is proportional to (times OutSpec::per)
enum Count : uint8_t {
    READS, READS_PLUS_1, EVENTS,
    SAMPLES,    // of the batch's span
    JNN_SLOTS,  // jnn_seg_capacity(): segment slots of the span's reads (SGPU_JNN_BASE)
};

constexpr int ANY_WANT = 0x100;  // OutSpec::empty flag: cleared for an empty batch whatever the want

struct OutSpec {
    size_t field;    // offset of its pointer in sgpu_result_t (LIVE_OUTS: sgpu_live_result_t)
    uint32_t size;   // bytes per element
    uint32_t want;   // SGPU_WANT_* bit of the product it belongs to
    Count count;
    uint32_t per;
    bool eager;      // allocated up front (returned by every device-resident run), else on the first run that wants it
    int empty;       // byte every element holds for a batch of empty records (| ANY_WANT), or -1: left as it is
    bool pa_in;      // produced by a run on the caller's pA floats (sgpu_run_device_pa, slots of pA records)
};

#define OUTPUT(field, want, count, per, eager, empty, pa_in) \
    { offsetof(sgpu_result_t, field), sizeof *sgpu_result_t{}.field, want, count, per, eager, empty, pa_in }
constexpr OutSpec OUTS[] = {  // in the order of Out
    //     field        want              count         per  eager  empty         pa_in
    OUTPUT(ev_off,      SGPU_WANT_EVENTS, READS_PLUS_1, 1,   true,  0 | ANY_WANT, true),
    OUTPUT(ev_start,    SGPU_WANT_EVENTS, EVENTS,       1,   true,  -1,           true),
    OUTPUT(ev_mean,     SGPU_WANT_EVENTS, EVENTS,       1,   true,  -1,           true),
    OUTPUT(ev_stdv,     SGPU_WANT_EVENTS, EVENTS,       1,   true,  -1,           true),
    OUTPUT(seq_order,   SGPU_WANT_EVENTS, READS,        1,   true,  0,            true),
    OUTPUT(fixups,      SGPU_WANT_EVENTS, READS,        1,   true,  0,            true),
    OUTPUT(stat,        SGPU_WANT_STAT,   READS,        6,   true,  0,            false),
    OUTPUT(ent,         SGPU_WANT_ENT,    READS,        3,   false, 0,            false),
    OUTPUT(jnn_cnt,     SGPU_WANT_JNN,    READS,        1,   false, 0,            false),
    OUTPUT(jnn_seg,     SGPU_WANT_JNN,    JNN_SLOTS,    2,   false, -1,           false),
    OUTPUT(prefix_pos,  SGPU_WANT_PREFIX, READS,        4,   false, 0xff,         false),  // -1: not longer than the window
    OUTPUT(prefix_stat, SGPU_WANT_PREFIX, READS,        6,   false, 0,            false),
    OUTPUT(pa,          SGPU_WANT_PA,     SAMPLES,      1,   false, -1,           false),
};
#undef OUTPUT
static_assert(sizeof OUTS / sizeof OUTS[0] == N_OUT, "one row per output");

// the events of a live run, entry by entry (EVENTS: at the capacity LiveScratch::ev_cap)
#define LIVE_OUTPUT(field, count, empty) \
    { offsetof(sgpu_live_result_t, field), sizeof *sgpu_live_result_t{}.field, SGPU_WANT_EVENTS, count, 1, true, empty, \
      false }
constexpr OutSpec LIVE_OUTS[] = {  // in the order of Live
    LIVE_OUTPUT(ev_off,   READS_PLUS_1, 0 | ANY_WANT),
    LIVE_OUTPUT(ev_start, EVENTS,       -1),
    LIVE_OUTPUT(ev_len,   EVENTS,       -1),
    LIVE_OUTPUT(ev_mean,  EVENTS,       -1),
    LIVE_OUTPUT(ev_stdv,  EVENTS,       -1),
};
#undef LIVE_OUTPUT
static_assert(sizeof LIVE_OUTS / sizeof LIVE_OUTS[0] == N_LIVE_OUT, "one row per output");

// the products a run on pA input can compute: those of its outputs (the others are defined on int16 raw samples, and
// pA is the input itself)
constexpr uint32_t pa_input_wants(int k = 0) {
    return k == N_OUT ? 0u : (OUTS[k].pa_in ? OUTS[k].want : 0u) | pa_input_wants(k + 1);
}
constexpr bool pa_input_want_ok(uint32_t want) { return want != 0 && (want & ~pa_input_wants()) == 0; }
static_assert(pa_input_wants() == SGPU_WANT_EVENTS, "a pA run computes the event table only");

// elements of output s for a batch of `reads` reads spanning `samples` samples with `events` events; at the
// context's (max_reads, max_samples) and the table's event capacity this is the output's capacity
uint64_t out_elems(const OutSpec& s, uint64_t reads, uint64_t samples, uint64_t events) {
    switch (s.count) {
        case READS: return s.per * reads;
        case READS_PLUS_1: return s.per * (reads + 1);
        case EVENTS: return s.per * events;
        case SAMPLES: return s.per * samples;
        case JNN_SLOTS: return s.per * jnn_seg_capacity(samples, (uint32_t)reads);
    }
    return 0;
}

// What a slot holds between two sgpu_slot_reset: records of one kind, never a mix (NONE: nothing appended yet; it submits
// as an empty batch of int16 records). allowed_wants() is what each kind can compute. LIVE and LIVE_PA are live entries
// of int16 samples and of pA floats.
enum class Input : uint8_t { NONE, RAW, SVBZD, PA, LIVE, LIVE_PA };

bool is_live(Input k) { return k == Input::LIVE || k == Input::LIVE_PA; }

uint32_t allowed_wants(Input k) {
    if (k == Input::PA) return pa_input_wants();
    if (is_live(k)) return SGPU_WANT_EVENTS;
    return 63u;
}

struct Slot {
    // pinned host input: the fields of `batch` (what sgpu_slot_batch hands out) point at the five arrays below it
    sgpu_batch_t batch{};
    PinBuf<int16_t> samples;
    PinBuf<uint64_t> read_off;
    PinBuf<uint32_t> read_len;
    PinBuf<float> offset_f, raw_unit_f;
    uint64_t used = 0;
    // device input
    DevBuf<int16_t> d_samples;
    DevBuf<uint64_t> d_read_off;
    DevBuf<uint32_t> d_read_len;
    DevBuf<float> d_offset, d_unit;
    DevBuf<void> dout[N_OUT];  // device outputs
    PinBuf<void> hout[N_OUT];  // their pinned host copies
    PinBuf<unsigned long long> h_counters;  // [4]
    PinBuf<int> h_status;
    cudaStream_t stream = nullptr;
    cudaEvent_t in_ready = nullptr, kernels_done = nullptr, small_back = nullptr;
    bool submitted = false;
    uint32_t want = 0;
    const DetParams* det = nullptr;  // the context's detector set at sgpu_submit (&det_set), or nullptr: the reference's
    DetParams det_set{};
    Input kind = Input::NONE;        // (PA, LIVE_PA: the floats are in the sample buffers, max_samples / 2 of them)
    // svb-zd input (allocated on first use): the batch's compressed streams, decoded in HBM by svbzd.cu
    PinBuf<uint8_t> h_comp;          // comp_cap bytes
    DevBuf<uint8_t> d_comp;          // comp_cap + 16 bytes
    PinBuf<uint64_t> h_comp_off; DevBuf<uint64_t> d_comp_off;
    PinBuf<uint32_t> h_comp_len; DevBuf<uint32_t> d_comp_len;
    uint64_t comp_used = 0, svb_blocks = 0;
    // live entries (allocated by sgpu_live_open): channel and flags of every entry, the run's events
    PinBuf<uint32_t> h_channel, h_flags; DevBuf<uint32_t> d_channel, d_flags;
    DevBuf<void> live_dout[N_LIVE_OUT];
    PinBuf<void> live_hout[N_LIVE_OUT];
    uint64_t live_dcap = 0, live_hcap = 0;   // the event capacity they were allocated for
    std::unique_ptr<uint32_t[]> live_claim;  // [n_channels] live_gen of the batch that holds an entry for the channel
    uint32_t live_gen = 0;

    ~Slot() {
        if (stream) cudaStreamDestroy(stream);
        if (in_ready) cudaEventDestroy(in_ready);
        if (kernels_done) cudaEventDestroy(kernels_done);
        if (small_back) cudaEventDestroy(small_back);
    }
};

}  // namespace

struct sgpu_ctx {
    int device = 0;
    int sm_count = 148;
    uint64_t max_samples = 0;
    uint32_t max_reads = 0;
    uint32_t n_slots = 0;
    uint32_t flags = 0;
    uint64_t ev_cap = 0;
    Scratch sc{};
    DevBuf<void> dev_out[N_OUT]; // outputs of the device-resident path
    std::unique_ptr<Slot[]> slots;
    SvbScratch svb{};            // workspace of the svb-zd decoder (allocated on first use)
    DevBuf<float> jnn_mom;       // [max_reads][2] mean / stdv of the clamped signal (allocated on first use)
    int pore_rna004 = 0;         // SGPU_PARAM_PORE: jnnv2 parameters of `prefix` (misc.c:74-101 picks them from the header)
    bool det_on = false;         // sgpu_set_detector: every event detection uses `det` instead of the reference's sets
    DetParams det{};
    DevBuf<uint32_t> ent_ovf;    // overflow histograms of ent_kernel (allocated on first use, kept all-zero)
    PaScratch pa{};              // workspace of the pA-input path (allocated on first use)
    LiveScratch live{};          // channel table and workspace of live runs (sgpu_live_open)
    DevBuf<void> live_dev_out[N_LIVE_OUT];    // outputs of sgpu_run_device_live
    uint64_t live_dev_cap = 0;
    std::unique_ptr<uint32_t[]> live_mirror;  // [n_channels] nopen of every channel after the submitted live slots
    std::unique_ptr<uint8_t[]> live_form;     // [n_channels] and the form of its open read (LiveScratch::form)
    bool live_mirror_stale = false;           // a device-resident live run changed channels since
    uint32_t live_gen = 0;
    uint64_t comp_cap = 0;       // bytes of compressed input a slot can hold
    cudaStream_t compute = nullptr;
    uint64_t last_launches = 0;
    // optional per-stage CUDA-event timers (SGPU_F_STAGE_TIMERS)
    static constexpr int MAX_STAGES = 16;
    cudaEvent_t stage_ev[MAX_STAGES + 1] = {};
    const char* stage_name[MAX_STAGES] = {};
    uint32_t stage_launches[MAX_STAGES] = {};
    int n_stages = 0;
    cudaStream_t stage_stream = nullptr;
    char err[512] = {0};

    ~sgpu_ctx() {
        if (compute) cudaStreamDestroy(compute);
        for (cudaEvent_t e : stage_ev) if (e) cudaEventDestroy(e);
    }
};

namespace {

bool cuda_fail(sgpu_ctx* c, cudaError_t e, const char* what, int line) {
    if (e == cudaSuccess) return false;
    if (c) snprintf(c->err, sizeof c->err, "%s: %s (%s) at capi.cu:%d", what, cudaGetErrorName(e),
                    cudaGetErrorString(e), line);
    return true;
}
#define CU(call)                                                         \
    do {                                                                 \
        if (cuda_fail(ctx, (call), #call, __LINE__)) return SGPU_E_CUDA; \
    } while (0)

uint64_t align_up(uint64_t v, uint64_t a) { return (v + a - 1) / a * a; }

// allocates (device or pinned) every output of the table `outs` that is eager or belongs to `want` and does not exist
// yet, at the context's max_reads, max_samples and the table's event capacity ev_cap
template <size_t N, bool PINNED>
cudaError_t alloc_outputs(const OutSpec (&outs)[N], const sgpu_ctx* ctx, uint64_t ev_cap, Buf<void, PINNED>* o,
                          uint32_t want) {
    for (size_t k = 0; k < N; k++) {
        if (!outs[k].eager && !(want & outs[k].want)) continue;
        const uint64_t n = out_elems(outs[k], ctx->max_reads, ctx->max_samples, ev_cap);
        const cudaError_t e = o[k].ensure(n * outs[k].size);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// points the fields of *r at the outputs of `want`, and at every eager output when `all_eager`; the others stay NULL
template <size_t N, typename R, bool PINNED>
void fill_result(const OutSpec (&outs)[N], R* r, const Buf<void, PINNED>* o, uint32_t want, bool all_eager) {
    for (size_t k = 0; k < N; k++)
        if ((want & outs[k].want) || (all_eager && outs[k].eager)) {
            void* const p = o[k];
            memcpy(reinterpret_cast<char*>(r) + outs[k].field, &p, sizeof p);
        }
}

// queues on the slot's stream the D2H copy (d to h) of every output of `want` that is sized by the batch's reads and
// samples, or (by_events) of every one sized by its n_events
template <size_t N>
cudaError_t queue_d2h(const OutSpec (&outs)[N], const DevBuf<void>* d, PinBuf<void>* h, const Slot& sl, uint32_t want,
                      bool by_events, uint64_t n_events) {
    for (size_t k = 0; k < N; k++) {
        if (!(want & outs[k].want) || (outs[k].count == EVENTS) != by_events) continue;
        const uint64_t n = out_elems(outs[k], sl.batch.n_reads, sl.used, n_events);
        const cudaError_t e = cudaMemcpyAsync(h[k], d[k], (size_t)n * outs[k].size, cudaMemcpyDeviceToHost, sl.stream);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// One run of a pipeline on a stream: start() zeroes the device status and counters, done() records a CUDA event after
// a kernel group when the context has stage timers, finish() checks the launches and keeps their number.
struct StageMarks {
    sgpu_ctx* ctx;
    cudaStream_t st;
    bool on;
    uint64_t launches = 0;
    StageMarks(sgpu_ctx* c, cudaStream_t s) : ctx(c), st(s), on((c->flags & SGPU_F_STAGE_TIMERS) != 0) {}
    int start() {
        CU(cudaMemsetAsync(ctx->sc.status, 0, sizeof(int), st));
        CU(cudaMemsetAsync(ctx->sc.counters, 0, 4 * sizeof(unsigned long long), st));
        ctx->n_stages = 0;
        ctx->stage_stream = st;
        if (on) cudaEventRecord(ctx->stage_ev[0], st);
        return SGPU_OK;
    }
    void done(const char* name, int n) {
        launches += (uint64_t)n;
        if (!on || ctx->n_stages >= sgpu_ctx::MAX_STAGES) return;
        const int k = ctx->n_stages++;
        ctx->stage_name[k] = name;
        ctx->stage_launches[k] = (uint32_t)n;
        cudaEventRecord(ctx->stage_ev[k + 1], st);
    }
    int finish() {
        CU(cudaGetLastError());
        ctx->last_launches = launches;
        return SGPU_OK;
    }
};

int alloc_svb_scratch(sgpu_ctx* ctx) {
    SvbScratch& w = ctx->svb;
    w.max_blocks = svbzd_max_blocks(ctx->max_samples, ctx->max_reads);
    CU(w.cnt.ensure(ctx->max_reads));
    CU(w.base.ensure((uint64_t)ctx->max_reads + 1));
    CU(w.blk_bytes.ensure(w.max_blocks));
    CU(w.blk_gpos.ensure(w.max_blocks + 1));
    CU(w.blk_sum.ensure(w.max_blocks));
    CU(w.blk_vpos.ensure(w.max_blocks + 1));
    CU(w.lane_sum.ensure(w.max_blocks * 32));
    CU(w.blk_read.ensure(w.max_blocks));
    return SGPU_OK;
}

// nothing but empty records: every per-read output gets its defined value for an empty record (no event, zero
// statistics / entropies / segments, "record not longer than the window" for prefix) instead of whatever the previous
// batch left in the buffers; the run launches no kernel
template <size_t N>
int clear_empty_batch(const OutSpec (&outs)[N], uint64_t reads, uint64_t span, uint32_t want, DevBuf<void>* o,
                      StageMarks& run) {
    sgpu_ctx* const ctx = run.ctx;
    for (size_t k = 0; k < N; k++) {
        const OutSpec& s = outs[k];
        if (s.empty < 0 || !((want & s.want) || (s.empty & ANY_WANT))) continue;
        const uint64_t n = out_elems(s, reads, span, 0);
        if (n) CU(cudaMemsetAsync(o[k], s.empty & 0xff, (size_t)n * s.size, run.st));
    }
    return run.finish();
}

bool fits(const sgpu_ctx* ctx, const DevBatch& b) {  // a batch of int16 or pA records the context can hold
    return b.n_reads <= ctx->max_reads && b.span <= ctx->max_samples && !(b.span & (SGPU_ALIGN - 1));
}

int alloc_pa_scratch(sgpu_ctx* ctx) {
    PaScratch& w = ctx->pa;
    w.max_tiles = pa_tile_capacity(ctx->max_samples, ctx->max_reads);
    CU(w.tile_cnt.ensure(ctx->max_reads));
    CU(w.tile_base.ensure((uint64_t)ctx->max_reads + 1));
    CU(w.tS.ensure(w.max_tiles));
    CU(w.tQ.ensure(w.max_tiles));
    CU(w.tA.ensure(w.max_tiles));
    CU(w.tB.ensure(w.max_tiles));
    CU(w.tmin.ensure(w.max_tiles));
    CU(w.ord_list.ensure(ctx->max_reads));
    CU(w.ord_sbase.ensure(ctx->max_reads));
    CU(w.ord_count.ensure(1));
    return SGPU_OK;
}

// The general route keeps its prefix sums and t-statistics at the reads' own offsets, so the sequential-order scratch
// must hold the whole span. Contexts over 64 Mi samples start with an eighth of that (sgpu_create); the first batch on
// the general route (pA records, or a batch with a detector set) that needs more grows it to max_samples for the rest
// of the context's life (later int16 batches use it too). The old arrays are freed only once the new ones exist
// (freeing waits for the device).
int grow_seq_scratch(sgpu_ctx* ctx) {
    Scratch& sc = ctx->sc;
    const uint64_t n = ctx->max_samples;
    DevBuf<double> S, Q;
    DevBuf<float> t1, t2;
    cudaError_t e = S.ensure(n);
    if (e == cudaSuccess) e = Q.ensure(n);
    if (e == cudaSuccess) e = t1.ensure(n);
    if (e == cudaSuccess) e = t2.ensure(n);
    if (e != cudaSuccess) {  // (the buffers that were allocated free themselves)
        cudaGetLastError();  // (an allocation failure is reported here, not by the next launch check)
        snprintf(ctx->err, sizeof ctx->err, "growing the sequential-order scratch to %llu samples: %s",
                 (unsigned long long)n, cudaGetErrorString(e));
        return SGPU_E_NOMEM;
    }
    sc.Sinc = std::move(S); sc.Qinc = std::move(Q); sc.t1 = std::move(t1); sc.t2 = std::move(t2);
    sc.gen_cap = n;
    return SGPU_OK;
}

// The general route's workspace for a batch of `span` samples: the tile arrays of pa_input.cu, and a sequential-order
// scratch that holds the whole span.
int prepare_general(sgpu_ctx* ctx, uint64_t span) {
    int rc = alloc_pa_scratch(ctx);
    if (!rc && span > ctx->sc.gen_cap) rc = grow_seq_scratch(ctx);
    return rc;
}

// The events of a batch on the general route into the device outputs `o`: the prefix sums by the witness-checked scan
// or in the reference's order (pa_input.cu), then the sequential-order kernels for every read. pa: the caller's
// floats, or nullptr: b's int16 samples through their calibration; set: the caller's detector set, or nullptr: the
// reference's chosen by b.rna. (prepare_general first.)
int general_events(sgpu_ctx* ctx, const DevBatch& b, const float* pa, const DetParams* set, DevBuf<void>* o,
                   StageMarks& marks) {
    Scratch& sc = ctx->sc;
    const cudaStream_t st = marks.st;
    const uint32_t n_tiles = fast_tiles_for(b.span);
    if (n_tiles > sc.max_tiles) return SGPU_E_INVAL;
    uint32_t* const seq = static_cast<uint32_t*>(o[SEQ_ORDER].get());
    uint32_t* const fix = static_cast<uint32_t*>(o[FIXUPS].get());
    CU(cudaMemsetAsync(sc.bitmap, 0, (size_t)n_tiles * (FAST_TILE / 32) * sizeof(uint32_t), st));
    const int force = (ctx->flags & SGPU_F_FORCE_GENERIC) ? 1 : 0;
    marks.done("pa_prefix", launch_pa_prefix(b, pa, ctx->pa, sc, seq, fix, force, ctx->sm_count, st));
    const WorkList ordered{ctx->pa.ord_list, ctx->pa.ord_sbase, ctx->pa.ord_count};
    const WorkList all{sc.seq_list, sc.seq_sbase, sc.seq_count};
    marks.done("sequential_order_detect",
               launch_generic_detect_pa(b, pa, set, ordered, all, sc, fix, ctx->sm_count, st));
    uint64_t* const ev_off = static_cast<uint64_t*>(o[EV_OFF].get());
    marks.done("rank_events", launch_rank_events(b, sc, ev_off, ctx->sm_count, st));
    marks.done("sequential_order_emit",
               launch_generic_emit(b, all, sc, ev_off, ctx->ev_cap, static_cast<uint32_t*>(o[EV_START].get()),
                                   static_cast<float*>(o[EV_MEAN].get()), static_cast<float*>(o[EV_STDV].get()),
                                   ctx->sm_count, st));
    return SGPU_OK;
}

// The kernel sequence of one batch into the device outputs `o`. No host synchronisation, no host<->device copies
// (except when the general route's scratch grows). set: the caller's detector set, whose events take the general
// route, or nullptr: the reference's sets on the fast path.
int run_pipeline(sgpu_ctx* ctx, const DevBatch& b, uint32_t want, DevBuf<void>* o, cudaStream_t st,
                 const DetParams* set, const SvbBatch* svb = nullptr, int16_t* svb_out = nullptr) {
    Scratch& sc = ctx->sc;
    if (!fits(ctx, b)) return SGPU_E_INVAL;
    CU(alloc_outputs(OUTS, ctx, ctx->ev_cap, o, want));
    const bool events = (want & SGPU_WANT_EVENTS) != 0;
    if (set && events)
        if (const int rc = prepare_general(ctx, b.span)) return rc;
    StageMarks marks(ctx, st);
    if (const int rc = marks.start()) return rc;
    if (b.n_reads == 0 || b.span == 0) return clear_empty_batch(OUTS, b.n_reads, b.span, want, o, marks);
    if (svb) marks.done("svbzd_decode", launch_svbzd_decode(*svb, ctx->svb, ctx->sc, svb_out, ctx->sm_count, st));
    const bool force_generic = (ctx->flags & SGPU_F_FORCE_GENERIC) != 0;
    float* const pa = (want & SGPU_WANT_PA) ? static_cast<float*>(o[PA].get()) : nullptr;
    uint32_t* const seq = static_cast<uint32_t*>(o[SEQ_ORDER].get());
    uint32_t* const fix = static_cast<uint32_t*>(o[FIXUPS].get());
    if (pa && (!events || force_generic || set))  // with events on the fast path the pA store is fused into walk_chunks_kernel
        marks.done("pa", launch_pa(b, pa, ctx->sm_count, st));
    if (want & SGPU_WANT_STAT) {
        float* const stat = static_cast<float*>(o[STAT].get());
        marks.done("stat_moments", launch_stat_moments(b, stat, ctx->sc.tune_stat_cta_min, ctx->sm_count, st));
        marks.done("stat_median", launch_stat_median(b, stat, ctx->sc.tune_stat_cta_min, ctx->sm_count, st));
    }
    if (want & SGPU_WANT_ENT) {
        if (!ctx->ent_ovf) {
            const uint64_t words = ent_overflow_words(ctx->sm_count);
            CU(ctx->ent_ovf.ensure(words));
            CU(cudaMemsetAsync(ctx->ent_ovf, 0, (size_t)words * sizeof(uint32_t), st));
        }
        marks.done("ent", launch_ent(b, ctx->ent_ovf, static_cast<double*>(o[ENT].get()), ctx->sm_count, st));
    }
    if (want & SGPU_WANT_JNN) {
        CU(ctx->jnn_mom.ensure((uint64_t)ctx->max_reads * 2));
        marks.done("jnn_moments", launch_jnn_moments(b, ctx->jnn_mom, ctx->sc.tune_stat_cta_min, ctx->sm_count, st));
        marks.done("jnn_walk", launch_jnn(b, ctx->jnn_mom, static_cast<uint32_t*>(o[JNN_CNT].get()),
                                          static_cast<int32_t*>(o[JNN_SEG].get()), ctx->sm_count, st));
    }
    if (want & SGPU_WANT_PREFIX)
        marks.done("prefix", launch_prefix(b, ctx->pore_rna004, static_cast<int32_t*>(o[PREFIX_POS].get()),
                                           static_cast<float*>(o[PREFIX_STAT].get()), ctx->sm_count, st));
    if (events && set) {
        if (const int rc = general_events(ctx, b, nullptr, set, o, marks)) return rc;
    } else if (events) {
        const uint32_t n_tiles = fast_tiles_for(b.span);
        if (n_tiles > sc.max_tiles) return SGPU_E_INVAL;
        int n = launch_init_reads(b, sc, seq, fix, ctx->sm_count, st);
        if (force_generic) {
            CU(cudaMemsetAsync(sc.bitmap, 0, (size_t)n_tiles * (FAST_TILE / 32) * sizeof(uint32_t), st));
            marks.done("init", n);
        } else {
            marks.done("init", n);
            marks.done("walk_chunks", launch_walk(b, sc, pa, seq, ctx->sm_count, st));
            marks.done("long_jobs", launch_long_jobs(b, sc, seq, ctx->sm_count, st));
            marks.done("verify_chunks", launch_verify_chunks(b, sc, seq, fix, ctx->sm_count, st));
        }
        n = launch_build_seq_list(b, sc, seq, force_generic ? 1 : 0, ctx->sm_count, st);
        WorkList wl{sc.seq_list, sc.seq_sbase, sc.seq_count};
        n += launch_generic_detect(b, wl, sc, ctx->sm_count, st);
        marks.done("sequential_order_detect", n);
        uint64_t* const ev_off = static_cast<uint64_t*>(o[EV_OFF].get());
        uint32_t* const ev_start = static_cast<uint32_t*>(o[EV_START].get());
        float* const ev_mean = static_cast<float*>(o[EV_MEAN].get());
        float* const ev_stdv = static_cast<float*>(o[EV_STDV].get());
        marks.done("rank_events", launch_rank_events(b, sc, ev_off, ctx->sm_count, st));
        marks.done("emit_events",
                   launch_fast_emit(b, sc, ctx->ev_cap, ev_start, ev_mean, ev_stdv, fix, ctx->sm_count, st));
        marks.done("sequential_order_emit",
                   launch_generic_emit(b, wl, sc, ev_off, ctx->ev_cap, ev_start, ev_mean, ev_stdv, ctx->sm_count, st));
    }
    return marks.finish();
}

// The kernel sequence of a batch of pA records (getevents(n, pa, rna), events.c:553-573) into the device outputs `o`:
// the general route (set: the caller's detector set, or nullptr: the reference's chosen by b.rna). No host
// synchronisation, no host<->device copies (except when the scratch grows).
int run_pipeline_pa(sgpu_ctx* ctx, const DevBatch& b, const float* pa, const DetParams* set, uint32_t want,
                    DevBuf<void>* o, cudaStream_t st) {
    if (!fits(ctx, b) || (b.n_reads && b.span && !pa)) return SGPU_E_INVAL;
    CU(alloc_outputs(OUTS, ctx, ctx->ev_cap, o, want));
    int rc = prepare_general(ctx, b.span);
    if (rc) return rc;
    StageMarks marks(ctx, st);
    if ((rc = marks.start())) return rc;
    if (b.n_reads == 0 || b.span == 0) return clear_empty_batch(OUTS, b.n_reads, b.span, want, o, marks);
    if ((rc = general_events(ctx, b, pa, set, o, marks))) return rc;
    return marks.finish();
}

// The kernels of a push of live entries into `o` (live.cu; pa: the entries are b.pa floats). No host synchronisation, no
// host<->device copies.
int run_pipeline_live(sgpu_ctx* ctx, const LiveBatch& b, bool pa, const DetParams* set, DevBuf<void>* o,
                      cudaStream_t st) {
    if (b.n_entries > ctx->max_reads || b.span > ctx->max_samples) return SGPU_E_INVAL;
    if (b.n_entries && (!b.samples || !b.read_off || !b.read_len || !b.channel || !b.flags ||
                        (!pa && (!b.offset || !b.unit))))
        return SGPU_E_INVAL;
    StageMarks marks(ctx, st);
    if (const int rc = marks.start()) return rc;
    // (entries without samples still open and close channels: only a push of no entry is empty)
    if (b.n_entries == 0) return clear_empty_batch(LIVE_OUTS, 0, b.span, SGPU_WANT_EVENTS, o, marks);
    marks.done(pa ? "live_pa" : "live",
               launch_live(b, pa, set, ctx->live, ctx->sc, static_cast<uint64_t*>(o[LIVE_EV_OFF].get()),
                           static_cast<uint32_t*>(o[LIVE_EV_START].get()), static_cast<uint32_t*>(o[LIVE_EV_LEN].get()),
                           static_cast<float*>(o[LIVE_EV_MEAN].get()), static_cast<float*>(o[LIVE_EV_STDV].get()),
                           ctx->sm_count, st));
    return marks.finish();
}

// The kernels of a slot's batch on the context's compute stream, from the slot's device input into its outputs.
int run_slot(sgpu_ctx* ctx, Slot& sl, uint32_t want) {
    const uint32_t nr = sl.batch.n_reads;
    const int rna = (int)sl.batch.rna;
    if (is_live(sl.kind)) {  // (LIVE_PA: the union's pa is the same pointer, the floats in the sample buffers)
        const LiveBatch b{sl.d_samples, sl.d_read_off, sl.d_read_len, sl.d_channel, sl.d_flags, sl.d_offset, sl.d_unit,
                          nr, sl.used};
        return run_pipeline_live(ctx, b, sl.kind == Input::LIVE_PA, sl.det, sl.live_dout, ctx->compute);
    }
    CU(alloc_outputs(OUTS, ctx, ctx->ev_cap, sl.hout, want));
    if (sl.kind == Input::PA)
        return run_pipeline_pa(ctx, DevBatch{nullptr, sl.d_read_off, sl.d_read_len, nullptr, nullptr, nr, rna, sl.used},
                               reinterpret_cast<const float*>(sl.d_samples.get()), sl.det, want, sl.dout, ctx->compute);
    const DevBatch b{sl.d_samples, sl.d_read_off, sl.d_read_len, sl.d_offset, sl.d_unit, nr, rna, sl.used};
    const SvbBatch svb{sl.d_comp, sl.comp_used, sl.d_comp_off, sl.d_comp_len, sl.d_read_off, sl.d_read_len, nr,
                       sl.svb_blocks};
    return run_pipeline(ctx, b, want, sl.dout, ctx->compute, sl.det, sl.kind == Input::SVBZD ? &svb : nullptr,
                        sl.d_samples);
}

// a slot that is not submitted takes a record of kind k when it is empty or holds records of kind k
bool accepts(const Slot& sl, Input k) { return !sl.submitted && (sl.kind == Input::NONE || sl.kind == k); }

// whether a record of n samples fits a slot of `cap` samples: never when n reaches `limit` or the record, padded to
// SGPU_ALIGN, exceeds cap (SGPU_E_TOOBIG); not now when the slot has no room left for it (SGPU_E_FULL)
int room_for(const sgpu_ctx* ctx, const Slot& sl, uint64_t n, uint64_t limit, uint64_t cap) {
    const uint64_t need = align_up(n, SGPU_ALIGN);
    if (n >= limit || need > cap) return SGPU_E_TOOBIG;
    if (sl.batch.n_reads >= ctx->max_reads || sl.used + need > cap) return SGPU_E_FULL;
    return SGPU_OK;
}

// The per-read tail of every sgpu_slot_add_*: records the read of n samples at sl.used as
// the batch's next read, with the scalars of its pA conversion.
int64_t append_record(Slot& sl, uint64_t n, double digitisation, double offset, double range) {
    sgpu_batch_t& b = sl.batch;
    const uint32_t r = b.n_reads;
    b.read_off[r] = sl.used;
    b.read_len[r] = (uint32_t)n;
    // misc.c:17-19,26: narrow the three doubles to float first, then ONE float division
    const float range_f = (float)range, dig_f = (float)digitisation, off_f = (float)offset;
    volatile float unit = range_f / dig_f;
    b.offset_f[r] = off_f;
    b.raw_unit_f[r] = unit;
    sl.used += align_up(n, SGPU_ALIGN);
    b.n_reads = r + 1;
    b.read_off[r + 1] = sl.used;
    return (int64_t)r;
}

// The checks of sgpu_slot_add_live and sgpu_slot_add_live_pa in their order, then the entry's channel and flags: an
// entry of kind k (LIVE or LIVE_PA) of n samples in a slot that holds `cap` of them. The caller copies the samples.
int add_live_entry(sgpu_ctx* ctx, Slot& sl, Input k, uint32_t channel, uint32_t flags, uint64_t n, uint64_t cap) {
    if (!accepts(sl, k) || !ctx->live.n_channels) return SGPU_E_STATE;
    if (channel >= ctx->live.n_channels || (flags & ~LIVE_FLAGS)) return SGPU_E_INVAL;
    // (2^31 samples: a read may not reach them, misc.c:20)
    if (const int rc = room_for(ctx, sl, n, 1ull << 31, cap)) return rc;
    if (sl.kind != k) {  // the slot's first entry: a new generation of its channel marks
        if (++ctx->live_gen == 0) {
            for (uint32_t s = 0; s < ctx->n_slots; s++)
                memset(ctx->slots[s].live_claim.get(), 0, (size_t)ctx->live.n_channels * sizeof(uint32_t));
            ctx->live_gen = 1;
        }
        sl.live_gen = ctx->live_gen;
    }
    if (sl.live_claim[channel] == sl.live_gen) return SGPU_E_INVAL;  // one entry per channel and slot
    sl.live_claim[channel] = sl.live_gen;
    sl.kind = k;
    sl.h_channel[sl.batch.n_reads] = channel;
    sl.h_flags[sl.batch.n_reads] = flags;
    return SGPU_OK;
}

int map_dev_status(int s) {
    if (s == SGPU_DEV_E_EVCAP) return SGPU_E_EVCAP;
    if (s == SGPU_DEV_E_INVAL) return SGPU_E_INVAL;
    if (s == SGPU_DEV_E_STATE) return SGPU_E_STATE;
    if (s == SGPU_DEV_E_TOOBIG) return SGPU_E_TOOBIG;
    if (s == SGPU_DEV_E_SCRATCH) return SGPU_E_SCRATCH;
    if (s == SGPU_DEV_E_STREAM) return SGPU_E_STREAM;
    return SGPU_OK;
}

uint8_t live_form_of(Input k) { return k == Input::LIVE_PA ? LIVE_FORM_PA : LIVE_FORM_INT16; }

// sgpu_submit of a live slot: the rules that depend on channel state, against the host mirror of the channels
// (entries of one slot have distinct channels); nothing is queued and no channel changes unless every entry passes
int check_live_entries(sgpu_ctx* ctx, const Slot& sl) {
    uint32_t* const mirror = ctx->live_mirror.get();
    uint8_t* const form = ctx->live_form.get();
    const uint32_t nc = ctx->live.n_channels;
    if (ctx->live_mirror_stale) {  // a device-resident live run changed channels: their state is read back once
        CU(cudaDeviceSynchronize());
        CU(cudaMemcpy(mirror, ctx->live.nopen, (size_t)nc * sizeof(uint32_t), cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(form, ctx->live.form, (size_t)nc * sizeof(uint8_t), cudaMemcpyDeviceToHost));
        ctx->live_mirror_stale = false;
    }
    const uint8_t my_form = live_form_of(sl.kind);
    for (uint32_t e = 0; e < sl.batch.n_reads; e++) {
        const uint32_t c = sl.h_channel[e], f = sl.h_flags[e], no = mirror[c], len = sl.batch.read_len[e];
        const bool start = (f & SGPU_LIVE_START) != 0;
        if (!start && !(no & LIVE_OPEN) && (len || (f & SGPU_LIVE_END))) return SGPU_E_STATE;
        if (!start && (no & LIVE_OPEN) && form[c] != my_form) return SGPU_E_STATE;  // a read of the other form
        if ((start ? 0ull : (uint64_t)(no & ~LIVE_OPEN)) + len > 0x7fffffffull) return SGPU_E_TOOBIG;
    }
    return SGPU_OK;
}

// the mirror of the channels as the kernels of a submitted live slot leave them
void advance_live_mirror(sgpu_ctx* ctx, const Slot& sl) {
    uint32_t* const mirror = ctx->live_mirror.get();
    for (uint32_t e = 0; e < sl.batch.n_reads; e++) {
        const uint32_t c = sl.h_channel[e], f = sl.h_flags[e], no = mirror[c], len = sl.batch.read_len[e];
        const bool start = (f & SGPU_LIVE_START) != 0;
        if (!start && !(no & LIVE_OPEN)) continue;
        mirror[c] = (f & SGPU_LIVE_END) ? 0u : (uint32_t)((start ? 0u : (no & ~LIVE_OPEN)) + len) | LIVE_OPEN;
        if (start) ctx->live_form[c] = live_form_of(sl.kind);
    }
}

// A detector set whose two detectors may emit more often than the reference's DNA set (8 events per 15 steps) needs
// the live staging of any set (live_stage_base, dense): a detector emits at most once per w/2 + 2 steps.
bool live_set_is_dense(const DetParams* set) {
    if (!set) return false;
    const int g1 = set->w1 / 2 + 2, g2 = set->w2 / 2 + 2;
    return 15 * (g1 + g2) > 8 * g1 * g2;
}

// The first live run under such a set grows the staging to the bound of any set for the rest of the context's life
// (waiting for the device first: queued runs still use the old arrays); the event outputs follow (fit_live_outputs).
int fit_live_staging(sgpu_ctx* ctx, const DetParams* set) {
    LiveScratch& w = ctx->live;
    if (w.dense || !live_set_is_dense(set)) return SGPU_OK;
    const uint64_t cap = live_stage_base(ctx->max_samples, ctx->max_reads, true);
    CU(cudaDeviceSynchronize());
    DevBuf<uint32_t> st, ln;
    DevBuf<float> mn, sd;
    CU(st.ensure(cap));
    CU(ln.ensure(cap));
    CU(mn.ensure(cap));
    CU(sd.ensure(cap));
    w.s_start = std::move(st); w.s_len = std::move(ln); w.s_mean = std::move(mn); w.s_stdv = std::move(sd);
    w.ev_cap = cap;
    w.dense = true;
    return SGPU_OK;
}

// (re)allocates the live outputs `o` at the context's live event capacity when they were made for another one
template <bool PINNED>
cudaError_t fit_live_outputs(const sgpu_ctx* ctx, Buf<void, PINNED> (&o)[N_LIVE_OUT], uint64_t& cap) {
    if (cap == ctx->live.ev_cap) return cudaSuccess;
    for (auto& buf : o) buf = Buf<void, PINNED>();
    const cudaError_t e = alloc_outputs(LIVE_OUTS, ctx, ctx->live.ev_cap, o, 0);
    if (e == cudaSuccess) cap = ctx->live.ev_cap;
    return e;
}

// sgpu_wait / sgpu_wait_live: the device status of the submitted slot, then its outputs `outs` (device d, pinned h)
// sized by the batch's events (at most ev_cap of them) copied back, and *out pointed at the pinned copies
template <size_t N, typename R>
int wait_slot(sgpu_ctx* ctx, Slot& sl, const OutSpec (&outs)[N], const DevBuf<void>* d, PinBuf<void>* h,
              uint64_t ev_cap, R* out) {
    CU(cudaSetDevice(ctx->device));
    sl.submitted = false;
    CU(cudaEventSynchronize(sl.small_back));
    memset(out, 0, sizeof *out);
    const int dev_rc = map_dev_status(*sl.h_status);
    if (dev_rc) return dev_rc;
    const uint32_t nr = sl.batch.n_reads;
    if (sl.want & SGPU_WANT_EVENTS) {
        const uint64_t ne = nr ? static_cast<const uint64_t*>(h[0].get())[nr] : 0;  // (row 0: ev_off)
        if (ne > ev_cap) return SGPU_E_EVCAP;
        CU(queue_d2h(outs, d, h, sl, SGPU_WANT_EVENTS, true, ne));
        CU(cudaStreamSynchronize(sl.stream));
        out->n_events = ne;
    }
    fill_result(outs, out, h, sl.want, false);
    return SGPU_OK;
}

}  // namespace

extern "C" {

int sgpu_abi_version(void) { return SGPU_ABI_VERSION; }

int sgpu_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

const char* sgpu_strerror(int code) {
    switch (code) {
        case SGPU_OK: return "success";
        case SGPU_E_INVAL: return "invalid argument";
        case SGPU_E_CUDA: return "CUDA error (no usable B200 / kernel failure); there is no CPU fallback";
        case SGPU_E_NOMEM: return "out of memory";
        case SGPU_E_FULL: return "slot full";
        case SGPU_E_TOOBIG: return "read larger than the context's max_samples";
        case SGPU_E_STATE: return "call out of order";
        case SGPU_E_EVCAP: return "event capacity exceeded";
        case SGPU_E_SCRATCH: return "sequential-order scratch too small";
        case SGPU_E_STREAM: return "malformed svb-zd stream (length does not match its keys)";
        default: return "unknown error";
    }
}

const char* sgpu_last_error(const sgpu_ctx_t* ctx) { return ctx ? ctx->err : "no context"; }

int sgpu_create(sgpu_ctx_t** out, int device, uint64_t max_samples, uint32_t max_reads, uint32_t n_slots,
                uint32_t flags) {
    if (!out || max_samples == 0 || max_reads == 0 || (flags & ~15u)) return SGPU_E_INVAL;
    *out = nullptr;
    if (flags & SGPU_F_NO_HOST_SLOTS) n_slots = 0; else if (n_slots == 0) n_slots = 2;
    sgpu_ctx* ctx = new (std::nothrow) sgpu_ctx();
    if (!ctx) return SGPU_E_NOMEM;
    auto fail = [&](int code) { sgpu_destroy(ctx); return code; };
    {
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || device < 0 || device >= ndev) {
            fprintf(stderr, "[sigtk_b200] no usable CUDA device %d (%s); this library has no CPU fallback\n", device,
                    e == cudaSuccess ? "index out of range" : cudaGetErrorString(e));
            delete ctx;
            return SGPU_E_CUDA;
        }
    }
#define CUC(call)                                                               \
    do {                                                                        \
        if (cuda_fail(ctx, (call), #call, __LINE__)) {                          \
            fprintf(stderr, "[sigtk_b200] %s\n", ctx->err);                     \
            return fail(SGPU_E_CUDA);                                           \
        }                                                                       \
    } while (0)
    CUC(cudaSetDevice(device));
    ctx->device = device;
    cudaDeviceProp prop;
    CUC(cudaGetDeviceProperties(&prop, device));
    ctx->sm_count = prop.multiProcessorCount;
    max_samples = align_up(max_samples, 64);
    ctx->max_samples = max_samples;
    ctx->max_reads = max_reads;
    ctx->n_slots = n_slots;
    ctx->flags = flags;
    // consecutive peaks are >= 3 samples apart (DNA; 5 for RNA) => <= n/3 + 2 events per read
    ctx->ev_cap = max_samples / 3 + 2ull * max_reads + 16;
    Scratch& sc = ctx->sc;
    // scratch of the sequential-order kernels (24 B/sample): everything for small contexts or when forced,
    // one eighth of the batch otherwise (reads that fail the fast path's checks are rare)
    // (SGPU_F_FULL_SEQ_SCRATCH: a context opened for one huge read must be able to redo that read in order)
    sc.gen_cap = (max_samples <= (64ull << 20) || (flags & (SGPU_F_FORCE_GENERIC | SGPU_F_FULL_SEQ_SCRATCH)))
                     ? max_samples : max_samples / 8;
    CUC(sc.Sinc.ensure(sc.gen_cap));
    CUC(sc.Qinc.ensure(sc.gen_cap));
    CUC(sc.t1.ensure(sc.gen_cap));
    CUC(sc.t2.ensure(sc.gen_cap));
    sc.max_tiles = fast_tiles_for(max_samples) + 1;
    sc.bitmap_words = (uint64_t)sc.max_tiles * (FAST_TILE / 32);
    CUC(sc.bitmap.ensure(sc.bitmap_words));
    sc.wk_slots = walk_state_slots(max_samples, max_reads);
    CUC(sc.wk_begin.ensure(sc.wk_slots * 8));
    CUC(sc.wk_end.ensure(sc.wk_slots * 8));
    CUC(sc.wk_cnt.ensure(max_reads));
    CUC(sc.wk_ibase.ensure((uint64_t)max_reads + 1));
    sc.job_cap = walk_job_capacity(max_samples);
    CUC(sc.jobs.ensure((uint64_t)sc.job_cap * 4));
    CUC(sc.job_count.ensure(1));
    sc.tune_chunk_len = 0; sc.tune_warmup = 0; sc.tune_thr_long = 9.0f;  // events.c:46,53: threshold of the long detector
    sc.tune_stat_cta_min = STAT_CTA_MIN_DEFAULT;
    CUC(sc.tile_cnt.ensure(sc.max_tiles));
    CUC(sc.tile_read0.ensure(sc.max_tiles));
    CUC(sc.tile_base.ensure((uint64_t)sc.max_tiles + 1));
    CUC(sc.wit_min.ensure(max_reads));
    CUC(sc.wit_max.ensure(max_reads));
    CUC(sc.seq_list.ensure(max_reads));
    CUC(sc.seq_sbase.ensure((uint64_t)max_reads + 1));
    CUC(sc.seq_count.ensure(1));
    CUC(sc.cursor.ensure(1));
    {
        uint64_t most = sc.max_tiles > max_reads ? sc.max_tiles : max_reads;
        const uint64_t svb_blocks = svbzd_max_blocks(max_samples, max_reads);
        if (svb_blocks > most) most = svb_blocks;
        CUC(sc.scan_status.ensure(scan_tiles_for((uint32_t)most) + 1));
    }
    ctx->comp_cap = 2 * max_samples;
    if (flags & SGPU_F_STAGE_TIMERS)
        for (int k = 0; k <= sgpu_ctx::MAX_STAGES; k++) CUC(cudaEventCreate(&ctx->stage_ev[k]));
    CUC(sc.scan_ticket.ensure(1));
    CUC(sc.status.ensure(1));
    CUC(sc.counters.ensure(4));
    CUC(cudaStreamCreateWithFlags(&ctx->compute, cudaStreamNonBlocking));
    CUC(alloc_outputs(OUTS, ctx, ctx->ev_cap, ctx->dev_out, 0));
    if (n_slots) {
        ctx->slots.reset(new (std::nothrow) Slot[n_slots]);
        if (!ctx->slots) return fail(SGPU_E_NOMEM);
        for (uint32_t s = 0; s < n_slots; s++) {
            Slot& sl = ctx->slots[s];
            CUC(sl.samples.ensure(max_samples));
            CUC(sl.read_off.ensure((uint64_t)max_reads + 1));
            CUC(sl.read_len.ensure(max_reads));
            CUC(sl.offset_f.ensure(max_reads));
            CUC(sl.raw_unit_f.ensure(max_reads));
            CUC(sl.d_samples.ensure(max_samples));
            CUC(sl.d_read_off.ensure((uint64_t)max_reads + 1));
            CUC(sl.d_read_len.ensure(max_reads));
            CUC(sl.d_offset.ensure(max_reads));
            CUC(sl.d_unit.ensure(max_reads));
            // every slot gets its own outputs (its D2H overlaps the next slot's kernels)
            CUC(alloc_outputs(OUTS, ctx, ctx->ev_cap, sl.dout, 0));
            CUC(alloc_outputs(OUTS, ctx, ctx->ev_cap, sl.hout, 0));
            CUC(sl.h_counters.ensure(4));
            CUC(sl.h_status.ensure(1));
            CUC(cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking));
            CUC(cudaEventCreateWithFlags(&sl.in_ready, cudaEventDisableTiming));
            CUC(cudaEventCreateWithFlags(&sl.kernels_done, cudaEventDisableTiming));
            CUC(cudaEventCreateWithFlags(&sl.small_back, cudaEventDisableTiming));
            sl.batch = sgpu_batch_t{sl.samples, sl.read_off, sl.read_len, sl.offset_f, sl.raw_unit_f, 0, 0};
            sl.batch.read_off[0] = 0;
        }
    }
#undef CUC
    *out = ctx;
    return SGPU_OK;
}

void sgpu_destroy(sgpu_ctx_t* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);  // its members free its arrays, streams and events on this device (one thread may
                                 // drive several GPUs)
    cudaDeviceSynchronize();
    delete ctx;
}

int sgpu_slot_batch(sgpu_ctx_t* ctx, uint32_t slot, sgpu_batch_t** out) {
    if (!ctx || !out || slot >= ctx->n_slots) return SGPU_E_INVAL;
    *out = &ctx->slots[slot].batch;
    return SGPU_OK;
}

int sgpu_slot_reset(sgpu_ctx_t* ctx, uint32_t slot, uint32_t rna) {
    if (!ctx || slot >= ctx->n_slots) return SGPU_E_INVAL;
    Slot& sl = ctx->slots[slot];
    if (sl.submitted) return SGPU_E_STATE;
    sl.batch.n_reads = 0;
    sl.batch.rna = rna ? 1u : 0u;
    sl.batch.read_off[0] = 0;
    sl.used = 0;
    sl.kind = Input::NONE;
    sl.comp_used = 0;
    sl.svb_blocks = 0;
    return SGPU_OK;
}

int64_t sgpu_slot_add_read(sgpu_ctx_t* ctx, uint32_t slot, const int16_t* raw, uint64_t n, double digitisation,
                           double offset, double range) {
    if (!ctx || slot >= ctx->n_slots || (!raw && n)) return SGPU_E_INVAL;
    Slot& sl = ctx->slots[slot];
    if (!accepts(sl, Input::RAW)) return SGPU_E_STATE;
    // (2^31 samples: the reference itself narrows to int32_t, misc.c:20)
    if (const int rc = room_for(ctx, sl, n, 1ull << 31, ctx->max_samples)) return rc;
    sl.kind = Input::RAW;
    memcpy(sl.batch.samples + sl.used, raw, (size_t)n * sizeof(int16_t));
    return append_record(sl, n, digitisation, offset, range);
}

int64_t sgpu_slot_add_read_svbzd(sgpu_ctx_t* ctx, uint32_t slot, const uint8_t* stream, uint64_t n_bytes,
                                 double digitisation, double offset, double range) {
    if (!ctx || slot >= ctx->n_slots || !stream) return SGPU_E_INVAL;
    Slot& sl = ctx->slots[slot];
    if (!accepts(sl, Input::SVBZD)) return SGPU_E_STATE;
    if (n_bytes != 0 && n_bytes < 4) return SGPU_E_STREAM;
    uint32_t count = 0;
    if (n_bytes) memcpy(&count, stream, 4);  // slow5_press.c:1093: the original length leads the stream
    const uint64_t n = count;                // (a record without signal stores no stream at all: n_bytes == 0)
    if (n_bytes && (4u + (n + 3u) / 4u + n > n_bytes || n_bytes > 4u + (n + 3u) / 4u + 4u * n)) return SGPU_E_STREAM;
    const uint64_t cneed = align_up(n_bytes, 16);
    if (n_bytes > 0xffffffffull || cneed > ctx->comp_cap) return SGPU_E_TOOBIG;  // (before the samples' SGPU_E_FULL)
    if (const int rc = room_for(ctx, sl, n, 1ull << 31, ctx->max_samples)) return rc;
    if (sl.comp_used + cneed > ctx->comp_cap) return SGPU_E_FULL;
    if (sl.kind != Input::SVBZD) {  // the batch's first stream: make sure the slot's svb-zd buffers exist
        CU(cudaSetDevice(ctx->device));
        const int rc = alloc_svb_scratch(ctx);
        if (rc) return rc;
        CU(sl.h_comp.ensure(ctx->comp_cap));
        CU(sl.d_comp.ensure(ctx->comp_cap + 16));
        CU(sl.h_comp_off.ensure(ctx->max_reads));
        CU(sl.d_comp_off.ensure(ctx->max_reads));
        CU(sl.h_comp_len.ensure(ctx->max_reads));
        CU(sl.d_comp_len.ensure(ctx->max_reads));
    }
    sl.kind = Input::SVBZD;
    const uint32_t r = sl.batch.n_reads;
    if (n_bytes) memcpy(sl.h_comp + sl.comp_used, stream, (size_t)n_bytes);
    sl.h_comp_off[r] = sl.comp_used;
    sl.h_comp_len[r] = (uint32_t)n_bytes;
    sl.comp_used += cneed;
    sl.svb_blocks += svbzd_blocks_of(n);
    return append_record(sl, n, digitisation, offset, range);
}

int64_t sgpu_slot_add_read_pa(sgpu_ctx_t* ctx, uint32_t slot, const float* pa, uint64_t n) {
    if (!ctx || slot >= ctx->n_slots || (!pa && n)) return SGPU_E_INVAL;
    Slot& sl = ctx->slots[slot];
    if (!accepts(sl, Input::PA)) return SGPU_E_STATE;
    // the slot's int16 sample buffers (pinned and device) hold the floats: max_samples / 2 of them
    if (const int rc = room_for(ctx, sl, n, 1ull << 32, ctx->max_samples / 2)) return rc;
    sl.kind = Input::PA;
    memcpy(reinterpret_cast<float*>(sl.batch.samples) + sl.used, pa, (size_t)n * sizeof(float));
    return append_record(sl, n, 1.0, 0.0, 1.0);  // (offset_f 0, raw_unit_f 1: the values are pA already)
}

int sgpu_submit(sgpu_ctx_t* ctx, uint32_t slot, uint32_t want) {
    if (!ctx || slot >= ctx->n_slots || (want & ~63u) || want == 0) return SGPU_E_INVAL;
    Slot& sl = ctx->slots[slot];
    if (sl.submitted) return SGPU_E_STATE;
    if (want & ~allowed_wants(sl.kind)) return SGPU_E_INVAL;
    CU(cudaSetDevice(ctx->device));
    const bool live = is_live(sl.kind);
    int rc = live ? check_live_entries(ctx, sl) : SGPU_OK;
    if (rc) return rc;
    sl.det_set = ctx->det;  // the slot runs the set in force now, whatever is set before it is waited for
    sl.det = ctx->det_on ? &sl.det_set : nullptr;
    if (live) {
        if ((rc = fit_live_staging(ctx, sl.det))) return rc;
        CU(fit_live_outputs(ctx, sl.live_dout, sl.live_dcap));
        CU(fit_live_outputs(ctx, sl.live_hout, sl.live_hcap));
    }
    const sgpu_batch_t& hb = sl.batch;
    const uint32_t nr = hb.n_reads;
    cudaStream_t st = sl.stream;
    if (sl.kind == Input::SVBZD) {
        CU(cudaMemcpyAsync(sl.d_comp, sl.h_comp, (size_t)sl.comp_used, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(sl.d_comp_off, sl.h_comp_off, (size_t)nr * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(sl.d_comp_len, sl.h_comp_len, (size_t)nr * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    } else {
        const size_t sample_size = sl.kind == Input::PA || sl.kind == Input::LIVE_PA ? sizeof(float) : sizeof(int16_t);
        CU(cudaMemcpyAsync(sl.d_samples, hb.samples, (size_t)sl.used * sample_size, cudaMemcpyHostToDevice, st));
    }
    CU(cudaMemcpyAsync(sl.d_read_off, hb.read_off, ((size_t)nr + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(sl.d_read_len, hb.read_len, (size_t)nr * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(sl.d_offset, hb.offset_f, (size_t)nr * sizeof(float), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(sl.d_unit, hb.raw_unit_f, (size_t)nr * sizeof(float), cudaMemcpyHostToDevice, st));
    if (live) {
        CU(cudaMemcpyAsync(sl.d_channel, sl.h_channel, (size_t)nr * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(sl.d_flags, sl.h_flags, (size_t)nr * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    }
    CU(cudaEventRecord(sl.in_ready, st));
    CU(cudaStreamWaitEvent(ctx->compute, sl.in_ready, 0));
    rc = run_slot(ctx, sl, want);
    if (rc) return rc;
    // small results come back right away; the big arrays are sized by n_events in sgpu_wait / sgpu_wait_live
    CU(cudaMemcpyAsync(sl.h_counters, ctx->sc.counters, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                       ctx->compute));
    CU(cudaMemcpyAsync(sl.h_status, ctx->sc.status, sizeof(int), cudaMemcpyDeviceToHost, ctx->compute));
    CU(cudaEventRecord(sl.kernels_done, ctx->compute));
    CU(cudaStreamWaitEvent(st, sl.kernels_done, 0));
    CU(live ? queue_d2h(LIVE_OUTS, sl.live_dout, sl.live_hout, sl, want, false, 0)
            : queue_d2h(OUTS, sl.dout, sl.hout, sl, want, false, 0));
    CU(cudaEventRecord(sl.small_back, st));
    if (live) advance_live_mirror(ctx, sl);
    sl.want = want;
    sl.submitted = true;
    return SGPU_OK;
}

int sgpu_wait(sgpu_ctx_t* ctx, uint32_t slot, sgpu_result_t* out) {
    if (!ctx || slot >= ctx->n_slots || !out) return SGPU_E_INVAL;
    Slot& sl = ctx->slots[slot];
    if (!sl.submitted || is_live(sl.kind)) return SGPU_E_STATE;
    return wait_slot(ctx, sl, OUTS, sl.dout, sl.hout, ctx->ev_cap, out);
}

int sgpu_run_device(sgpu_ctx_t* ctx, const sgpu_dev_batch_t* batch, uint32_t want, void* stream,
                    sgpu_result_t* out) {
    if (!ctx || !batch || !out || (want & ~63u) || want == 0) return SGPU_E_INVAL;
    CU(cudaSetDevice(ctx->device));
    DevBatch b{batch->samples, batch->read_off, batch->read_len, batch->offset_f, batch->raw_unit_f,
               batch->n_reads, (int)batch->rna, batch->span};
    const int rc = run_pipeline(ctx, b, want, ctx->dev_out, reinterpret_cast<cudaStream_t>(stream),
                                ctx->det_on ? &ctx->det : nullptr);
    if (rc) return rc;
    memset(out, 0, sizeof *out);
    fill_result(OUTS, out, ctx->dev_out, want, true);
    return SGPU_OK;
}

int sgpu_run_device_pa(sgpu_ctx_t* ctx, const sgpu_dev_pa_batch_t* batch, uint32_t want, void* stream,
                       sgpu_result_t* out) {
    if (!ctx || !batch || !out || !pa_input_want_ok(want)) return SGPU_E_INVAL;
    CU(cudaSetDevice(ctx->device));
    const DevBatch b{nullptr, batch->read_off, batch->read_len, nullptr, nullptr, batch->n_reads, (int)batch->rna,
                     batch->span};
    const int rc = run_pipeline_pa(ctx, b, batch->pa, ctx->det_on ? &ctx->det : nullptr, want, ctx->dev_out,
                                   reinterpret_cast<cudaStream_t>(stream));
    if (rc) return rc;
    memset(out, 0, sizeof *out);
    fill_result(OUTS, out, ctx->dev_out, want, false);
    return SGPU_OK;
}

int sgpu_decode_svbzd_device(sgpu_ctx_t* ctx, const sgpu_svb_dev_batch_t* batch, int16_t* samples_out, void* stream) {
    if (!ctx || !batch || !samples_out) return SGPU_E_INVAL;
    if (batch->n_reads > ctx->max_reads || batch->n_blocks > svbzd_max_blocks(ctx->max_samples, ctx->max_reads))
        return SGPU_E_INVAL;
    CU(cudaSetDevice(ctx->device));
    const int arc = alloc_svb_scratch(ctx);
    if (arc) return arc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    CU(cudaMemsetAsync(ctx->sc.status, 0, sizeof(int), st));
    SvbBatch s{batch->bytes, batch->n_bytes, batch->comp_off, batch->comp_len, batch->read_off, batch->read_len,
               batch->n_reads, batch->n_blocks};
    ctx->last_launches = (uint64_t)launch_svbzd_decode(s, ctx->svb, ctx->sc, samples_out, ctx->sm_count, st);
    CU(cudaGetLastError());
    return SGPU_OK;
}

int sgpu_counters(sgpu_ctx_t* ctx, sgpu_counters_t* out) {
    if (!ctx || !out) return SGPU_E_INVAL;
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    unsigned long long c[4];
    int status = 0;
    CU(cudaMemcpy(c, ctx->sc.counters, sizeof c, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(&status, ctx->sc.status, sizeof status, cudaMemcpyDeviceToHost));
    out->n_events = c[0];
    out->n_seq_order_reads = c[1];
    out->n_fixups = c[2];
    out->n_kernel_launches = ctx->last_launches;
    out->status = map_dev_status(status);
    out->n_long_jobs = c[3];
    return SGPU_OK;
}

int sgpu_set_param(sgpu_ctx_t* ctx, int key, double value) {
    if (!ctx) return SGPU_E_INVAL;
    Scratch& sc = ctx->sc;
    switch (key) {
        case SGPU_PARAM_CHUNK_LEN:
            if (value < 0 || value > (double)(1u << 20)) return SGPU_E_INVAL;
            sc.tune_chunk_len = (uint32_t)value;
            return SGPU_OK;
        case SGPU_PARAM_WARMUP:
            if (value < 0 || value > 4096) return SGPU_E_INVAL;
            sc.tune_warmup = (uint32_t)value;
            return SGPU_OK;
        case SGPU_PARAM_PORE:
            if (value != 0 && value != 1) return SGPU_E_INVAL;
            ctx->pore_rna004 = (int)value;
            return SGPU_OK;
        case SGPU_PARAM_STAT_CTA_MIN:
            if (value < 0 || value > 4294967295.0) return SGPU_E_INVAL;
            sc.tune_stat_cta_min = (uint32_t)value;
            return SGPU_OK;
        case SGPU_PARAM_THR_LONG:
            if (!(value > 0 && value < 1e6)) return SGPU_E_INVAL;
            sc.tune_thr_long = (float)value;
            return SGPU_OK;
        default: return SGPU_E_INVAL;
    }
}

int sgpu_set_detector(sgpu_ctx_t* ctx, const sgpu_detector_t* p) {
    if (!ctx) return SGPU_E_INVAL;
    if (!p) { ctx->det_on = false; return SGPU_OK; }
    const bool windows = p->w_short >= 2 && p->w_short <= 14 && p->w_long >= 2 && p->w_long <= 14;
    if (!windows || !std::isfinite(p->thr_short) || !std::isfinite(p->thr_long) || !std::isfinite(p->peak_height))
        return SGPU_E_INVAL;
    ctx->det = DetParams{(int)p->w_short, (int)p->w_long, p->thr_short, p->thr_long, p->peak_height};
    ctx->det_on = true;
    return SGPU_OK;
}

int sgpu_stage_times(sgpu_ctx_t* ctx, sgpu_stage_time_t* out, uint32_t cap) {
    if (!ctx || (!out && cap)) return SGPU_E_INVAL;
    if (!(ctx->flags & SGPU_F_STAGE_TIMERS)) return SGPU_E_STATE;
    CU(cudaSetDevice(ctx->device));
    if (ctx->n_stages == 0) return 0;
    CU(cudaEventSynchronize(ctx->stage_ev[ctx->n_stages]));
    int n = 0;
    for (int k = 0; k < ctx->n_stages && (uint32_t)k < cap; k++, n++) {
        float ms = 0.0f;
        CU(cudaEventElapsedTime(&ms, ctx->stage_ev[k], ctx->stage_ev[k + 1]));
        out[k].name = ctx->stage_name[k];
        out[k].ms = ms;
        out[k].launches = ctx->stage_launches[k];
    }
    return n;
}

int sgpu_memcpy_d2h(sgpu_ctx_t* ctx, void* dst, const void* src, uint64_t bytes) {
    if (!ctx || (!dst && bytes) || (!src && bytes)) return SGPU_E_INVAL;
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    if (bytes) CU(cudaMemcpy(dst, src, (size_t)bytes, cudaMemcpyDeviceToHost));
    return SGPU_OK;
}

int sgpu_live_open(sgpu_ctx_t* ctx, uint32_t n_channels) {
    if (!ctx || n_channels == 0) return SGPU_E_INVAL;
    LiveScratch& w = ctx->live;
    if (w.n_channels) return SGPU_E_STATE;
    CU(cudaSetDevice(ctx->device));
    w.ev_cap = live_stage_base(ctx->max_samples, ctx->max_reads, w.dense);
    CU(w.chan.ensure(n_channels));
    CU(w.nopen.ensure(n_channels));
    CU(w.claim.ensure(n_channels));
    CU(w.form.ensure(n_channels));
    CU(w.cnt.ensure(ctx->max_reads));
    CU(w.s_start.ensure(w.ev_cap));
    CU(w.s_len.ensure(w.ev_cap));
    CU(w.s_mean.ensure(w.ev_cap));
    CU(w.s_stdv.ensure(w.ev_cap));
    CU(cudaMemset(w.nopen, 0, (size_t)n_channels * sizeof(uint32_t)));
    CU(cudaMemset(w.claim, 0, (size_t)n_channels * sizeof(uint32_t)));
    CU(cudaMemset(w.form, LIVE_FORM_INT16, (size_t)n_channels * sizeof(uint8_t)));
    ctx->live_mirror.reset(new (std::nothrow) uint32_t[n_channels]());
    ctx->live_form.reset(new (std::nothrow) uint8_t[n_channels]());
    if (!ctx->live_mirror || !ctx->live_form) return SGPU_E_NOMEM;
    for (uint32_t s = 0; s < ctx->n_slots; s++) {
        Slot& sl = ctx->slots[s];
        CU(sl.h_channel.ensure(ctx->max_reads));
        CU(sl.h_flags.ensure(ctx->max_reads));
        CU(sl.d_channel.ensure(ctx->max_reads));
        CU(sl.d_flags.ensure(ctx->max_reads));
        CU(fit_live_outputs(ctx, sl.live_dout, sl.live_dcap));
        CU(fit_live_outputs(ctx, sl.live_hout, sl.live_hcap));
        sl.live_claim.reset(new (std::nothrow) uint32_t[n_channels]());
        if (!sl.live_claim) return SGPU_E_NOMEM;
    }
    w.n_channels = n_channels;  // (last: an open that failed can be repeated, the arrays it made are kept)
    return SGPU_OK;
}

int64_t sgpu_slot_add_live(sgpu_ctx_t* ctx, uint32_t slot, uint32_t channel, uint32_t flags, const int16_t* raw,
                           uint64_t n, double digitisation, double offset, double range) {
    if (!ctx || slot >= ctx->n_slots || (!raw && n)) return SGPU_E_INVAL;
    Slot& sl = ctx->slots[slot];
    if (const int rc = add_live_entry(ctx, sl, Input::LIVE, channel, flags, n, ctx->max_samples)) return rc;
    memcpy(sl.batch.samples + sl.used, raw, (size_t)n * sizeof(int16_t));
    return append_record(sl, n, digitisation, offset, range);
}

int64_t sgpu_slot_add_live_pa(sgpu_ctx_t* ctx, uint32_t slot, uint32_t channel, uint32_t flags, const float* pa,
                              uint64_t n) {
    if (!ctx || slot >= ctx->n_slots || (!pa && n)) return SGPU_E_INVAL;
    Slot& sl = ctx->slots[slot];
    // the slot's int16 sample buffers (pinned and device) hold the floats: max_samples / 2 of them
    if (const int rc = add_live_entry(ctx, sl, Input::LIVE_PA, channel, flags, n, ctx->max_samples / 2)) return rc;
    memcpy(reinterpret_cast<float*>(sl.batch.samples) + sl.used, pa, (size_t)n * sizeof(float));
    return append_record(sl, n, 1.0, 0.0, 1.0);  // (offset_f 0, raw_unit_f 1: the values are pA already)
}

int sgpu_wait_live(sgpu_ctx_t* ctx, uint32_t slot, sgpu_live_result_t* out) {
    if (!ctx || slot >= ctx->n_slots || !out) return SGPU_E_INVAL;
    Slot& sl = ctx->slots[slot];
    if (!sl.submitted || !is_live(sl.kind)) return SGPU_E_STATE;
    return wait_slot(ctx, sl, LIVE_OUTS, sl.live_dout, sl.live_hout, ctx->live.ev_cap, out);
}

int sgpu_run_device_live(sgpu_ctx_t* ctx, const sgpu_dev_live_batch_t* batch, void* stream, sgpu_live_result_t* out) {
    if (!ctx || !batch || !out) return SGPU_E_INVAL;
    if (!ctx->live.n_channels) return SGPU_E_STATE;
    CU(cudaSetDevice(ctx->device));
    const DetParams* const set = ctx->det_on ? &ctx->det : nullptr;
    if (const int rc = fit_live_staging(ctx, set)) return rc;
    CU(fit_live_outputs(ctx, ctx->live_dev_out, ctx->live_dev_cap));
    const LiveBatch b{batch->samples, batch->read_off, batch->read_len, batch->channel, batch->flags, batch->offset_f,
                      batch->raw_unit_f, batch->n_entries, batch->span};
    const int rc = run_pipeline_live(ctx, b, false, set, ctx->live_dev_out, reinterpret_cast<cudaStream_t>(stream));
    if (rc) return rc;
    ctx->live_mirror_stale = true;
    memset(out, 0, sizeof *out);
    fill_result(LIVE_OUTS, out, ctx->live_dev_out, SGPU_WANT_EVENTS, false);
    return SGPU_OK;
}

int sgpu_run_device_live_pa(sgpu_ctx_t* ctx, const sgpu_dev_live_pa_batch_t* batch, void* stream,
                            sgpu_live_result_t* out) {
    if (!ctx || !batch || !out) return SGPU_E_INVAL;
    if (!ctx->live.n_channels) return SGPU_E_STATE;
    CU(cudaSetDevice(ctx->device));
    const DetParams* const set = ctx->det_on ? &ctx->det : nullptr;
    if (const int rc = fit_live_staging(ctx, set)) return rc;
    CU(fit_live_outputs(ctx, ctx->live_dev_out, ctx->live_dev_cap));
    LiveBatch b{nullptr, batch->read_off, batch->read_len, batch->channel, batch->flags, nullptr, nullptr,
                batch->n_entries, batch->span};
    b.pa = batch->pa;
    const int rc = run_pipeline_live(ctx, b, true, set, ctx->live_dev_out, reinterpret_cast<cudaStream_t>(stream));
    if (rc) return rc;
    ctx->live_mirror_stale = true;
    memset(out, 0, sizeof *out);
    fill_result(LIVE_OUTS, out, ctx->live_dev_out, SGPU_WANT_EVENTS, false);
    return SGPU_OK;
}

}  // extern "C"
