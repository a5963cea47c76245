// kernels.cuh -- internal interfaces between the kernel translation units and capi.cu
#pragma once
#include <type_traits>

#include "common.cuh"

namespace sgpu {

// An owning pointer to an array in device memory (or, PINNED, in pinned host memory; T = void: an array of bytes).
// Its destructor frees the array, so the code that sizes an array is the only place that lists it. It converts to
// T*, so launchers take its members as plain pointers. Host code only.
template <typename T, bool PINNED = false>
class Buf {
  public:
    Buf() = default;
    Buf(const Buf&) = delete;
    Buf& operator=(const Buf&) = delete;
    Buf(Buf&& o) noexcept : p_(o.p_) { o.p_ = nullptr; }
    Buf& operator=(Buf&& o) noexcept {
        if (this != &o) { release(); p_ = o.p_; o.p_ = nullptr; }
        return *this;
    }
    ~Buf() { release(); }  // (holding nothing, it makes no CUDA call)

    // Allocates max(count, 1) elements unless it holds some already, and keeps the pointer only on success: an
    // allocation that failed part-way through a list is completed by the next call instead of leaving a NULL
    // pointer behind a non-NULL one.
    cudaError_t ensure(uint64_t count) {
        if (p_) return cudaSuccess;
        size_t bytes = (size_t)(count ? count : 1);
        if constexpr (!std::is_void_v<T>) bytes *= sizeof(T);
        void* q = nullptr;
        const cudaError_t e = PINNED ? cudaHostAlloc(&q, bytes, cudaHostAllocDefault) : cudaMalloc(&q, bytes);
        if (e == cudaSuccess) p_ = static_cast<T*>(q);
        return e;
    }
    T* get() const { return p_; }
    operator T*() const { return p_; }

  private:
    void release() {
        if (!p_) return;
        if (PINNED) cudaFreeHost(p_); else cudaFree(p_);
    }
    T* p_ = nullptr;
};
template <typename T> using DevBuf = Buf<T, false>;
template <typename T> using PinBuf = Buf<T, true>;

// device-side status codes (mapped to SGPU_E_* by capi.cu)
enum { SGPU_DEV_OK = 0, SGPU_DEV_E_EVCAP = 1, SGPU_DEV_E_SCRATCH = 2, SGPU_DEV_E_STREAM = 3, SGPU_DEV_E_INVAL = 4,
       SGPU_DEV_E_STATE = 5, SGPU_DEV_E_TOOBIG = 6 };

constexpr int FAST_TILE = 2048;  // samples per tile of the fast path; the event-start bitmap is tiled the same way

// A list of reads to be processed by the sequential-order kernels.
//   list  : read indices
//   sbase : base of each entry in the per-sample scratch arrays
//   count : device pointer to the list length
struct WorkList {
    const uint32_t* list;
    const uint64_t* sbase;
    const uint32_t* count;
};

// Device workspace owned by a context.
struct Scratch {
    // sequential-order scratch (gen_cap samples)
    DevBuf<double> Sinc, Qinc; DevBuf<float> t1, t2;
    uint64_t gen_cap;
    // event-start bitmap over the flat sample span: bit p set <=> an event starts at flat sample p
    DevBuf<uint32_t> bitmap; uint64_t bitmap_words;
    // per tile
    DevBuf<uint32_t> tile_cnt; DevBuf<uint64_t> tile_base;
    DevBuf<uint32_t> tile_read0;     // first read that can intersect a 2048-sample tile (emit_events_kernel); the
                                     // walker sets the top bit of tiles that hold LOW samples (pA <= 0 or barely above)
    // chunk walker (walk.cu)
    DevBuf<uint32_t> wk_cnt;         // [max_reads] interior chunks per read
    DevBuf<uint64_t> wk_ibase;       // [max_reads+1] exclusive scan of wk_cnt
    DevBuf<int> wk_begin, wk_end;    // [wk_slots*8] detector state after the warm-up / after the last step of a chunk
    uint64_t wk_slots;
    DevBuf<int> jobs;                // [job_cap * 4] lives of the long detector to replay: {read, chunk, l_start, end}
    DevBuf<uint32_t> job_count;      // device scalar
    uint32_t job_cap;
    // development / test parameters (sgpu_set_param): 0 = automatic
    uint32_t tune_chunk_len, tune_warmup;
    float tune_thr_long;             // the long detector's threshold (9.0)
    uint32_t tune_stat_cta_min;      // reads of at least this many samples get a CTA in the moments kernels (stat.cu)
    uint32_t max_tiles;
    // per read
    DevBuf<uint32_t> wit_min, wit_max;  // exact-sum witness: min nonzero |pA| / max |pA| bit patterns
    DevBuf<uint32_t> seq_list;  // compacted list of reads routed to the sequential-order kernels
    DevBuf<uint64_t> seq_sbase;
    DevBuf<uint32_t> seq_count; // device scalar
    DevBuf<unsigned long long> cursor;  // device scalar: used scratch samples
    // scan
    DevBuf<unsigned long long> scan_status; DevBuf<uint32_t> scan_ticket;
    // device-side status / counters
    DevBuf<int> status; DevBuf<unsigned long long> counters;  // [0]=n_events [1]=n_seq [2]=n_fixups
};

// generic.cu (sequential-order kernels)
constexpr int GD_CHUNK = 1024;  // positions per chunk of the warp-chunked detectors
__device__ void clear_read_bits(uint32_t* __restrict__ bitmap, uint64_t p0, uint64_t p1);
// the detector of one read in the reference's own order (one thread): events.c:371-443
__device__ void detect_read_in_order(const DetParams& p, const float* __restrict__ t1, const float* __restrict__ t2,
                                     uint64_t base, uint64_t foff, uint32_t n, uint32_t* __restrict__ bitmap);
int launch_generic_detect(const DevBatch& b, const WorkList& wl, Scratch& sc, int sm_count, cudaStream_t st);
int launch_generic_emit(const DevBatch& b, const WorkList& wl, Scratch& sc, const uint64_t* ev_off, uint64_t ev_cap,
                        uint32_t* ev_start, float* ev_mean, float* ev_stdv, int sm_count, cudaStream_t st);
// the general route's ordered prefix sums, t-statistics and detector (pa: the caller's floats, or nullptr: b's int16
// samples; set: the caller's detector set, or nullptr: the reference's chosen by b.rna)
int launch_generic_detect_pa(const DevBatch& b, const float* pa, const DetParams* set, const WorkList& ordered,
                             const WorkList& all, Scratch& sc, uint32_t* fixups, int sm_count, cudaStream_t st);
// detect_set.cu: the warp-chunked detector of the reads of wl on the t arrays with a caller's set; fixups[r] = the
// read's mismatched chunks
int launch_detect_set(const DevBatch& b, const WorkList& wl, Scratch& sc, uint32_t* fixups, const DetParams& set,
                      int sm_count, cudaStream_t st);
int launch_scan_u32(const uint32_t* cnt, uint32_t n, uint64_t* off, uint64_t* total_out, Scratch& sc, cudaStream_t st);
uint32_t scan_tiles_for(uint32_t n);

// fast.cu (witness evaluation, event ranks) and emit.cu (event table)
uint32_t fast_tiles_for(uint64_t span);
int launch_init_reads(const DevBatch& b, Scratch& sc, uint32_t* seq_flag, uint32_t* fixups, int sm_count,
                      cudaStream_t st);
// walk.cu (chunk walker: pA, t-statistics, peak detector -> event-start bitmap)
int launch_walk(const DevBatch& b, Scratch& sc, float* pa_out, uint32_t* seq_flag, int sm_count, cudaStream_t st);
int launch_long_jobs(const DevBatch& b, Scratch& sc, uint32_t* seq_flag, int sm_count, cudaStream_t st);
int launch_verify_chunks(const DevBatch& b, Scratch& sc, uint32_t* seq_flag, uint32_t* fixups, int sm_count, cudaStream_t st);
uint64_t walk_state_slots(uint64_t max_samples, uint32_t max_reads);
uint32_t walk_chunk_len(uint64_t span, uint32_t n_reads, int rna, int sm_count, uint32_t forced);
uint32_t walk_warmup(int rna, uint32_t forced);
uint32_t walk_job_capacity(uint64_t max_samples);
int launch_build_seq_list(const DevBatch& b, Scratch& sc, uint32_t* seq_flag, int force_all, int sm_count,
                          cudaStream_t st);
int launch_rank_events(const DevBatch& b, Scratch& sc, uint64_t* ev_off, int sm_count, cudaStream_t st);
int launch_fast_emit(const DevBatch& b, Scratch& sc, uint64_t ev_cap, uint32_t* ev_start, float* ev_mean,
                     float* ev_stdv, const uint32_t* fixups, int sm_count, cudaStream_t st);
int launch_pa(const DevBatch& b, float* pa, int sm_count, cudaStream_t st);

// pa_input.cu (the general route of event detection -- the caller's pA floats, or any batch with a caller's detector
// set: exactness witness and parallel scan of the prefix sums)
struct PaScratch {                 // allocated on the first pA batch
    DevBuf<uint32_t> tile_cnt;     // [max_reads] tiles of every read
    DevBuf<uint64_t> tile_base;    // [max_reads+1] their exclusive scan
    DevBuf<double> tS, tQ;         // [max_tiles] the tiles' sums, then their prefixes within the read
    DevBuf<double> tA, tB;         // [max_tiles] upper bounds of sum |x| and sum fl(x*x)
    DevBuf<uint2> tmin;            // [max_tiles] smallest nonzero |x| and fl(x*x) (float bits)
    DevBuf<uint32_t> ord_list;     // reads summed in the reference's order
    DevBuf<uint64_t> ord_sbase; DevBuf<uint32_t> ord_count;
    uint64_t max_tiles;
};
uint64_t pa_tile_capacity(uint64_t max_samples, uint32_t max_reads);
// pa: the caller's floats, or nullptr: b's int16 samples through their calibration
int launch_pa_prefix(const DevBatch& b, const float* pa, PaScratch& w, Scratch& sc, uint32_t* seq_flag,
                     uint32_t* fixups, int force_all, int sm_count, cudaStream_t st);

// svbzd.cu (svb-zd signal streams -> int16 samples in HBM)
struct SvbBatch {
    const uint8_t*  bytes;     // the streams of the batch back to back, each starting on a 16-byte boundary;
    uint64_t        n_bytes;   // the allocation extends at least 8 bytes past n_bytes
    const uint64_t* comp_off;  // [n_reads] byte offset of every stream
    const uint32_t* comp_len;  // [n_reads] stream length in bytes (header + keys + data)
    const uint64_t* read_off;  // [n_reads+1] where the samples go (multiples of 8)
    const uint32_t* read_len;  // [n_reads] = the count in every stream's header
    uint32_t n_reads;
    uint64_t n_blocks;         // sum of svbzd_blocks_of(read_len)
};
struct SvbScratch {
    DevBuf<uint32_t> cnt; DevBuf<uint64_t> base;            // [max_reads], [max_reads+1]
    DevBuf<uint32_t> blk_bytes; DevBuf<uint64_t> blk_gpos;  // [max_blocks], [max_blocks+1]
    DevBuf<uint32_t> blk_sum; DevBuf<uint64_t> blk_vpos;
    DevBuf<uint32_t> lane_sum;                // [max_blocks*32]
    DevBuf<uint32_t> blk_read;                // [max_blocks] read of every block
    uint64_t max_blocks;
};
uint64_t svbzd_max_blocks(uint64_t max_samples, uint32_t max_reads);
uint32_t svbzd_blocks_of(uint64_t n);
int launch_svbzd_decode(const SvbBatch& s, SvbScratch& w, Scratch& sc, int16_t* samples, int sm_count, cudaStream_t st);

// live.cu (event detection on signal that arrives in chunks: sgpu_slot_add_live, sgpu_run_device_live)
constexpr uint32_t LIVE_FLAGS = 7u;        // SGPU_LIVE_START | SGPU_LIVE_END | SGPU_LIVE_RNA
constexpr uint32_t LIVE_OPEN = 1u << 31;   // LiveScratch::nopen: samples so far | LIVE_OPEN while a read is open
constexpr int LIVE_TAIL = 28;              // prefix sums a channel carries: 2 * w2 of the RNA parameters
// LiveScratch::form: the form of the entry that started a channel's read (sgpu_slot_add_live or sgpu_slot_add_live_pa)
constexpr uint8_t LIVE_FORM_INT16 = 0, LIVE_FORM_PA = 1;
// What a channel carries from one entry to the next (in HBM; its length and open flag are in LiveScratch::nopen).
struct LiveChan {
    double tS[LIVE_TAIL], tQ[LIVE_TAIL];  // S[j], Q[j] for j = n-LIVE_TAIL+1 .. n (0 for j <= 0)
    double pS[2], pQ[2];                  // at the peak_pos of the short / long detector
    double aS, aQ;                        // at the open event's start
    DetState det[2];                      // short, long
    uint32_t a;                           // the open event's start
    float offset, unit;                   // the read's calibration (misc.c:17-19,26)
    uint32_t rna;
    uint32_t custom;                      // 1: the read runs the detector set in force at its START (`set`)
    DetParams set;
};
struct LiveBatch {                         // entry e: samples (or pa)[read_off[e] .. +read_len[e]) of channel[e]
    union {
        const int16_t* samples;            // int16 entries, with offset and unit
        const float* pa;                   // pA entries (launch_live's pa): offset and unit are not read
    };
    const uint64_t* read_off;              // [n_entries+1]
    const uint32_t* read_len;
    const uint32_t* channel;
    const uint32_t* flags;
    const float* offset;                   // used with SGPU_LIVE_START only
    const float* unit;
    uint32_t n_entries;
    uint64_t span;
};
// where entry e (at sample offset `off`) stages its events before compaction. The detector steps at most
// len + max(w1, w2) - 1 < len + 14 positions in an entry, and a detector that emits at step i emits next at step
// i + w/2 + 2 or later (its peak is set at i + 1 at the earliest and must be more than w/2 behind): at most
// ceil(m/3) + ceil(m/5) events in m steps (DNA; RNA fewer) plus the read's last one, which the stride of
// 8/15 per sample + 24 per entry covers. `dense` (LiveScratch::dense): any detector set (w >= 2: gaps of 3 or more
// for both detectors), ceil(m/3) + ceil(m/3) + 1, covered by 2/3 per sample + 24 per entry. Evaluated at
// (max_samples, max_reads) it is the capacity.
__host__ __device__ inline uint64_t live_stage_base(uint64_t off, uint64_t e, bool dense) {
    return (dense ? off / 3 * 2 : off / 15 * 8) + 24 * e;
}
struct LiveScratch {                       // allocated by sgpu_live_open
    DevBuf<LiveChan> chan;                 // [n_channels]
    DevBuf<uint32_t> nopen;                // [n_channels]
    DevBuf<uint32_t> claim;                // [n_channels] stamp of the last run that had an entry for the channel
    DevBuf<uint8_t> form;                  // [n_channels] LIVE_FORM_* of the open read (written at START)
    DevBuf<uint32_t> cnt;                  // [max_reads] events of every entry
    DevBuf<uint32_t> s_start, s_len;       // [ev_cap] staged events
    DevBuf<float> s_mean, s_stdv;
    uint32_t n_channels = 0;
    uint64_t ev_cap = 0;
    uint32_t stamp = 0;
    bool dense = false;                    // staged at the bound of any detector set (live_stage_base)
};
// the events of entry e go to ev_start, ev_len, ev_mean, ev_stdv [ev_off[e], ev_off[e+1]) (ev_off: [n_entries+1]);
// pa: the entries are b.pa floats; set: the detector set a START entry gives its read, or nullptr: the reference's
int launch_live(const LiveBatch& b, bool pa, const DetParams* set, LiveScratch& w, Scratch& sc, uint64_t* ev_off,
                uint32_t* ev_start, uint32_t* ev_len, float* ev_mean, float* ev_stdv, int sm_count, cudaStream_t st);

// stat.cu
constexpr uint32_t STAT_CTA_MIN_DEFAULT = 131072u;
int launch_stat_moments(const DevBatch& b, float* stat6, uint32_t cta_min, int sm_count, cudaStream_t st);
int launch_stat_median(const DevBatch& b, float* stat6, uint32_t cta_min, int sm_count, cudaStream_t st);
int launch_jnn_moments(const DevBatch& b, float* moments2, uint32_t cta_min, int sm_count, cudaStream_t st);

// jnn.cu (`sigtk jnn`: band from the clamped signal's mean / stdv, counter machine per read -> (start, end) pairs)
uint64_t jnn_seg_capacity(uint64_t max_samples, uint32_t max_reads);
int launch_jnn(const DevBatch& b, const float* moments, uint32_t* seg_cnt, int32_t* seg, int sm_count, cudaStream_t st);


// prefix.cu (`sigtk prefix`: adaptor by jnnv2 on the rolling mean, poly-A by jnn_core on pA, statistics of both)
int launch_prefix(const DevBatch& b, int rna004, int32_t* pos4, float* st6, int sm_count, cudaStream_t st);

// ent.cu (`sigtk ent`: entropies of the raw samples, their zig-zag deltas and the deltas' byte planes)
uint64_t ent_overflow_words(int sm_count);
int launch_ent(const DevBatch& b, uint32_t* overflow, double* out3, int sm_count, cudaStream_t st);

}  // namespace sgpu
