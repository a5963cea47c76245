// walk.cu -- walk_chunks_kernel: the first (and dominant) kernel of the fast path.
//
// Every read is cut into CHUNKS of L samples (the last chunk takes the remainder, 1..L samples); ONE THREAD
// walks one chunk with the register-resident walker of walk_core.cuh. A chunk starts W samples early from a cold
// detector state (plus two ring-fill blocks), so chunks are independent: no shared memory, no barriers, no
// inter-thread communication. The detector state a chunk reaches at its first owned position (after the warm-up)
// and the state it ends in are written out (32 B each); verify_chunks_kernel compares every chunk's warm-up state
// with its predecessor's end state. By induction from the read's first chunk (which starts from the reference's
// initial state) all chunks of a read are proven to follow the reference's trajectory; a mismatch routes the read
// to the sequential-order kernels and is counted in fixups[read].
//
// Peaks are owned by the STEP that emits them (not by position): every detector step belongs to exactly one
// chunk, so every peak of the true trajectory is recorded exactly once, with a RED.OR into the event-start bitmap.
//
// The LONG detector is not stepped by the walker (walk_core.cuh): a chunk only tracks where the long detector's
// current life starts and whether one of its stepped positions MAY exceed the long threshold (a conservative float
// test on exact integer window sums). Such lives -- about one per 10,000 samples -- are written to a job list and
// replayed by long_jobs_kernel with the reference's own operations; what they emit is ORed into the same bitmap.
//
// Thread blocks [0, edge_blocks) walk the first / last chunks of the reads (bounds-checked variant, they take
// longest and start first); the remaining blocks walk the interior chunks with the unchecked variant.
#include <cstdlib>

#include "kernels.cuh"
#include "walk_core.cuh"

namespace sgpu {

namespace {

using namespace walk;

// launch shape (measured, tools/run_variants.sh; profiles/r02_variants_occupancy.txt, r02_variants_nt.txt, r02_variants_rna.txt):
// 128-thread blocks, 3 per SM for DNA (168 registers, almost no spills, 3 warps per scheduler) and 2 per SM for RNA
// (254 registers, 2 warps per scheduler). 64 x 6 / 64 x 4: 1 % (DNA) and 4 % (RNA) slower; 4 warps per scheduler
// means 128 registers and spills: 2-8 % slower (DNA), 168 registers for RNA: 12 % slower.
#ifndef WALK_NT
#define WALK_NT 128
#endif
#ifndef WALK_MINB
#define WALK_MINB 3
#endif
#ifndef WALK_MINB_RNA
#define WALK_MINB_RNA 2
#endif
constexpr int WNT = WALK_NT;  // threads per block of walk_chunks_kernel

struct WalkParams {
    DevBatch b;
    int L, W;                       // chunk length, detector warm-up (multiples of U; L >= W + 2U)
    const uint64_t* ibase;          // [n_reads+1] exclusive scan of the interior chunk counts
    float* pa;                      // optional pA output (same layout as samples)
    uint32_t* bitmap;
    int* st_begin;                  // [(2*n_reads + n_interior) * 8] state after the warm-up
    int* st_end;                    // same indexing: state after the chunk's last step
    uint32_t* wit_min;
    uint32_t* wit_max;
    uint32_t* tile_read0;
    uint32_t edge_blocks;
    float thr_long;                 // the long detector's threshold (9.0; a context parameter for tests)
    int4* jobs;                     // [job_cap] {read, chunk, l_start, end}: lives of the long detector to replay
    uint32_t* job_count;
    uint32_t job_cap;
    uint32_t* seq_flag;             // a read whose job does not fit the list goes to the sequential-order kernels
    unsigned long long* counters;   // [3] = number of replayed lives
};

// the memory side of one chunk walk (see walk_core.cuh)
struct DevIo {
    const int16_t* __restrict__ sp;   // the read's first sample
    float* __restrict__ pa;           // the read's first pA (or null)
    uint32_t* __restrict__ bm;        // the bitmap word that holds the read's first sample
    int* __restrict__ st_begin;       // this chunk's state slots
    int* __restrict__ st_end;
    uint32_t* __restrict__ wit_min;   // this read's witness
    uint32_t* __restrict__ wit_max;
    uint32_t* __restrict__ tile_read0;  // per 2048-sample tile; the top bit marks tiles with LOW samples
    uint64_t base;                      // flat position of the read's first sample
    float off, unit;
    int4* __restrict__ jobs;            // job list (walk_core.cuh: lives of the long detector that may emit)
    uint32_t* __restrict__ job_count;
    uint32_t job_cap;
    uint32_t* __restrict__ seq_flag;
    int read, chunk;
    unsigned lanes;              // the lanes of the warp that walk edge chunks together (walk_edge_dev)

    __device__ __forceinline__ void load8(int t, int (&v)[4]) const {
        const int4 w = __ldg(reinterpret_cast<const int4*>(sp + t));
        v[0] = w.x; v[1] = w.y; v[2] = w.z; v[3] = w.w;
    }
    __device__ __forceinline__ bool want_pa() const { return pa != nullptr; }
    // the line that holds sample t on its way into L1 (a thread walks its chunk 16 bytes at a time, a 128-byte line of
    // its own per 8 blocks: asked for a few blocks ahead, the load that crosses into a new line finds it there)
    __device__ __forceinline__ void prefetch(int t) const {
#if !defined(WALK_NO_PREFETCH)
        asm volatile("prefetch.global.L1 [%0];" ::"l"(sp + t));
#endif
    }
    // largest v among the lanes of the warp that walk edge chunks together (`lanes`: their ballot): walk_edge
    __device__ __forceinline__ int warp_max(int v) const { return __reduce_max_sync(lanes, v); }
    __device__ __forceinline__ void store_pa8(int t, const float* x) const {
        float4* dst = reinterpret_cast<float4*>(pa + t);
        __stcs(dst, make_float4(x[0], x[1], x[2], x[3]));      // streaming: nothing on the device reads pA back
        __stcs(dst + 1, make_float4(x[4], x[5], x[6], x[7]));
    }
    __device__ __forceinline__ void store_pa1(int t, float x) const { pa[t] = x; }
    __device__ __forceinline__ void peak(int pos) const { atomicOr(bm + ((uint32_t)pos >> 5), 1u << (pos & 31)); }
    // the peaks of one block: bit k of mk <=> a peak at shifted position ub + k (ub may be negative at the start
    // of a read: those bits are zero, and a zero part is never written)
    __device__ __forceinline__ void peaks32(int ub, uint32_t mk) const {
        const uint32_t s = (uint32_t)ub & 31u;
        const uint32_t lo = mk << s, hi = __funnelshift_l(mk, 0u, s);
        uint32_t* w = bm + (ub >> 5);
        if (lo) atomicOr(w, lo);
        if (hi) atomicOr(w + 1, hi);
    }
    static __device__ __forceinline__ void store_canon(int* __restrict__ dst, const Canon& c) {
        int4* p = reinterpret_cast<int4*>(dst);
        p[0] = make_int4(c.v[0], c.v[1], c.v[2], c.v[3]);
        p[1] = make_int4(c.v[4], c.v[5], c.v[6], c.v[7]);
    }
    __device__ __forceinline__ void put_begin(const Canon& c) const { store_canon(st_begin, c); }
    __device__ __forceinline__ void put_end(const Canon& c) const { store_canon(st_end, c); }
    // Exact-sum witness of a chunk from the extreme raw values: pA is monotone in raw (unit > 0 is checked by
    // build_seq_list_kernel), so the extreme pA sit at the ends of [rmin, rmax]. build_seq_list_kernel needs the
    // smallest NONZERO |pA| and the largest |pA| of the read. Samples with raw <= low_t (LOW: pA <= 0 or barely above;
    // walk_core.cuh) are not covered by the range's lower end: their blocks report their own magnitudes
    // (low_samples), so the minimum published here starts at pA(low_t + 1) > 0.
    __device__ __forceinline__ void witness(int rmin, int rmax, int low_t) const {
        const float xh = __fmul_rn(__fadd_rn((float)rmax, off), unit);
        const float xa = __fmul_rn(__fadd_rn((float)rmin, off), unit);
        atomicMax(wit_max, max(__float_as_uint(xa) & 0x7fffffffu, __float_as_uint(xh) & 0x7fffffffu));
        const int gmin = rmin > low_t ? rmin : low_t + 1;  // smallest raw value that is not LOW
        if (gmin <= rmax) {
            const float xl = __fmul_rn(__fadd_rn((float)gmin, off), unit);
            atomicMin(wit_min, xl > 0.0f ? __float_as_uint(xl) : 1u);  // (xl > 0 by the definition of low_t)
        }
    }
    __device__ __forceinline__ void job(int l_start, int end) const {
        const uint32_t k = atomicAdd(job_count, 1u);
        if (k < job_cap) jobs[k] = make_int4(read, chunk, l_start, end);
        else seq_flag[read] = 1u;       // (list full: the read is redone in order)
    }
    // LOW samples in the group of 8 that holds read index t: magnitudes to the witness, and the 2048-sample tile is
    // marked (top bit of tile_read0) so that emit_events_kernel sums its events with real conversions
    __device__ __forceinline__ void low_samples(int t, uint32_t lo, uint32_t hi) const {
        atomicMin(wit_min, lo);
        atomicMax(wit_max, hi);
        atomicOr(tile_read0 + ((base + (uint64_t)(uint32_t)t) / FAST_TILE), 0x80000000u);
    }
};

__device__ __forceinline__ DevIo make_io(const WalkParams& p, uint32_t r, uint64_t sid, int chunk, int* sh) {
    const uint64_t base = p.b.read_off[r];
    *sh = (int)(base & 31u);
    DevIo io;
    io.sp = p.b.samples + base;
    io.pa = p.pa ? p.pa + base : nullptr;
    io.bm = p.bitmap + (base >> 5);
    io.st_begin = p.st_begin + sid * 8;
    io.st_end = p.st_end + sid * 8;
    io.wit_min = p.wit_min + r;
    io.wit_max = p.wit_max + r;
    io.tile_read0 = p.tile_read0;
    io.base = base;
    io.off = p.b.offset[r];
    io.unit = p.b.unit[r];
    io.jobs = p.jobs; io.job_count = p.job_count; io.job_cap = p.job_cap; io.seq_flag = p.seq_flag;
    io.read = (int)r; io.chunk = chunk;
    return io;
}

template <int RNA>
__device__ __noinline__ void walk_edge_dev(const WalkParams& p, uint32_t r, int last, unsigned lanes) {
    int sh;
    const int n = (int)p.b.read_len[r];
    DevIo io = make_io(p, r, 2ull * r + (uint64_t)last, last ? (int)n_chunks((uint32_t)n, (uint32_t)p.L) - 1 : 0, &sh);
    io.lanes = lanes;
    walk_edge<RNA>(io, n, io.off, io.unit, sh, p.L, p.W, last, p.thr_long);
}

// largest r with ibase[r] <= i (ibase is non-decreasing, ibase[n_reads] > i)
__device__ __forceinline__ uint32_t find_chunk_read(const uint64_t* __restrict__ ibase, uint32_t n_reads, uint64_t i) {
    uint32_t lo = 0, hi = n_reads;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (ibase[mid] <= i) lo = mid; else hi = mid;
    }
    return lo;
}

template <int RNA>
__global__ void __launch_bounds__(WNT, RNA ? WALK_MINB_RNA : WALK_MINB) walk_chunks_kernel(const WalkParams p) {
    if (blockIdx.x < p.edge_blocks) {
        // first chunks of all reads, then (from a warp boundary) their last chunks: the lanes of a warp walk chunks of
        // the same kind and meet between the phases of walk_edge
        const uint32_t per_kind = (p.b.n_reads + 31u) & ~31u;
        const uint64_t e = (uint64_t)blockIdx.x * WNT + threadIdx.x;
        const int last = e >= per_kind;
        const uint64_t r = last ? e - per_kind : e;
        const bool have = r < p.b.n_reads && e < 2ull * per_kind;
        const unsigned lanes = __ballot_sync(0xffffffffu, have);
        if (have) walk_edge_dev<RNA>(p, (uint32_t)r, last, lanes);
        return;
    }
    const uint64_t i = (uint64_t)(blockIdx.x - p.edge_blocks) * WNT + threadIdx.x;
    if (i >= p.ibase[p.b.n_reads]) return;
    const uint32_t r = find_chunk_read(p.ibase, p.b.n_reads, i);
    int sh;
    const int k = (int)(i - p.ibase[r]) + 1;
    DevIo io = make_io(p, r, 2ull * p.b.n_reads + i, k, &sh);
    walk_interior<RNA>(io, (int)p.b.read_len[r], io.off, io.unit, sh, p.L, p.W, k, p.thr_long);
}

// ---- the lives of the long detector that may emit -------------------------------------------------------------------
// One thread per job: long_job() of walk_core.cuh replays the long detector over the life with the reference's own
// operations from the raw samples and ORs what it emits into the bitmap. It reads the END records of the read's
// chunks (where an earlier chunk's life started; the short detector's state at the end of the job's chunk).
struct JobIo {
    const int16_t* __restrict__ sp;
    uint32_t* __restrict__ bm;
    const int* __restrict__ st_end;    // all END records
    uint64_t sid_first, sid_last, sid_int0;   // slots of the read's first / last / first interior chunk
    int nch;
    __device__ __forceinline__ void load8(int t, int (&v)[4]) const {
        const int4 w = __ldg(reinterpret_cast<const int4*>(sp + t));
        v[0] = w.x; v[1] = w.y; v[2] = w.z; v[3] = w.w;
    }
    __device__ __forceinline__ void peak(int pos) const { atomicOr(bm + ((uint32_t)pos >> 5), 1u << (pos & 31)); }
    __device__ __forceinline__ const int* rec(int kk) const {
        const uint64_t sid = kk == 0 ? sid_first : kk == nch - 1 ? sid_last : sid_int0 + (uint64_t)(kk - 1);
        return st_end + sid * 8;
    }
    __device__ __forceinline__ int end_lstart(int kk) const { return rec(kk)[6]; }
    __device__ __forceinline__ void end_short(int kk, float* pv, int* ps) const {
        const int* q = rec(kk);
        *pv = __int_as_float(q[0]); *ps = q[1];
    }
};

// long_job() (walk_core.cuh) with a WARP per life: the lanes form the exact t-statistics of 32 consecutive positions at
// once (each from its own two windows: the double divisions and the square root of events.c:338-361 are a chain of
// ~2,500 cycles per position when one thread steps alone), then every lane steps the detector over the 32 values in
// order. Same operations, same order per position; what is emitted is ORed into the bitmap by lane 0.
// Used for the RNA parameters, whose lives are few and long (windows of 14 and 28 samples, a life per ~50,000
// samples); the DNA batches hold ~30 short lives per 100,000 samples and keep one thread per life.
template <int RNA>
__device__ void long_job_warp(const JobIo& io, int n, int sh, float off, float unit, int L, int k, int l_start, int end,
                              float thr_long, int lane) {
    using C = Cfg<RNA>;
    constexpr int w1 = C::w1, w2 = C::w2;
    for (int kk = k - 1; l_start == LS_PRED && kk >= 0; kk--) l_start = io.end_lstart(kk);
    if (l_start == LS_PRED) return;
    const int stop = n + sh;
    const int own_end = end == LS_CONT ? (k + 1) * L - C::LAG + sh : (end < stop ? end : stop);
    float pv = FLT_MAX; int ps = PS_NONE;
    PeakAcc unused; unused.mk = 0u; unused.oldest = 0;
    bool b2; int p2;
    auto t_at = [&](int u, int w) -> float {
        const int i = u - sh;
        return (i >= w && i + w <= n) ? tstat_exact(io, i, w, n, off, unit) : 0.0f;
    };
    auto emit = [&](int pos) { if (lane == 0) io.peak(pos); };
    for (int base = l_start; base < own_end; base += 32) {
        const float t = base + lane < own_end ? t_at(base + lane, w2) : 0.0f;
        const int cnt = min(32, own_end - base);
        for (int q = 0; q < cnt; q++)
            det_one<false, RNA>(pv, ps, 0, base + q, __shfl_sync(0xffffffffu, t, q), thr_long, unused, b2, p2, emit);
    }
    if (end != LS_CONT) return;
    float spv; int sps;
    io.end_short(k, &spv, &sps);
    for (int base = own_end; base < stop; base += 32) {   // (l_start <= own_end: the life was alive at the chunk's last owned step)
        const bool in = base + lane < stop;
        const float t1 = in ? t_at(base + lane, w1) : 0.0f, t2 = in ? t_at(base + lane, w2) : 0.0f;
        const int cnt = min(32, stop - base);
        for (int q = 0; q < cnt; q++) {
            det_one<true, RNA>(spv, sps, 0, base + q, __shfl_sync(0xffffffffu, t1, q), thr_short<RNA>(), unused, b2, p2, NoEmit());
            if (b2) return;              // reset: the life ended before the long detector's step here
            det_one<false, RNA>(pv, ps, 0, base + q, __shfl_sync(0xffffffffu, t2, q), thr_long, unused, b2, p2, emit);
        }
    }
}

template <int RNA>
__global__ void __launch_bounds__(128) long_jobs_kernel(const WalkParams p) {
    const uint32_t nj = min(*p.job_count, p.job_cap);
    if (blockIdx.x == 0 && threadIdx.x == 0) p.counters[3] = nj;
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
    const int lane = threadIdx.x & 31;
    for (uint32_t j = RNA ? tid >> 5 : tid; j < nj; j += RNA ? nt >> 5 : nt) {
        const int4 job = p.jobs[j];
        const uint32_t r = (uint32_t)job.x;
        const uint64_t base = p.b.read_off[r];
        const int n = (int)p.b.read_len[r];
        JobIo io;
        io.sp = p.b.samples + base;
        io.bm = p.bitmap + (base >> 5);
        io.st_end = p.st_end;
        io.sid_first = 2ull * r; io.sid_last = 2ull * r + 1; io.sid_int0 = 2ull * p.b.n_reads + p.ibase[r];
        io.nch = (int)n_chunks((uint32_t)n, (uint32_t)p.L);
        if (RNA) long_job_warp<RNA>(io, n, (int)(base & 31u), p.b.offset[r], p.b.unit[r], p.L, job.y, job.z, job.w, p.thr_long, lane);
        else long_job<RNA>(io, n, (int)(base & 31u), p.b.offset[r], p.b.unit[r], p.L, job.y, job.z, job.w, p.thr_long);
    }
}

// ---- chunk counts and verification ----------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) chunk_count_kernel(DevBatch b, uint32_t L, uint32_t* __restrict__ cnt) {
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < b.n_reads; r += gridDim.x * blockDim.x) {
        const uint32_t nch = n_chunks(b.read_len[r], L);
        cnt[r] = nch > 2u ? nch - 2u : 0u;
    }
}

// every chunk that started from a speculative (warm-up) state must have reached its predecessor's end state
__global__ void __launch_bounds__(256) verify_chunks_kernel(DevBatch b, uint32_t L, const uint64_t* __restrict__ ibase,
                                                            const int* __restrict__ st_begin,
                                                            const int* __restrict__ st_end,
                                                            uint32_t* __restrict__ seq_flag,
                                                            uint32_t* __restrict__ fixups) {
    const uint64_t n_int = ibase[b.n_reads];
    const uint64_t total = n_int + b.n_reads;  // interior chunks, then the last chunk of every read
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t r;
        uint64_t cur, prev;
        if (t < n_int) {
            r = find_chunk_read(ibase, b.n_reads, t);
            cur = 2ull * b.n_reads + t;
            prev = (t == ibase[r]) ? 2ull * r : cur - 1;
        } else {
            r = (uint32_t)(t - n_int);
            const uint32_t nch = n_chunks(b.read_len[r], L);
            if (nch < 2u) continue;
            cur = 2ull * r + 1;
            prev = (nch == 2u) ? 2ull * r : 2ull * b.n_reads + ibase[r + 1] - 1;
        }
        const int4* a = reinterpret_cast<const int4*>(st_begin + cur * 8);
        const int4* e = reinterpret_cast<const int4*>(st_end + prev * 8);
        const int4 a0 = a[0], a1 = a[1], e0 = e[0], e1 = e[1];
        const bool same = a0.x == e0.x && a0.y == e0.y && a0.z == e0.z && a0.w == e0.w && a1.x == e1.x && a1.y == e1.y;
        if (!same) {
            seq_flag[r] = 1u;
            atomicAdd(&fixups[r], 1u);
        }
    }
}

}  // namespace

// chunk length for a batch: as long as possible (the warm-up is amortised over it) while the batch still yields
// a few waves of chunks. `forced` != 0: the context's development parameter SGPU_PARAM_CHUNK_LEN.
// (measured on the 653 M-sample batches, profiles/r02_chunk_sweep.txt, last section: DNA 512 ... 1536 samples within
//  1 % of each other, powers of two or not, 2048: +3 %, 4096: +5 %; RNA 2048 best, 1024: +10 %, 4096: +2 % -- the
//  reads' first and last chunks grow with the chunk, and fewer waves of blocks even out worse)
uint32_t walk_chunk_len(uint64_t span, uint32_t n_reads, int rna, int sm_count, uint32_t forced) {
    const uint32_t lmin = rna ? 512u : 128u;
    // (measured: for DNA one wave of resident threads is enough, the warm-up is what longer chunks save;
    //  the RNA instantiation does better with four times as many)
    const uint64_t want_chunks = (uint64_t)sm_count * (rna ? 2048ull : 384ull);
    uint32_t L = rna ? 4096u : 1024u;
    while (L > lmin && span / L < want_chunks) L >>= 1;
    // short reads: a read's first and last chunks cost more than the ones in between (and the lanes of a warp wait
    // for the longest last chunk), so a read should be a dozen chunks or more (the reference's 100 real reads, 4,700
    // samples on average: 384 samples per chunk 9 % faster than 1,024)
    if (n_reads) {
        const uint64_t per_read = span / n_reads / 12u / 128u * 128u;
        if (per_read < L) L = per_read > lmin ? (uint32_t)per_read : lmin;
    }
    if (forced >= lmin && forced % 32u == 0u) L = forced;
    return L;
}
uint32_t walk_warmup(int rna, uint32_t forced) {
    // measured boundary mismatches per 10^6 chunk boundaries (bench batches): DNA W=24: 20, 32: 0.4, >= 40: 0 in
    // 2.5 x 10^6; RNA W=192: 24, 256: 0.8, 320: 0 in 1.3 x 10^6. The rate falls by ~50x per 8 (DNA) / ~30x per 64 (RNA)
    // samples; a mismatch only costs the read its place on the fast path.
    // `forced` != 0: SGPU_PARAM_WARMUP (tests force short warm-ups to exercise the mismatch path).
    uint32_t W = rna ? 384u : 48u;
    const uint32_t u = rna ? 16u : 8u;
    if (forced != 0u && forced % u == 0u && forced <= W) W = forced;
    return W;
}
uint64_t walk_state_slots(uint64_t max_samples, uint32_t max_reads) { return 2ull * max_reads + max_samples / 128u + 1u; }
uint32_t walk_job_capacity(uint64_t max_samples) { return (uint32_t)(max_samples / 64u + 4096u); }  // (16 B each)

static WalkParams walk_params(const DevBatch& b, Scratch& sc, float* pa_out, uint32_t* seq_flag, int sm_count) {
    const uint32_t L = walk_chunk_len(b.span, b.n_reads, b.rna, sm_count, sc.tune_chunk_len), W = walk_warmup(b.rna, sc.tune_warmup);
    WalkParams p;
    p.b = b; p.L = (int)L; p.W = (int)W; p.ibase = sc.wk_ibase; p.pa = pa_out; p.bitmap = sc.bitmap;
    p.st_begin = sc.wk_begin; p.st_end = sc.wk_end; p.wit_min = sc.wit_min; p.wit_max = sc.wit_max; p.tile_read0 = sc.tile_read0;
    p.edge_blocks = (uint32_t)((2ull * ((b.n_reads + 31u) & ~31u) + WNT - 1) / WNT);   // (first and last chunks: whole warps each)
    p.thr_long = sc.tune_thr_long;
    p.jobs = reinterpret_cast<int4*>(sc.jobs.get()); p.job_count = sc.job_count; p.job_cap = sc.job_cap; p.seq_flag = seq_flag;
    p.counters = sc.counters;
    return p;
}

int launch_walk(const DevBatch& b, Scratch& sc, float* pa_out, uint32_t* seq_flag, int sm_count, cudaStream_t st) {
    const WalkParams p = walk_params(b, sc, pa_out, seq_flag, sm_count);
    const uint64_t words = (uint64_t)fast_tiles_for(b.span) * (FAST_TILE / 32);
    cudaMemsetAsync(sc.bitmap, 0, (size_t)words * sizeof(uint32_t), st);
    cudaMemsetAsync(sc.job_count, 0, sizeof(uint32_t), st);
    chunk_count_kernel<<<grid_cap(b.n_reads, 256, sm_count * 8), 256, 0, st>>>(b, (uint32_t)p.L, sc.wk_cnt);
    int n = 1 + launch_scan_u32(sc.wk_cnt, b.n_reads, sc.wk_ibase, nullptr, sc, st);
    const uint64_t max_interior = b.span / (uint32_t)p.L;  // every interior chunk covers L distinct samples
    const uint64_t grid = (uint64_t)p.edge_blocks + (max_interior + WNT - 1) / WNT;
    if (b.rna) walk_chunks_kernel<1><<<(unsigned)grid, WNT, 0, st>>>(p);
    else walk_chunks_kernel<0><<<(unsigned)grid, WNT, 0, st>>>(p);
    return n + 1;
}

// the lives of the long detector that may emit (a few per 100,000 samples), replayed exactly
int launch_long_jobs(const DevBatch& b, Scratch& sc, uint32_t* seq_flag, int sm_count, cudaStream_t st) {
    const WalkParams p = walk_params(b, sc, nullptr, seq_flag, sm_count);
    if (b.rna) long_jobs_kernel<1><<<sm_count * 16, 128, 0, st>>>(p);  // (a warp per life)
    else long_jobs_kernel<0><<<sm_count * 4, 128, 0, st>>>(p);
    return 1;
}

int launch_verify_chunks(const DevBatch& b, Scratch& sc, uint32_t* seq_flag, uint32_t* fixups, int sm_count, cudaStream_t st) {
    const uint32_t L = walk_chunk_len(b.span, b.n_reads, b.rna, sm_count, sc.tune_chunk_len);
    const uint64_t max_interior = b.span / L;
    verify_chunks_kernel<<<grid_cap(max_interior + b.n_reads, 256, sm_count * 8), 256, 0, st>>>(
        b, L, sc.wk_ibase, sc.wk_begin, sc.wk_end, seq_flag, fixups);
    return 1;
}

}  // namespace sgpu
