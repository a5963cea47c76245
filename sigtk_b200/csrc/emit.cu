// emit.cu -- emit_events_kernel: the event table (create_events / create_event, events.c:457-504) from the
// event-start bitmap. One WARP per 1024 consecutive samples of the flat array (32 bitmap words), no block-level
// barriers, no scan over the samples. The sums are exact (see walk_core.cuh), so every grouping of the additions
// gives the reference's bits.
//
//   1. every lane takes one bitmap word; a warp scan of the popcounts gives every event start its index in the
//      warp tile, and the lanes scatter the start positions into a warp-private list in shared memory;
//   2. FAST PATH (the warp tile lies inside one read; reads are much longer than 1024 samples): every lane walks the
//      32 samples of its word once and cuts the running sums of x and x*x at its event-start bits: the piece
//      before its first bit (`head`), and one piece per bit (up to the next bit or the end of the word), all
//      stored in shared memory. Every lane does the same 32 steps: no divergence in the sample loop.
//   3. the events are dealt to the lanes in order (event j0+lane); an event is its own piece, plus -- when it is
//      the last one of its word -- the heads of the following words up to the next event start. Only the last
//      event of the tile can run past it; its lane adds those few samples straight from global memory.
//      Consecutive lanes write consecutive event slots.
//   GENERAL PATH (a read starts or ends inside the warp tile): every lane sums the samples of its event directly.
#include "kernels.cuh"
#include "walk_core.cuh"

namespace sgpu {

namespace {

constexpr int EWT = 1024;                // samples per warp tile
constexpr int EWARPS = 4;                // warps per CTA
constexpr int ELIST = EWT / 2 + 8;       // event starts are >= 3 samples apart inside a read; tiny reads add their starts
constexpr int EFAST = EWT / 3 + 8;       // bound inside ONE read
constexpr int ELONG = 48;                // general path: an event longer than this is finished by the whole warp

struct EmitWarp {
    double S[EFAST + 32];                // pieces by event index, then the 32 heads
    double Q[EFAST + 32];
    uint16_t list[ELIST];
};

// read that contains flat position p of a 2048-sample tile whose first candidate read is r0 (tile_read0)
__device__ __forceinline__ uint32_t locate_read(const DevBatch& b, uint32_t r0, uint64_t p) {
    uint32_t r = r0;
#pragma unroll 1
    for (int k = 0; k < 4; k++) {
        if (r + 1 >= b.n_reads || b.read_off[r + 1] > p) return r;
        r++;
    }
    return find_read(b.read_off, b.n_reads, p);
}

__device__ __forceinline__ void add_raw(int raw, float off, float unit, double& as, double& aq) {
    const float x = __fmul_rn(__fadd_rn((float)raw, off), unit);
    // widen_pos: exact for the positive pA of every read that keeps the fast path's results (walk_core.cuh)
    as = __dadd_rn(as, walk::widen_pos(x));
    aq = __dadd_rn(aq, walk::widen_pos(__fmul_rn(x, x)));
}
// the same for any sample when `safe` (tiles marked by the walker as holding LOW samples): real conversions for the
// values the shortcut does not cover
__device__ __forceinline__ void add_raw_any(int raw, float off, float unit, double& as, double& aq, bool safe) {
    const float x = __fmul_rn(__fadd_rn((float)raw, off), unit);
    if (!safe || x > 0.0f) {
        as = __dadd_rn(as, walk::widen_pos(x));
        aq = __dadd_rn(aq, walk::widen_pos(__fmul_rn(x, x)));
    } else {
        as = __dadd_rn(as, (double)x);
        aq = __dadd_rn(aq, (double)__fmul_rn(x, x));
    }
}

// next event start at or after bitmap word w0, bounded by the end of the read
__device__ __forceinline__ long long next_start(const uint32_t* __restrict__ bitmap, uint64_t w0, uint64_t n_words,
                                                long long rend) {
    for (uint64_t w = w0; w < n_words && (long long)(w << 5) < rend; w++) {
        const uint32_t nx = bitmap[w];
        if (nx) {
            const long long e = (long long)(w << 5) + __ffs(nx) - 1;
            return e < rend ? e : rend;
        }
    }
    return rend;
}

}  // namespace

// launch shape (measured, tools/run_variants.sh): 7 CTAs of 4 warps per SM (72 registers) and a grid of 64 CTAs per SM --
// warp tiles differ in cost (read boundaries, event density), a finer static partition evens the tail out
#ifndef EMIT_MINB
#define EMIT_MINB 7
#endif
#ifndef EMIT_GRID
#define EMIT_GRID 64
#endif
__global__ void __launch_bounds__(EWARPS * 32, EMIT_MINB) emit_events_kernel(DevBatch b, uint32_t n_tiles,
                                                                  const uint32_t* __restrict__ bitmap,
                                                                  const uint64_t* __restrict__ tile_base, uint64_t ev_cap,
                                                                  uint32_t* __restrict__ ev_start,
                                                                  float* __restrict__ ev_mean, float* __restrict__ ev_stdv,
                                                                  int* __restrict__ status,
                                                                  const uint32_t* __restrict__ tile_read0) {
    __shared__ EmitWarp smem[EWARPS];
    const int lane = threadIdx.x & 31;
    EmitWarp& sm = smem[threadIdx.x >> 5];
    const uint64_t n_wt = (uint64_t)n_tiles * (FAST_TILE / EWT);
    const uint64_t n_words = (uint64_t)n_tiles * (FAST_TILE / 32);
    const uint64_t warp0 = (uint64_t)blockIdx.x * EWARPS + (threadIdx.x >> 5), n_warps = (uint64_t)gridDim.x * EWARPS;
    const long long span = (long long)b.span;
    // the bitmap word and the 32 samples of a lane are loaded one warp tile ahead (their latency hides behind the
    // previous tile's work)
    auto load_tile = [&](uint64_t wt, uint32_t& word, int4 (&rv)[4]) {
        const long long p0 = (long long)wt * EWT + lane * 32;
        word = 0u;
#pragma unroll
        for (int g = 0; g < 4; g++) rv[g] = make_int4(0, 0, 0, 0);
        if (wt < n_wt && (long long)wt * EWT < span) {
            word = bitmap[wt * 32 + lane];
            const int4* __restrict__ src = reinterpret_cast<const int4*>(b.samples + p0);
#pragma unroll
            for (int g = 0; g < 4; g++) if (p0 + 8 * g + 8 <= span) rv[g] = __ldg(src + g);
        }
    };
    uint32_t word_n;
    int4 rv_n[4];
    load_tile(warp0, word_n, rv_n);
    for (uint64_t wt = warp0; wt < n_wt; wt += n_warps) {
        const long long flat0 = (long long)wt * EWT;
        if (flat0 >= span) break;
        const uint32_t tile = (uint32_t)(wt / (FAST_TILE / EWT)), half = (uint32_t)(wt % (FAST_TILE / EWT));
        const uint32_t word = word_n;
        int4 rv[4];
#pragma unroll
        for (int g = 0; g < 4; g++) rv[g] = rv_n[g];
        load_tile(wt + n_warps, word_n, rv_n);
        const uint64_t tbase = tile_base[tile];
        const uint32_t tr0_raw = tile_read0[tile];
        const uint32_t tr0 = tr0_raw & 0x7fffffffu;
        const bool tile_low = (tr0_raw >> 31) != 0u;  // the walker found LOW samples (pA <= 0 or barely above) in this tile
        uint32_t before = half ? (uint32_t)__popc(bitmap[(uint64_t)tile * (FAST_TILE / 32) + lane]) : 0u;
        before = __reduce_add_sync(0xffffffffu, before);  // FAST_TILE / EWT == 2: at most one warp tile before this one
        uint32_t incl = __popc(word);
        const uint32_t own = incl;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
        if (total == 0u) continue;
        if (total > (uint32_t)ELIST) { total = ELIST; if (lane == 0) atomicExch(status, SGPU_DEV_E_EVCAP); }  // malformed bitmap
        __syncwarp();  // the previous tile's readers are done with the shared arrays
        {
            uint32_t rem = word, idx = incl - own;
            while (rem) {
                if (idx < (uint32_t)ELIST) sm.list[idx] = (uint16_t)(lane * 32 + __ffs(rem) - 1);
                idx++;
                rem &= rem - 1u;
            }
        }
        const uint64_t kbase = tbase + before;
        // the read of the tile's first sample; when it covers the whole warp tile every event of the tile shares
        // its parameters
        const uint32_t r_first = locate_read(b, tr0, (uint64_t)flat0);
        const long long rs_first = (long long)b.read_off[r_first];
        const long long rend_first = rs_first + (long long)b.read_len[r_first];
        const float off_first = b.offset[r_first], unit_first = b.unit[r_first];
        // (a tile with LOW samples takes the general path: its sums need real conversions)
        const bool one_read = rs_first <= flat0 && flat0 + EWT <= rend_first && total <= (uint32_t)EFAST && !tile_low;
        if (one_read) {
            // the tile's last event runs on past the tile: the next tile's bitmap words and the first 32 samples behind
            // the tile are asked for now, one per lane, and used after step 2 (when one lane looked for the event's end
            // and added its samples on its own, the other 31 waited on its loads at the end of every tile)
            const uint64_t w_next = (wt + 1) * 32 + (uint64_t)lane;
            const bool w_valid = w_next < n_words && (long long)(w_next << 5) < rend_first;
            const uint32_t next_bits = w_valid ? bitmap[w_next] : 0u;
            const long long i_behind = flat0 + EWT + lane;
            const int raw_behind = i_behind < rend_first ? (int)__ldg(b.samples + i_behind) : 0;
            // ---- fast path, step 2: the pieces of this lane's 32 samples ----------------------------------------------
            int slot = EFAST + lane;             // where the running piece goes: first the head of this word
            int next = (int)(incl - own);        // index of this word's first event
            double as = 0.0, aq = 0.0;
#pragma unroll
            for (int g = 0; g < 4; g++) {
                const int v[4] = {rv[g].x, rv[g].y, rv[g].z, rv[g].w};
                float x[8];
                walk::cvt8(v, off_first, unit_first, x);           // misc.c:28, two samples per instruction, no conversion unit
                float xq[8];
#pragma unroll
                for (int m = 0; m < 8; m += 2) {
                    const walk::F2 p = {x[m], x[m + 1]};
                    const walk::F2 q = walk::f2sq(p);              // float squares (events.c:301)
                    xq[m] = q.lo; xq[m + 1] = q.hi;
                }
#pragma unroll
                for (int m = 0; m < 8; m++) {
                    if ((word >> (8 * g + m)) & 1u) {  // an event starts here: the running piece is complete
                        sm.S[slot] = as;
                        sm.Q[slot] = aq;
                        slot = next++;
                        as = 0.0;
                        aq = 0.0;
                    }
                    // widen_pos: exact for the positive pA of every read that keeps the fast path's results
                    as = __dadd_rn(as, walk::widen_pos(x[m]));
                    aq = __dadd_rn(aq, walk::widen_pos(xq[m]));
                }
            }
            sm.S[slot] = as;
            sm.Q[slot] = aq;
            __syncwarp();
            // the head of a word with event starts (and the empty words before it) belongs to the last event of the
            // previous word with starts: exactly one lane adds to any event
            const uint32_t nz = __ballot_sync(0xffffffffu, own != 0u);
            if (own != 0u && incl != own) {
                double hs = sm.S[EFAST + lane], hq = sm.Q[EFAST + lane];
                const uint32_t lower = nz & ((1u << lane) - 1u);   // non-empty because incl != own
                for (int l2 = lane - 1; l2 > 31 - __clz(lower); l2--) {
                    hs = __dadd_rn(hs, sm.S[EFAST + l2]);
                    hq = __dadd_rn(hq, sm.Q[EFAST + l2]);
                }
                const int prev = (int)(incl - own) - 1;
                sm.S[prev] = __dadd_rn(sm.S[prev], hs);
                sm.Q[prev] = __dadd_rn(sm.Q[prev], hq);
            }
            __syncwarp();
            const int last_word = 31 - __clz(nz);
            // where the tile's last event ends (the next start, at most the read's end), and what it has beyond its
            // own piece: the heads of the empty words behind it and the samples past the tile -- by the whole warp
            long long e_tail;
            {
                const uint32_t m = __ballot_sync(0xffffffffu, next_bits != 0u);
                const uint32_t all_valid = __ballot_sync(0xffffffffu, w_valid);
                if (m) {
                    const int l0 = __ffs(m) - 1;
                    const uint32_t bits0 = __shfl_sync(0xffffffffu, next_bits, l0);
                    e_tail = (long long)(((wt + 1) * 32 + (uint64_t)l0) << 5) + __ffs(bits0) - 1;
                    if (e_tail > rend_first) e_tail = rend_first;
                } else if (all_valid == 0xffffffffu) {
                    e_tail = next_start(bitmap, (wt + 2) * 32, n_words, rend_first);   // (an event of more than 1,024 samples)
                } else {
                    e_tail = rend_first;
                }
            }
            double tail_s = lane > last_word ? sm.S[EFAST + lane] : 0.0, tail_q = lane > last_word ? sm.Q[EFAST + lane] : 0.0;
            if (i_behind < e_tail) add_raw_any(raw_behind, off_first, unit_first, tail_s, tail_q, true);
            for (long long i = i_behind + 32; i < e_tail; i += 32) add_raw_any((int)__ldg(b.samples + i), off_first, unit_first, tail_s, tail_q, true);
#pragma unroll
            for (int o = 16; o; o >>= 1) {   // (exact sums: any order)
                tail_s = __dadd_rn(tail_s, __shfl_xor_sync(0xffffffffu, tail_s, o));
                tail_q = __dadd_rn(tail_q, __shfl_xor_sync(0xffffffffu, tail_q, o));
            }
            // ---- step 3: events in order ---------------------------------------------------------------------------------
            for (uint32_t j0 = 0; j0 < total; j0 += 32) {
                const uint32_t j = j0 + lane;
                if (j >= total) continue;
                const int pos = sm.list[j];
                double es = sm.S[j], eq = sm.Q[j];
                long long e;
                if (j + 1 < total) {
                    e = flat0 + sm.list[j + 1];
                } else {  // the last event of the tile: the empty words after it, then past the tile
                    es = __dadd_rn(es, tail_s);
                    eq = __dadd_rn(eq, tail_q);
                    e = e_tail;
                }
                const uint64_t k = kbase + j;
                if (k >= ev_cap) { atomicExch(status, SGPU_DEV_E_EVCAP); continue; }
                const long long s = flat0 + pos;
                float mean, stdv;
                event_stats(es, eq, (uint32_t)(e - s), &mean, &stdv);
                ev_start[k] = (uint32_t)(s - rs_first);
                ev_mean[k] = mean;
                ev_stdv[k] = stdv;
            }
            continue;
        }
        // ---- general path: a read boundary inside the warp tile ---------------------------------------------------------
        __syncwarp();
        // an event may run on into the next tile(s), whose marks are not known here: only a tile of one read that is
        // itself unmarked keeps the shortcut for every sample
        const bool safe = true;
        for (uint32_t j0 = 0; j0 < total; j0 += 32) {
            const uint32_t j = j0 + lane;
            const bool have = j < total;
            long long i = 0, e = 0, rs = 0;
            float off = 0.0f, unit = 0.0f;
            double as = 0.0, aq = 0.0;
            uint32_t len = 0;
            if (have) {
                const long long s = flat0 + sm.list[j];
                const uint32_t r = locate_read(b, r_first, (uint64_t)s);
                rs = (long long)b.read_off[r];
                const long long rend = rs + (long long)b.read_len[r];
                off = b.offset[r];
                unit = b.unit[r];
                e = j + 1 < total ? flat0 + sm.list[j + 1] : next_start(bitmap, (wt + 1) * 32, n_words, rend);
                if (e > rend) e = rend;
                len = (uint32_t)(e - s);
                i = s;
                const long long stop = e - s > ELONG ? s + ELONG : e;
                for (; i < stop; i++) add_raw_any((int)__ldg(b.samples + i), off, unit, as, aq, safe);
            }
            // long events (rare): the whole warp sums the rest
            uint32_t longs = __ballot_sync(0xffffffffu, have && i < e);
            while (longs) {
                const int src = __ffs(longs) - 1;
                longs &= longs - 1u;
                const long long li = __shfl_sync(0xffffffffu, i, src), le = __shfl_sync(0xffffffffu, e, src);
                const float lo = __shfl_sync(0xffffffffu, off, src), lu = __shfl_sync(0xffffffffu, unit, src);
                double ps = 0.0, pq = 0.0;
                for (long long p = li + lane; p < le; p += 32) add_raw_any((int)__ldg(b.samples + p), lo, lu, ps, pq, safe);
#pragma unroll
                for (int o = 16; o; o >>= 1) {
                    ps = __dadd_rn(ps, __shfl_xor_sync(0xffffffffu, ps, o));
                    pq = __dadd_rn(pq, __shfl_xor_sync(0xffffffffu, pq, o));
                }
                if (lane == src) { as = __dadd_rn(as, ps); aq = __dadd_rn(aq, pq); }
            }
            if (have) {
                const uint64_t k = kbase + j;
                if (k >= ev_cap) { atomicExch(status, SGPU_DEV_E_EVCAP); continue; }
                float mean, stdv;
                event_stats(as, aq, len, &mean, &stdv);
                ev_start[k] = (uint32_t)(e - (long long)len - rs);
                ev_mean[k] = mean;
                ev_stdv[k] = stdv;
            }
        }
    }
}

__global__ void __launch_bounds__(256) sum_fixups_kernel(uint32_t n_reads, const uint32_t* __restrict__ fixups,
                                                         unsigned long long* __restrict__ counters) {
    unsigned long long acc = 0;
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < n_reads; r += gridDim.x * blockDim.x) acc += fixups[r];
    if (acc) atomicAdd(&counters[2], acc);
}

int launch_fast_emit(const DevBatch& b, Scratch& sc, uint64_t ev_cap, uint32_t* ev_start, float* ev_mean,
                     float* ev_stdv, const uint32_t* fixups, int sm_count, cudaStream_t st) {
    const uint32_t n_tiles = fast_tiles_for(b.span);
    const uint64_t n_wt = (uint64_t)n_tiles * (FAST_TILE / EWT);
    emit_events_kernel<<<grid_cap(n_wt, EWARPS, sm_count * EMIT_GRID), EWARPS * 32, 0, st>>>(
        b, n_tiles, sc.bitmap, sc.tile_base, ev_cap, ev_start, ev_mean, ev_stdv, sc.status, sc.tile_read0);
    sum_fixups_kernel<<<grid_cap(b.n_reads, 256, sm_count * 4), 256, 0, st>>>(b.n_reads, fixups, sc.counters);
    return 2;
}

}  // namespace sgpu
