// jnn.cu -- `sigtk jnn`: the stall / homopolymer-stretch segmenter of the reference (src/jnn.c:176-282 jnn_core +
// jnn_raw, parameters jnn.h:24-45 as jnn_print picks them, jnn.c:305-312, or the caller's set: sgpu_set_jnn).
// SURVEY 8f rank 3 (the jnn half).
//
// Per read:   sig = clamp(raw, 0, 1200)                     (rm_outlier, jnn.c:58-75)
//             band = mean(sig) -/+ std_scale * stdv(sig)    (float sums in sample order: stat.cu, exact replay)
//             a counter machine over one bit per sample ("inside the band"), emitting (start, end) pairs.
// The machine is inherently sequential inside a read (its counters carry across the whole read: `w` never resets),
// but when its corrector provably cannot act (error < corrector) it is an automaton of error + 2 states over the
// in-band bit (see below), and automata compose: one WARP takes one read, all lanes turn 1024 samples into 32 in-band
// masks (the test on integers: sig is integer-valued, so `sig < top && sig > bot` is `lo_i <= v <= hi_i` for the
// integers just inside the float band), a prefix scan of the words' state maps gives every lane its starting state,
// and the few stretches long enough to count are handed to lane 0 in order. Other sets step the counters themselves
// (jnn_exact_kernel).
#include "kernels.cuh"

namespace sgpu {

// ---- the machine as an automaton ----------------------------------------------------------------------------------------
// The reference's counters (jnn.c:192-228) are c (samples of the open stretch, tolerated outliers included), w (the
// corrector: `corrector` + every in-band sample of the read so far, never reset), err (tolerated outliers, < error)
// and prev_err (outliers at the very end of the stretch). err is decremented when c >= window, c >= w and c % w == 0.
// That never happens when error < corrector: while err has never been decremented, err <= error, so c = in-band
// samples of the stretch + err <= in-band samples + error < corrector + in-band samples <= w, and the decrement needs
// c >= w; by induction it never happens. (The reference's sets: error 5 < corrector 50.) What remains is: a stretch
// OPENS at an in-band sample and CLOSES at the (error+1)-th out-of-band sample after it, whatever lies in between.
// Where stretches open and close is decided by a finite automaton over the in-band bit with error + 2 states -- open
// with e = 0..error tolerated outliers, or closed (error + 1) -- and the counters are positions: c = closing sample -
// opening sample, prev_err = the out-of-band samples right before the closing one. A 32-sample word is a map of
// states -> states in 3-bit fields (error <= 6: at most 8 states); maps compose, so a warp finds the state at the
// start of each of its 32 words with one prefix scan and all lanes work in parallel. Only a stretch that came in open
// can be long enough to count (sgpu_set_jnn accepts window > 31 and window * stall_len > 31 only, so c >= 32), i.e.
// at most one candidate per word: the first close of a word entered open. Its prev_err <= error <= 6 outliers reach
// into the previous word at most. (tests: every fixture and stall batch vs the oracle, which keeps w and steps sample
// by sample.) Every other set (error >= corrector, where the decrement can act, or error > 6) takes jnn_exact_kernel.
constexpr int JNN_AUTOMATON_MAX_ERR = 6;   // error + 2 <= 8 states in 3-bit fields

// state after the m samples of a word (bit k of `in` = sample k in band, `zeros` = out-of-band samples, both
// limited to m bits), entered in state s; `closed` = error + 1
__device__ __forceinline__ int jnn_word_end(uint32_t in, uint32_t zeros, int m, int s, int closed) {
    int j = 0;
    while (j < m) {
        if (s == closed) {
            const uint32_t rest = in >> j;
            if (rest == 0u) return closed;
            j += __ffs(rest) - 1;
            s = 0;
        }
        uint32_t z = zeros >> j;
        const int need = closed - s, nz = __popc(z);
        if (nz < need) return s + nz;
        for (int k = 1; k < need; k++) z &= z - 1u;
        j += __ffs(z);  // one past the closing sample
        s = closed;
    }
    return s;
}

// (then o first) as packed maps of NS 3-bit fields; NS >= closed + 1 (the fields above `closed` are never read, and
// hold states, so composing them stays in range)
template <int NS>
__device__ __forceinline__ uint32_t jnn_compose(uint32_t first, uint32_t then) {
    uint32_t f = 0;
#pragma unroll
    for (int s = 0; s < NS; s++) f |= ((then >> (3 * ((first >> (3 * s)) & 7u))) & 7u) << (3 * s);
    return f;
}

// the integers just inside the float band mean -/+ fl(sd * std_scale) (jnn.c:184-185): sig is an integer in
// [0, 1200], so sig < top <=> sig <= ceil(top)-1 and sig > bot <=> sig >= floor(bot)+1 (a NaN band -- never for finite
// input and a finite std_scale -- leaves the band empty like the float comparisons do)
__device__ __forceinline__ void jnn_band(float mn, float sd, float std_scale, int& lo_i, int& hi_i) {
    const float band = __fmul_rn(sd, std_scale);
    const float top = __fadd_rn(mn, band), bot = __fsub_rn(mn, band);
    hi_i = -1; lo_i = 0;
    if (top == top && bot == bot) {
        hi_i = (int)ceilf(fminf(fmaxf(top, -1.0f), 2000.0f)) - 1;
        lo_i = (int)floorf(fminf(fmaxf(bot, -2.0f), 2000.0f)) + 1;
    }
}

// bit k = sample k of the lane's 32 (the four 128-bit words `cur`) clamped to [0, 1200] inside [lo_i, hi_i]
__device__ __forceinline__ uint32_t jnn_in_mask(const uint4 (&cur)[4], int lo_i, int hi_i) {
    uint32_t in = 0;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const uint32_t wd[4] = {cur[q].x, cur[q].y, cur[q].z, cur[q].w};
#pragma unroll
        for (int h = 0; h < 8; h++) {
            const int v = (int)(int16_t)(wd[h >> 1] >> ((h & 1) * 16));
            const int sv = min(max(v, 0), 1200);
            in |= (uint32_t)(sv >= lo_i && sv <= hi_i) << (q * 8 + h);
        }
    }
    return in;
}

// seg: pairs (x, y) of read r at seg[2*(base(r)+k)], base(r) = read_off[r]/32 + r (a read of n samples has at most
// n/32 + 1 segments: every counted stretch is at least 32 samples long, sgpu_set_jnn's window rule).
//
// One WARP per read, 1024 samples per step: every lane loads 32 of them (64 contiguous bytes; the next 1024 are
// already in flight) and reduces them to a 32-bit in-band mask, its word's state map and, after the scan, its
// events; lane 0 applies the segment rules (threshold, first-segment rule, merge: jnn.c:230-245) to the few
// candidates in order. (One thread per read: 15 ms on the 651 M-sample batch and 240 ms on 320 reads of 2 M samples;
// one lane stepping through the masks of a warp-loaded block: 15 ms / 78 ms.) NS: 3-bit fields a map composes,
// P.error + 2 rounded up to 7 (8 only for error 6, so the reference's sets compose seven fields as before). CLOSED:
// error + 1 when it is known at compile time (6: error 5, the reference's sets, whose loops over the states then unroll
// as they did before the sets were runtime values: a runtime `closed` costs 7 % of jnn_walk on the bench batch), or 0.
template <int NS, int CLOSED>
__global__ void __launch_bounds__(128) jnn_walk_kernel(DevBatch b, const JnnParams P, const float* __restrict__ moments,
                                                       uint32_t* __restrict__ seg_cnt, int32_t* __restrict__ seg) {
    const int closed = CLOSED > 0 ? CLOSED : P.error + 1;
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    // the state map of every 8-sample pattern: a full word's map is the composition of its four bytes' maps (three
    // compositions, no data-dependent loop; the stepping form above costs a loop per entry state)
    __shared__ uint32_t byte_map[256];
    for (int v = threadIdx.x; v < 256; v += blockDim.x) {
        uint32_t f = 0;
        for (int s = 0; s <= closed; s++)
            f |= (uint32_t)jnn_word_end((uint32_t)v, ~(uint32_t)v & 0xffu, 8, s, closed) << (3 * s);
        byte_map[v] = f;
    }
    __syncthreads();
    for (uint32_t r = warp; r < b.n_reads; r += n_warps) {
        const int16_t* __restrict__ raw = b.samples + b.read_off[r];
        const int n = (int)b.read_len[r];
        int32_t* out = seg + 2 * ((b.read_off[r] >> 5) + r);
        if (n == 0) { if (lane == 0) seg_cnt[r] = 0; continue; }
        int lo_i, hi_i;
        jnn_band(moments[2 * r], moments[2 * r + 1], P.std_scale, lo_i, hi_i);
        const float first_min = __fmul_rn((float)P.window, P.stall_len);      // jnn.c:232
        const float cand_min = fminf((float)P.window, first_min);
        int n_seg = 0, last_y = 0;              // live on lane 0
        int state = closed;                     // automaton state at the start of the block (uniform)
        int open_pos = 0;                       // where the stretch open at the start of the block began (uniform)
        uint32_t last_word = 0xffffffffu;       // the word before the block (uniform)
        const uint4* __restrict__ src = reinterpret_cast<const uint4*>(raw);
        const int n_words = (n + 7) >> 3;       // 128-bit words that hold samples of this read
        uint4 cur[4], nxt[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int wq = lane * 4 + q;
            cur[q] = wq < n_words ? __ldg(src + wq) : make_uint4(0, 0, 0, 0);
        }
        for (int t0 = 0; t0 < n; t0 += 1024) {
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int wq = ((t0 + 1024) >> 3) + lane * 4 + q;
                nxt[q] = wq < n_words ? __ldg(src + wq) : make_uint4(0, 0, 0, 0);
            }
            uint32_t in = jnn_in_mask(cur, lo_i, hi_i);
            const int i0 = t0 + lane * 32;
            const int m = max(0, min(32, n - i0));                            // samples of this lane's word in the read
            const uint32_t valid = m == 32 ? 0xffffffffu : (1u << m) - 1u;
            in &= valid;
            const uint32_t zeros = ~in & valid;
            // 1. the word as a map of states, and the state at its start
            uint32_t f = 0;
            if (m == 32) {
                f = jnn_compose<NS>(jnn_compose<NS>(byte_map[in & 0xffu], byte_map[(in >> 8) & 0xffu]),
                                    jnn_compose<NS>(byte_map[(in >> 16) & 0xffu], byte_map[in >> 24]));
            } else {   // the last words of a read
                for (int s = 0; s <= closed; s++) f |= (uint32_t)jnn_word_end(in, zeros, m, s, closed) << (3 * s);
            }
            uint32_t incl = f;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t before = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl = jnn_compose<NS>(before, incl);
            }
            uint32_t excl = __shfl_up_sync(0xffffffffu, incl, 1);
            const int s_in = lane ? (int)((excl >> (3 * state)) & 7u) : state;
            uint32_t prev_in = __shfl_up_sync(0xffffffffu, in, 1);
            if (lane == 0) prev_in = last_word;
            // 2. this word's events: the close of the stretch that came in open (the only possible candidate) and
            //    the last stretch opened here
            int close_at = -1, perr = 0, last_open = -1;
            {
                int j = 0, s = s_in;
                while (j < m) {
                    if (s == closed) {
                        const uint32_t rest = in >> j;
                        if (rest == 0u) break;
                        j += __ffs(rest) - 1;
                        s = 0;
                        last_open = i0 + j;
                    }
                    uint32_t z = zeros >> j;
                    const int need = closed - s;
                    if (__popc(z) < need) break;
                    for (int k = 1; k < need; k++) z &= z - 1u;
                    const int pos = j + __ffs(z) - 1;                         // the closing sample
                    if (j == 0 && s_in != closed && close_at < 0) {
                        close_at = pos;
                        const uint32_t below = pos ? (in & ((1u << pos) - 1u)) : 0u;
                        // out-of-band samples right before it (they reach into the previous word when nothing in
                        // band precedes it here; at most error <= 6, all tolerated)
                        perr = below ? (pos - 1) - (31 - __clz(below)) : pos + __clz(prev_in);
                    }
                    j = pos + 1;
                    s = closed;
                }
            }
            // 3. where the stretch open at the start of each word began: the last opening before it
            int open_incl = last_open;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) open_incl = max(open_incl, __shfl_up_sync(0xffffffffu, open_incl, d));
            int open_before = __shfl_up_sync(0xffffffffu, open_incl, 1);
            open_before = lane ? max(open_before, open_pos) : open_pos;
            int c = 0, c_start = 0, c_end = 0;
            bool cand = false;
            if (close_at >= 0) {
                c_start = open_before;
                c = i0 + close_at - c_start;
                c_end = i0 + close_at - perr;
                cand = (float)c >= cand_min;
            }
            // 4. lane 0 takes the candidates in order (jnn.c:230-245)
            uint32_t todo = __ballot_sync(0xffffffffu, cand);
            while (todo) {
                const int src_lane = __ffs(todo) - 1;
                todo &= todo - 1u;
                const int cc = __shfl_sync(0xffffffffu, c, src_lane);
                const int st = __shfl_sync(0xffffffffu, c_start, src_lane);
                const int en = __shfl_sync(0xffffffffu, c_end, src_lane);
                if (lane == 0 && (cc >= P.window || (!n_seg && (float)cc >= first_min))) {
                    if (n_seg && st - last_y < P.seg_dist) {
                        out[2 * (n_seg - 1) + 1] = en;
                    } else {
                        out[2 * n_seg] = st;
                        out[2 * n_seg + 1] = en;
                        n_seg++;
                    }
                    last_y = en;
                }
            }
            // carry to the next block
            state = (int)((__shfl_sync(0xffffffffu, incl, 31) >> (3 * state)) & 7u);
            open_pos = max(open_pos, __shfl_sync(0xffffffffu, open_incl, 31));
            last_word = __shfl_sync(0xffffffffu, in, 31);
#pragma unroll
            for (int q = 0; q < 4; q++) cur[q] = nxt[q];
        }
        if (lane == 0) seg_cnt[r] = (uint32_t)n_seg;
    }
}

// ---- the exact route: the reference's counter machine, corrector included ----------------------------------------------
// For sets where the automaton does not hold (error >= corrector: the decrement of err can act, so a stretch may
// tolerate any number of outliers; or error > 6: more states than 3-bit fields hold). One WARP per read loads 1024
// samples per step and turns them into 32 in-band masks as jnn_walk_kernel does; lane 0 then steps c, w, err and
// prev_err through them exactly as jnn.c:192-245 does, sample by sample, except that it crosses a closed gap (no
// counter changes on an out-of-band sample there) and an in-band run during which c < w (c and w both grow by one per
// in-band sample, so the decrement's c >= w stays false) in one step. w is kept in 64 bits (corrector + in-band
// samples so far may pass 2^31 - 1 for a corrector near it; where the decrement is tested, 1 <= w <= c < 2^31).
__global__ void __launch_bounds__(128) jnn_exact_kernel(DevBatch b, const JnnParams P, const float* __restrict__ moments,
                                                        uint32_t* __restrict__ seg_cnt, int32_t* __restrict__ seg) {
    __shared__ uint32_t masks[4][32];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t r = warp; r < b.n_reads; r += n_warps) {
        const int16_t* __restrict__ raw = b.samples + b.read_off[r];
        const int n = (int)b.read_len[r];
        int32_t* out = seg + 2 * ((b.read_off[r] >> 5) + r);
        if (n == 0) { if (lane == 0) seg_cnt[r] = 0; continue; }
        int lo_i, hi_i;
        jnn_band(moments[2 * r], moments[2 * r + 1], P.std_scale, lo_i, hi_i);
        const float first_min = __fmul_rn((float)P.window, P.stall_len);      // jnn.c:232
        // the counters (live on lane 0): c, w, err, prev_err of jnn.c:192, and the open stretch's first sample
        bool open = false;
        int c = 0, err = 0, prev_err = 0, first = 0, n_seg = 0, last_y = 0;
        long long w = P.corrector;
        const uint4* __restrict__ src = reinterpret_cast<const uint4*>(raw);
        const int n_words = (n + 7) >> 3;
        uint4 cur[4], nxt[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int wq = lane * 4 + q;
            cur[q] = wq < n_words ? __ldg(src + wq) : make_uint4(0, 0, 0, 0);
        }
        for (int t0 = 0; t0 < n; t0 += 1024) {
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int wq = ((t0 + 1024) >> 3) + lane * 4 + q;
                nxt[q] = wq < n_words ? __ldg(src + wq) : make_uint4(0, 0, 0, 0);
            }
            masks[wib][lane] = jnn_in_mask(cur, lo_i, hi_i);
            __syncwarp();
            if (lane == 0) {
                for (int k = 0; k < 32 && t0 + 32 * k < n; k++) {
                    const int i0 = t0 + 32 * k, m = min(32, n - i0);
                    const uint32_t in = masks[wib][k] & (m == 32 ? 0xffffffffu : (1u << m) - 1u);
                    int j = 0;
                    while (j < m) {
                        if (!open) {                   // out-of-band samples of a closed gap change nothing
                            const uint32_t rest = in >> j;
                            if (rest == 0u) break;
                            j += __ffs(rest) - 1;
                            open = true;
                            first = i0 + j;
                        }
                        if ((in >> j) & 1u) {          // in band: c++, w++, prev_err = 0, then the corrector
                            const uint32_t outs = ~(in >> j);  // (zero only for a word all in band, j = 0)
                            const int run = min(outs ? __ffs(outs) - 1 : 32, m - j);   // in-band samples from j on
                            prev_err = 0;
                            if ((long long)c < w) {    // c - w is the same after each of them: never c >= w
                                c += run; w += run; j += run;
                            } else {
                                for (int e = 0; e < run; e++) {
                                    c++; w++;
                                    if (c >= P.window && (long long)c >= w && c % (int)w == 0) err--;
                                }
                                j += run;
                            }
                        } else if (err < P.error) {    // a tolerated outlier
                            c++; err++; prev_err++;
                            if (c >= P.window && (long long)c >= w && c % (int)w == 0) err--;
                            j++;
                        } else {                       // the stretch closes at sample i0 + j (jnn.c:230-245)
                            if (c >= P.window || (!n_seg && (float)c >= first_min)) {
                                const int stop = i0 + j - prev_err;
                                if (n_seg && first - last_y < P.seg_dist) {
                                    out[2 * (n_seg - 1) + 1] = stop;
                                } else {
                                    out[2 * n_seg] = first;
                                    out[2 * n_seg + 1] = stop;
                                    n_seg++;
                                }
                                last_y = stop;
                            }
                            open = false; c = 0; err = 0; prev_err = 0;
                            j++;
                        }
                    }
                }
            }
            __syncwarp();
#pragma unroll
            for (int q = 0; q < 4; q++) cur[q] = nxt[q];
        }
        if (lane == 0) seg_cnt[r] = (uint32_t)n_seg;
    }
}

uint64_t jnn_seg_capacity(uint64_t max_samples, uint32_t max_reads) { return max_samples / 32 + max_reads + 1; }

// moments: [n_reads][2] from launch_jnn_moments (stat.cu); seg_cnt: [n_reads]; seg: [2 * jnn_seg_capacity]
int launch_jnn(const DevBatch& b, const JnnParams& p, const float* moments, uint32_t* seg_cnt, int32_t* seg,
               int sm_count, cudaStream_t st) {
    if (b.n_reads == 0) return 0;
    // one warp per read; few reads: one warp per block so that they spread over the SMs
    const int threads = b.n_reads < (uint32_t)sm_count * 4u ? 32 : 128;
    const int g = (int)((b.n_reads + (threads / 32) - 1) / (threads / 32));
    if (p.error > JNN_AUTOMATON_MAX_ERR || p.error >= p.corrector)
        jnn_exact_kernel<<<g, threads, 0, st>>>(b, p, moments, seg_cnt, seg);
    else if (p.error == 5)
        jnn_walk_kernel<7, 6><<<g, threads, 0, st>>>(b, p, moments, seg_cnt, seg);
    else if (p.error < 5)
        jnn_walk_kernel<7, 0><<<g, threads, 0, st>>>(b, p, moments, seg_cnt, seg);
    else
        jnn_walk_kernel<8, 0><<<g, threads, 0, st>>>(b, p, moments, seg_cnt, seg);
    return 1;
}

}  // namespace sgpu
