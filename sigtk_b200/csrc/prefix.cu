// prefix.cu -- `sigtk prefix` (reference src/cfunc.c:169-234): the adaptor stretch at the start of a direct-RNA
// read, the poly-A stretch behind it, and the float statistics of both.
//
//   find_adaptor = jnnv2 (jnn.c:99-179) with JNNV2_RNA_R9_ADAPTOR / JNNV2_RNA_RNA004_ADAPTOR (jnn.h:88-102), or the
//     caller's adaptor set (sgpu_set_prefix): the raw samples clamped to [0, 1200] (rm_outlier, jnn.c:58-75), their
//     rolling mean over `window` (2,000) samples (rolling_window, jnn.c:20-50: a running FLOAT sum -- of integers
//     <= 1200 * window <= 2^24, hence exact in any order -- divided by the window), meanf / stdvf of the rolling means
//     IN SAMPLE ORDER (stat.h:17-44: order dependent, reproduced with the parity-map scan of float_order.cuh), the runs
//     of rolling means below mean - std_scale * stdv merged when closer than seg_dist (1,500), and the first run of a
//     plausible length;
//   meanf / stdvf / medianf of the adaptor's pA (cfunc.c:178-180);
//   find_polya = jnn_pa + jnn_core (jnn.c:190-279, 352-374) with JNNV1_R9_POLYA, or the caller's poly-A set, on the pA
//     behind the adaptor and the band (adaptor mean + 30) -/+ 20 (cfunc.c:189): a stretch opens at an in-band sample
//     and, while error < corrector, closes at the (error+1)-th out-of-band sample after it (31st for the reference's
//     set: the corrector never acts, see prefix_polya_exact); only the first segment is wanted, extended while the
//     following ones start within seg_dist (200) samples of the last end;
//   the same three statistics of the poly-A stretch (cfunc.c:202-204).
//
// prefix_walk_kernel (the reference's sets) / prefix_set_walk_kernel (a caller's set): one WARP per read (everything
// above except the medians); prefix_median_kernel: one CTA per read, two radix selections on sub-ranges of the int16
// samples (the pA map is monotone in raw).
#include "float_order.cuh"
#include "kernels.cuh"

namespace sgpu {

namespace {

constexpr int PW = 2000;          // jnnv2 window
constexpr int P_MERGE = 1500;     // seg_dist
constexpr int P_HI = 200000;      // hi_thresh
constexpr int A_WINDOW = 250;     // JNNV1_R9_POLYA: window (stall_len 1.0: the same bound for the first segment)
constexpr int A_TOLERATED = 30;   // error
constexpr int A_MERGE = 200;      // seg_dist
constexpr int A_CORRECTOR = 50;   // corrector

__device__ __forceinline__ int clamp_raw(int v) { return min(max(v, 0), 1200); }   // rm_outlier, jnn.c:58-75
__device__ __forceinline__ uint32_t clamp2(uint32_t two) {                          // the same on two packed int16
    return __vmins2(__vmaxs2(two, 0u), 1200u * 0x10001u);
}
static_assert(PW % 8 == 0, "the two ranges of a window difference are loaded with the same alignment");

// mean and standard deviation (float, sample order) of the pA of raw[a .. a + len)
__device__ void range_moments(const int16_t* __restrict__ raw, int a, int len, float off, float unit, float* add,
                              int lane, float* mean_out, float* stdv_out) {
    const float nf = (float)len;
    float mean = 0.0f;
    for (int pass = 0; pass < 2; pass++) {
        float acc = 0.0f;
        for (int t0 = 0; t0 < len; t0 += SB) {
            __syncwarp();
#pragma unroll 4
            for (int q = 0; q < 32; q++) {       // tile q, column lane: sample t0 + 32 q + lane (coalesced)
                const int i = t0 + q * 32 + lane;
                float v = 0.0f;
                if (i < len) {
                    v = pa_of(__ldg(raw + a + i), off, unit);
                    if (pass) { const float d = __fsub_rn(v, mean); v = __fmul_rn(d, d); }
                }
                add[q * SB_STRIDE + lane] = v;
            }
            __syncwarp();
            acc = chain_superblock(add, (min(SB, len - t0) + 31) >> 5, acc, lane, t0 == 0);
        }
        if (pass == 0) { mean = __fdiv_rn(acc, nf); *mean_out = mean; }
        else *stdv_out = __fsqrt_rn(__fdiv_rn(acc, nf));
    }
}

struct RunState {   // jnnv2's scan over the rolling means (jnn.c:125-153) and its pick (jnn.c:155-167)
    int begin, start, end;
    int have, lx, ly;      // the last segment (still open to merging)
    int chosen, cx, cy;
};
__device__ __forceinline__ bool plausible(int a, int b, int lo, int hi) { return !(b - a > hi) && !(b - a < lo); }
__device__ __forceinline__ void close_run(RunState& s, int lo, int merge, int hi) {
    if (s.have && s.start - s.ly < merge) {
        s.ly = s.end;
    } else {
        if (s.have && !s.chosen && plausible(s.lx, s.ly, lo, hi)) { s.chosen = 1; s.cx = s.lx; s.cy = s.ly; }
        s.lx = s.start; s.ly = s.end; s.have = 1;
    }
    s.start = 0; s.end = 0; s.begin = 0;
}

// ---- poly-A of a set with error >= corrector: the reference's counters, sample by sample --------------------------------
// jnn_core (jnn.c:192-245) keeps c (samples of the open stretch, tolerated outliers included), w (the corrector:
// `corrector` + every in-band sample of the record so far, never reset), err (tolerated outliers, < error) and prev_err
// (outliers at the very end of the stretch), and decrements err when c >= window, c >= w and c % w == 0. That never
// happens when error < corrector: while err has never been decremented, err <= error, so c = in-band samples of the
// stretch + err < corrector + in-band samples <= w (w counted from the start of find_polya's record, the pA behind the
// adaptor). The automaton route rests on that; the sets where it does not hold step the counters here, on the in-band
// bits `in` of the m samples from t0 (uniform across the warp). A closed gap (no counter changes on an out-of-band
// sample there) and an in-band run during which c < w (c and w both grow by one per in-band sample, so c >= w stays
// false) are crossed in one step. w is kept in 64 bits; where c % w is taken, 1 <= w <= c < 2^31 (the stretch holds an
// in-band sample and corrector >= 0).
__device__ __forceinline__ void prefix_polya_exact(uint32_t in, int m, int t0, int window,
                                                   float first_min, int error, int merge, int& open, int& first,
                                                   int& c, int& err, int& prev_err, long long& w, int& n_seg,
                                                   int& sx0, int& sy0, int& last_y) {
    int j = 0;
    while (j < m && n_seg < 2) {
        if (!open) {
            const uint32_t rest = in >> j;
            if (rest == 0u) break;
            j += __ffs(rest) - 1;
            open = 1; first = t0 + j; c = 0; err = 0; prev_err = 0;
        }
        if ((in >> j) & 1u) {                          // in band: c++, w++, prev_err = 0, then the corrector
            const uint32_t outs = ~(in >> j);          // (zero only for a word all in band, j = 0)
            const int run = min(outs ? __ffs(outs) - 1 : 32, m - j);
            prev_err = 0;
            if ((long long)c < w) {
                c += run; w += run;
            } else {
                for (int e = 0; e < run; e++) {
                    c++; w++;
                    if (c >= window && (long long)c >= w && c % (int)w == 0) err--;
                }
            }
            j += run;
        } else if (err < error) {                      // a tolerated outlier
            c++; err++; prev_err++;
            if (c >= window && (long long)c >= w && c % (int)w == 0) err--;
            j++;
        } else {                                       // the stretch closes at sample t0 + j (jnn.c:230-245)
            if (c >= window || (n_seg == 0 && (float)c >= first_min)) {
                const int stop = t0 + j - prev_err;
                if (n_seg && first - last_y < merge) { if (n_seg == 1) sy0 = stop; }
                else { if (n_seg == 0) { sx0 = first; sy0 = stop; } n_seg++; }
                last_y = stop;
            }
            open = 0; c = 0; err = 0; prev_err = 0;
            j++;
        }
    }
}

}  // namespace

// pos4[r] = {adaptor x, adaptor y, poly-A x, poly-A y} as jnnv2 / find_polya return them (poly-A relative to the
// adaptor's end; (0,0): no adaptor, (-1,-1): record not longer than the window / no poly-A / DNA);
// st6[r] = mean, stdv of the adaptor's pA, [2] unused here (median: prefix_median_kernel), the same for the poly-A.
//
// ROUTE: PREFIX_REF, the reference's window 2000, merge distance 1500, longest run 200000 and JNNV1_R9_POLYA as
// constants (P gives std_scale and lo_thresh only); or the caller's set (sgpu_set_prefix) in P, with the poly-A found by
// the automaton (PREFIX_AUTOMATON: error < corrector) or by the reference's counters stepped per sample (PREFIX_EXACT).
enum { PREFIX_REF = 0, PREFIX_AUTOMATON = 1, PREFIX_EXACT = 2 };

template <int ROUTE>
__device__ __forceinline__ void prefix_walk(const DevBatch& b, const PrefixParams& P, int32_t* __restrict__ pos4,
                                            float* __restrict__ st6) {
    constexpr bool REF = ROUTE == PREFIX_REF;
    const int aw = REF ? PW : P.a_window;              // every set has 2 <= aw <= 13981: 1200 * aw <= 2^24
    const float std_scale = P.a_std_scale;
    const int lo_thresh = P.a_lo;
    __shared__ float add_all[4][32 * SB_STRIDE];
    float* add = add_all[threadIdx.x >> 5];
    int* dbuf = reinterpret_cast<int*>(add);
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t r = warp; r < b.n_reads; r += n_warps) {
        const int16_t* __restrict__ raw = b.samples + b.read_off[r];
        const int n = (int)b.read_len[r];
        const float off = b.offset[r], unit = b.unit[r];
        int ax = -1, ay = -1, px = -1, py = -1;
        float st[6] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
        if (n > aw) {
            const int nt = n - aw;
            const float ntf = (float)nt;
            // the first window's sum (exact integer)
            int s_first = 0;
            for (int w = lane; w < aw / 8; w += 32) {   // 128-bit loads (a read starts 16-byte aligned)
                const uint4 q = __ldg(reinterpret_cast<const uint4*>(raw) + w);
                const uint32_t c4[4] = {clamp2(q.x), clamp2(q.y), clamp2(q.z), clamp2(q.w)};
#pragma unroll
                for (int h = 0; h < 4; h++) s_first += (int)(c4[h] & 0xffffu) + (int)(c4[h] >> 16);
            }
            if (!REF)   // the last aw % 8 samples of the window
                for (int i = (aw & ~7) + lane; i < aw; i += 32) s_first += clamp_raw(__ldg(raw + i));
            for (int o = 16; o; o >>= 1) s_first += __shfl_xor_sync(0xffffffffu, s_first, o);
            float mn = 0.0f, floor_ = 0.0f;
            RunState rs = {0, 0, 0, 0, 0, 0, 0, 0, 0};
            for (int pass = 0; pass < 3 && !rs.chosen; pass++) {
                float acc = 0.0f;
                int s_base = s_first;
                for (int t0 = 0; t0 < nt; t0 += SB) {
                    __syncwarp();
                    // d[i] = c[i + aw] - c[i]: the window sum moves by d[i] from position i to i + 1.
                    // Lane L takes the 128-bit words q * 32 + L of both ranges (eight loads in flight per lane), two
                    // samples per clamp / subtraction. With the reference's window (a multiple of 8) both ranges are
                    // aligned alike; with a set's, the upper range starts aw % 8 samples into an aligned word, and its
                    // 8 samples are that word and the next one shifted down by aw % 8 samples (the next word is loaded
                    // only when it is part of the read: the read is padded to 8 samples, not beyond)
                    {
                        const uint4* __restrict__ lo = reinterpret_cast<const uint4*>(raw + t0);
                        const uint4* __restrict__ hi = reinterpret_cast<const uint4*>(raw + t0 + (aw & ~7));
                        const int rot = aw & 7;
                        uint4 a[4], c[4], c_next[4];
#pragma unroll
                        for (int q = 0; q < 4; q++) {
                            const int wq = q * 32 + lane;
                            const bool in = t0 + wq * 8 < nt;   // (the word's first position; the read is padded to 8 samples)
                            a[q] = in ? __ldg(lo + wq) : make_uint4(0, 0, 0, 0);
                            c[q] = in ? __ldg(hi + wq) : make_uint4(0, 0, 0, 0);
                            if (!REF)
                                c_next[q] = in && rot && t0 + (aw & ~7) + (wq + 1) * 8 < n ? __ldg(hi + wq + 1)
                                                                                          : make_uint4(0, 0, 0, 0);
                        }
#pragma unroll
                        for (int q = 0; q < 4; q++) {
                            uint32_t av[4] = {a[q].x, a[q].y, a[q].z, a[q].w}, cv[4] = {c[q].x, c[q].y, c[q].z, c[q].w};
                            if (!REF) {   // shift the 16 samples of the two words down by rot: 32-bit steps, then 16 bits
                                const uint32_t u[8] = {c[q].x, c[q].y, c[q].z, c[q].w,
                                                       c_next[q].x, c_next[q].y, c_next[q].z, c_next[q].w};
                                uint32_t t2[6], t1[5];
#pragma unroll
                                for (int h = 0; h < 6; h++) t2[h] = (rot & 4) ? u[h + 2] : u[h];
#pragma unroll
                                for (int h = 0; h < 5; h++) t1[h] = (rot & 2) ? t2[h + 1] : t2[h];
#pragma unroll
                                for (int h = 0; h < 4; h++) cv[h] = __funnelshift_r(t1[h], t1[h + 1], (rot & 1) * 16);
                            }
#pragma unroll
                            for (int h = 0; h < 4; h++) {
                                const uint32_t d2 = __vsub2(clamp2(cv[h]), clamp2(av[h]));   // two differences in [-1200, 1200]
                                const int j = q * 256 + lane * 8 + 2 * h;                     // position in the superblock
                                const int i = t0 + j;
                                const int d0 = (int)(int16_t)(d2 & 0xffffu), d1 = (int)d2 >> 16;
                                dbuf[(j >> 5) * SB_STRIDE + (j & 31)] = i < nt ? d0 : 0;
                                dbuf[(j >> 5) * SB_STRIDE + (j & 31) + 1] = i + 1 < nt ? d1 : 0;
                            }
                        }
                    }
                    __syncwarp();
                    // lane L owns tile L: its 32 consecutive positions
                    int* row = dbuf + lane * SB_STRIDE;
                    int rowsum = 0;
#pragma unroll 8
                    for (int k = 0; k < 32; k++) rowsum += row[k];
                    int incl = rowsum;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int t = __shfl_up_sync(0xffffffffu, incl, o);
                        if (lane >= o) incl += t;
                    }
                    int s = s_base + incl - rowsum;
                    uint32_t below = 0u, above = 0u;
#pragma unroll 8
                    for (int k = 0; k < 32; k++) {
                        const int i = t0 + lane * 32 + k;
                        const int d = row[k];
                        float v = 0.0f;
                        if (i < nt) {
                            // rolling_window, jnn.c:41,46: (float)s / window. The reference's window: by the reciprocal
                            // and one residual correction (equal to the IEEE quotient for every integer s <= 2^24:
                            // oracle/proofs/div_window_check.c); a set's window: the IEEE division itself
                            const float sf = (float)s;
                            float t;
                            if (REF) {
                                const float q0 = __fmul_rn(sf, 1.0f / (float)PW);
                                t = __fmaf_rn(__fmaf_rn(-(float)PW, q0, sf), 1.0f / (float)PW, q0);
                            } else {
                                t = __fdiv_rn(sf, (float)aw);
                            }
                            if (pass == 0) v = t;
                            else if (pass == 1) { const float dv = __fsub_rn(t, mn); v = __fmul_rn(dv, dv); }
                            else { below |= (t < floor_ ? 1u : 0u) << k; above |= (t > floor_ ? 1u : 0u) << k; }
                        }
                        reinterpret_cast<float*>(row)[k] = v;
                        s += d;
                    }
                    s_base += __shfl_sync(0xffffffffu, incl, 31);
                    __syncwarp();
                    const int ntiles = (min(SB, nt - t0) + 31) >> 5;
                    if (pass < 2) {
                        acc = chain_superblock(add, ntiles, acc, lane, t0 == 0);
                    } else {
                        // the run logic, every lane the same (uniform): tile after tile, transition after transition
                        for (int tl = 0; tl < ntiles && !rs.chosen; tl++) {
                            const uint32_t bm = __shfl_sync(0xffffffffu, below, tl), am = __shfl_sync(0xffffffffu, above, tl);
                            const int p0 = t0 + tl * 32;
                            int cur = 0;
                            while (cur < 32) {
                                const uint32_t rest = 0xffffffffu << cur;
                                if (!rs.begin) {
                                    const uint32_t m = bm & rest;
                                    if (!m) break;
                                    const int k = __ffs(m) - 1;
                                    rs.start = p0 + k; rs.begin = 1;
                                    cur = k + 1;
                                } else {
                                    const uint32_t ma = am & rest;
                                    const int ka = ma ? __ffs(ma) - 1 : 32;
                                    const uint32_t mb = bm & rest & (ka < 32 ? ((1u << ka) - 1u) : 0xffffffffu);
                                    if (mb) rs.end = p0 + 31 - __clz(mb);
                                    if (ka == 32) break;
                                    if (REF) close_run(rs, lo_thresh, P_MERGE, P_HI);
                                    else close_run(rs, lo_thresh, P.a_seg_dist, P.a_hi);
                                    cur = ka + 1;
                                }
                            }
                        }
                    }
                }
                if (pass == 0) mn = __fdiv_rn(acc, ntf);
                else if (pass == 1) floor_ = __fsub_rn(mn, __fmul_rn(__fsqrt_rn(__fdiv_rn(acc, ntf)), std_scale));
            }
            const int a_hi = REF ? P_HI : P.a_hi;
            if (!rs.chosen && rs.have && plausible(rs.lx, rs.ly, lo_thresh, a_hi)) { rs.chosen = 1; rs.cx = rs.lx; rs.cy = rs.ly; }
            ax = 0; ay = 0;
            if (rs.chosen) { ax = rs.cx + aw / 2 - 1; ay = rs.cy + aw / 2 - 1; }
            if (ay > 0) {
                range_moments(raw, ax, ay - ax, off, unit, add, lane, &st[0], &st[1]);
                if (b.rna) {
                    // ---- poly-A: the counter machine of jnn_core over one bit per sample (in the band or not) ----
                    const float top = __fadd_rn(__fadd_rn(st[0], 30.0f), 20.0f), bot = __fsub_rn(__fadd_rn(st[0], 30.0f), 20.0f);
                    const int m = n - ay;
                    const int tolerated = REF ? A_TOLERATED : P.p_error, merge = REF ? A_MERGE : P.p_seg_dist;
                    const int window = REF ? A_WINDOW : P.p_window;
                    const float first_min = REF ? (float)A_WINDOW : __fmul_rn((float)P.p_window, P.p_stall_len);
                    // automaton: open, first, bad, tail; exact: open, first, c, bad (err), tail (prev_err), w
                    int open = 0, first = 0, bad = 0, tail = 0, n_seg = 0, sx0 = 0, sy0 = 0, last_y = 0, c = 0;
                    long long w = REF ? 0 : P.p_corrector;
                    for (int t0 = 0; t0 < m && n_seg < 2; t0 += 32) {
                        const int i = t0 + lane;
                        bool in = false;
                        if (i < m) {
                            float v = pa_of(__ldg(raw + ay + i), off, unit);
                            v = v > 1200.0f ? 1200.0f : v < 0.0f ? 0.0f : v;   // rm_outlierf, jnn.c:79-95
                            in = v < top && v > bot;
                        }
                        const uint32_t wd = __ballot_sync(0xffffffffu, in);
                        const uint32_t valid = m - t0 >= 32 ? 0xffffffffu : ((1u << (m - t0)) - 1u);
                        if (ROUTE == PREFIX_EXACT) {
                            prefix_polya_exact(wd, min(32, m - t0), t0, window, first_min, tolerated, merge,
                                               open, first, c, bad, tail, w, n_seg, sx0, sy0, last_y);
                            continue;
                        }
                        int cur = 0;
                        while (cur < 32 && ((valid >> cur) & 1u) && n_seg < 2) {
                            const uint32_t rest = (0xffffffffu << cur) & valid;
                            if (!open) {
                                const uint32_t mi = wd & rest;
                                if (!mi) break;
                                const int k = __ffs(mi) - 1;
                                open = 1; first = t0 + k; bad = 0; tail = 0;
                                cur = k + 1;
                            } else {
                                const uint32_t z = ~wd & rest;                 // out-of-band samples from cur on
                                const int nz = __popc(z);
                                // the stretch survives this word (written so that error = INT32_MAX cannot overflow)
                                if (REF ? bad + nz <= tolerated : nz <= tolerated - bad) {
                                    bad += nz;
                                    const uint32_t ones = wd & rest;
                                    const int hi = 31 - __clz(valid);          // last valid bit
                                    tail = ones ? hi - (31 - __clz(ones)) : tail + (hi + 1 - cur);
                                    break;
                                }
                                // the (error + 1)-th outlier of the stretch (tolerated - bad < nz <= 32 here)
                                const int k = (int)__fns(z, 0u, tolerated - bad + 1);
                                const uint32_t before = wd & rest & ((1u << k) - 1u);     // in-band samples in [cur, k)
                                const int tl = before ? k - 1 - (31 - __clz(before)) : tail + (k - cur);
                                const int iclose = t0 + k;
                                const int run = iclose - first;                // every sample of the stretch
                                // jnn.c:232: run >= window, or the first segment's fl(window * stall_len) (the
                                // reference's set: both 250)
                                if (REF ? run >= window : run >= window || (n_seg == 0 && (float)run >= first_min)) {
                                    const int stop = iclose - tl;
                                    if (n_seg && first - last_y < merge) { if (n_seg == 1) sy0 = stop; }
                                    else { if (n_seg == 0) { sx0 = first; sy0 = stop; } n_seg++; }
                                    last_y = stop;
                                }
                                open = 0; bad = 0; tail = 0;
                                cur = k + 1;
                            }
                        }
                    }
                    if (n_seg > 0) { px = sx0; py = sy0; }
                    if (py > 0) range_moments(raw, ay + px, py - px, off, unit, add, lane, &st[3], &st[4]);
                }
            }
        }
        if (lane == 0) {
            int32_t* p = pos4 + (size_t)r * 4;
            p[0] = ax; p[1] = ay; p[2] = px; p[3] = py;
            float* o = st6 + (size_t)r * 6;
            o[0] = st[0]; o[1] = st[1]; o[3] = st[3]; o[4] = st[4];
        }
    }
}

// the reference's adaptor sets (JNNV2_RNA_R9_ADAPTOR / JNNV2_RNA_RNA004_ADAPTOR differ in std_scale and lo_thresh only)
// with JNNV1_R9_POLYA
__global__ void __launch_bounds__(128, 4) prefix_walk_kernel(DevBatch b, float std_scale, int lo_thresh,
                                                            int32_t* __restrict__ pos4, float* __restrict__ st6) {
    PrefixParams P;
    P.a_std_scale = std_scale;
    P.a_lo = lo_thresh;
    prefix_walk<PREFIX_REF>(b, P, pos4, st6);
}

// the caller's set (sgpu_set_prefix); ROUTE: PREFIX_AUTOMATON or PREFIX_EXACT
template <int ROUTE>
__global__ void __launch_bounds__(128, 4) prefix_set_walk_kernel(DevBatch b, const PrefixParams P,
                                                                int32_t* __restrict__ pos4, float* __restrict__ st6) {
    prefix_walk<ROUTE>(b, P, pos4, st6);
}

// medianf of the two stretches: the sample of rank len/2 (stat.h:56-64, ks_ksmall) among the raw values of the
// stretch, mapped to pA (monotone in raw; rank from the other end for a negative unit)
__global__ void __launch_bounds__(256) prefix_median_kernel(DevBatch b, const int32_t* __restrict__ pos4,
                                                            float* __restrict__ st6) {
    __shared__ uint32_t hist[MED_BINS];
    __shared__ uint32_t part[256];
    __shared__ uint32_t sh[4];
    for (uint32_t r = blockIdx.x; r < b.n_reads; r += gridDim.x) {
        const int16_t* __restrict__ raw = b.samples + b.read_off[r];
        const int32_t* p = pos4 + (size_t)r * 4;
        const int ax = p[0], ay = p[1], px = p[2], py = p[3];
        const float off = b.offset[r], unit = b.unit[r];
        float med[2] = {0.0f, 0.0f};
        for (int k = 0; k < 2; k++) {
            const int a = k ? ay + px : ax, len = k ? py - px : ay - ax;
            const bool have = k ? (ay > 0 && py > 0) : ay > 0;   // (uniform across the CTA)
            if (!have || len <= 0) continue;
            uint32_t rank = (uint32_t)(len / 2);
            if (unit < 0.0f) rank = (uint32_t)len - 1u - rank;
            const int v = select_rank_i16<false>(raw + a, (uint32_t)len, rank, hist, part, sh);
            med[k] = pa_of((int16_t)v, off, unit);
        }
        if (threadIdx.x == 0) { st6[(size_t)r * 6 + 2] = med[0]; st6[(size_t)r * 6 + 5] = med[1]; }
    }
}

int launch_prefix(const DevBatch& b, const PrefixParams& p, int32_t* pos4, float* st6, int sm_count, cudaStream_t st) {
    if (b.n_reads == 0) return 0;
    int g1 = (int)((b.n_reads + 3) / 4);  // one warp per read
    if (g1 > sm_count * 16) g1 = sm_count * 16;
    // the reference's window, merge distance, longest run and poly-A set (JNNV2_RNA_R9_ADAPTOR and
    // JNNV2_RNA_RNA004_ADAPTOR, given or not, among them) take the kernel with these as constants
    if (p.a_window == PW && p.a_seg_dist == P_MERGE && p.a_hi == P_HI && p.p_window == A_WINDOW &&
        p.p_stall_len == 1.0f && p.p_error == A_TOLERATED && p.p_seg_dist == A_MERGE && p.p_corrector == A_CORRECTOR)
        prefix_walk_kernel<<<g1, 128, 0, st>>>(b, p.a_std_scale, p.a_lo, pos4, st6);
    else if (p.p_error < p.p_corrector)
        prefix_set_walk_kernel<PREFIX_AUTOMATON><<<g1, 128, 0, st>>>(b, p, pos4, st6);
    else
        prefix_set_walk_kernel<PREFIX_EXACT><<<g1, 128, 0, st>>>(b, p, pos4, st6);
    int g2 = (int)b.n_reads;
    if (g2 > sm_count * 8) g2 = sm_count * 8;
    prefix_median_kernel<<<g2, 256, 0, st>>>(b, pos4, st6);
    return 2;
}

}  // namespace sgpu
