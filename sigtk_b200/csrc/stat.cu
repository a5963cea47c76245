// stat.cu -- the per-read statistics of `sigtk stat` (reference src/cfunc.c:126-159, src/stat.h:17-73).
//
// The reference accumulates in FLOAT, sequentially: the result depends on the
// summation order (SURVEY 8(a) a11), so a tree reduction cannot be bit-exact.
// stat_moments_kernel therefore reproduces the float recurrence exactly ("exact
// emulation"), one warp per read: runs of 32 values are summarised in parallel by
// what they do to the accumulator for either parity of its last bit (see below).  Medians are order-free: a two-level
// radix selection on the int16 samples, one CTA per read; pa_median follows
// from raw_median because the pA map is monotone in raw.
#include "kernels.cuh"
#include "float_order.cuh"

namespace sgpu {

// One WARP per read (reads shorter than `cta_min` samples); per pass and superblock of 1024 samples all lanes load
// the samples (coalesced) and compute the addends -- (float)raw and pA in the first pass (meani16 / meanf:
// sum += x[i]), the squared deviations in the second (stdvi16 / stdvf: sum += (x[i]-m)*(x[i]-m)) -- into shared
// memory; chain_superblock adds them up in the reference's order. Positions past the end of the read hold +0, which
// no float sum notices.
// JNN = true: ONE channel, the samples clamped to [0, 1200] (rm_outlier, jnn.c:58-75), i.e. meanf / stdvf of the
// signal jnn_core thresholds (jnn.c:181-185); out = [n_reads][2] (mean, stdv).

// the addends of one superblock (samples t0 .. t0+1023 of the read, 4 x 128-bit words per lane: lane L holds the
// words q*32 + L) into the warp's shared rows: tile j/32, column j%32
template <bool JNN, bool FULL, int PASS>
__device__ __forceinline__ void fill_addends_(const uint4 (&cur)[4], int t0, int n, int lane, int pass, float mean_r,
                                              float mean_p, float off, float unit, float (*add)[32 * SB_STRIDE]) {
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const uint32_t wd[4] = {cur[q].x, cur[q].y, cur[q].z, cur[q].w};
#pragma unroll
        for (int h = 0; h < 8; h++) {
            const int j = q * 256 + lane * 8 + h;
            const int i = t0 + j;
            float ar = 0.0f, ap = 0.0f;
            if (FULL || i < n) {
                const int16_t v = (int16_t)(wd[h >> 1] >> ((h & 1) * 16));
                if (JNN) {
                    ar = (float)min(max((int)v, 0), 1200);
                } else {
                    ar = (float)v;
                    ap = pa_of(v, off, unit);
                }
                if (PASS) {
                    const float dr = __fsub_rn(ar, mean_r), dp = __fsub_rn(ap, mean_p);
                    ar = __fmul_rn(dr, dr);
                    ap = __fmul_rn(dp, dp);
                }
            }
            const int at = (j >> 5) * SB_STRIDE + (j & 31);
            add[0][at] = ar;
            if (!JNN) add[JNN ? 0 : 1][at] = ap;
        }
    }
}

template <bool JNN>
__device__ __forceinline__ void fill_addends(const uint4 (&cur)[4], int t0, int n, int lane, int pass, float mean_r,
                                             float mean_p, float off, float unit, float (*add)[32 * SB_STRIDE]) {
    if (t0 + SB <= n) {  // (no per-sample bound)
        if (pass) fill_addends_<JNN, true, 1>(cur, t0, n, lane, pass, mean_r, mean_p, off, unit, add);
        else fill_addends_<JNN, true, 0>(cur, t0, n, lane, pass, mean_r, mean_p, off, unit, add);
    } else {
        if (pass) fill_addends_<JNN, false, 1>(cur, t0, n, lane, pass, mean_r, mean_p, off, unit, add);
        else fill_addends_<JNN, false, 0>(cur, t0, n, lane, pass, mean_r, mean_p, off, unit, add);
    }
}

template <bool JNN>
__device__ __forceinline__ void store_moments(float* __restrict__ out, uint32_t r, int pass, float acc_r, float acc_p,
                                              float nf, float& mean_r, float& mean_p, bool writer) {
    if (pass == 0) {
        mean_r = __fdiv_rn(acc_r, nf);
        mean_p = __fdiv_rn(acc_p, nf);
        if (writer) {
            if (JNN) out[(size_t)r * 2] = mean_r;
            else { out[(size_t)r * 6] = mean_r; out[(size_t)r * 6 + 1] = mean_p; }
        }
    } else if (writer) {
        if (JNN) out[(size_t)r * 2 + 1] = __fsqrt_rn(__fdiv_rn(acc_r, nf));
        else {
            out[(size_t)r * 6 + 2] = __fsqrt_rn(__fdiv_rn(acc_r, nf));
            out[(size_t)r * 6 + 3] = __fsqrt_rn(__fdiv_rn(acc_p, nf));
        }
    }
}

constexpr int CW = 8;    // warps per CTA
constexpr size_t moments_smem(bool jnn) { return (size_t)CW * (jnn ? 1 : 2) * 32 * SB_STRIDE * sizeof(float); }

// ---- role 1: one WARP per read ------------------------------------------------------------------------------------
template <bool JNN>
__device__ __forceinline__ void moments_by_warp(const DevBatch& b, float* __restrict__ out, uint32_t cta_min,
                                                float (*add)[32 * SB_STRIDE], uint32_t warp, uint32_t n_warps, int lane) {
    for (uint32_t r = warp; r < b.n_reads; r += n_warps) {
        if (b.read_len[r] >= cta_min) continue;  // the CTA role's
        const int16_t* __restrict__ raw = b.samples + b.read_off[r];
        const int n = (int)b.read_len[r];  // stat.h takes `int n`
        const float off = JNN ? 0.0f : b.offset[r], unit = JNN ? 0.0f : b.unit[r];
        const float nf = (float)n;
        float mean_r = 0.0f, mean_p = 0.0f;
        // 128-bit loads: lane L takes the words q*32 + L of a superblock (4 per lane, 512 contiguous bytes per
        // instruction); the next superblock's are in flight while this one is added up
        const uint4* __restrict__ src = reinterpret_cast<const uint4*>(raw);
        const int n_words = (n + 7) >> 3;
        uint4 cur[4], nxt[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int w = q * 32 + lane;
            cur[q] = w < n_words ? __ldg(src + w) : make_uint4(0, 0, 0, 0);
        }
        for (int pass = 0; pass < 2; pass++) {
            float acc_r = 0.0f, acc_p = 0.0f;
            for (int t0 = 0; t0 < n; t0 += SB) {
                __syncwarp();  // the previous superblock's readers are done
                {
                    const int tn = t0 + SB < n ? t0 + SB : 0;  // after the last superblock: the first one again (pass 2)
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        const int w = (tn >> 3) + q * 32 + lane;
                        nxt[q] = w < n_words ? __ldg(src + w) : make_uint4(0, 0, 0, 0);
                    }
                }
                fill_addends<JNN>(cur, t0, n, lane, pass, mean_r, mean_p, off, unit, add);
#pragma unroll
                for (int q = 0; q < 4; q++) cur[q] = nxt[q];
                __syncwarp();
                const int ntiles = (min(SB, n - t0) + 31) >> 5;
                acc_r = chain_superblock(add[0], ntiles, acc_r, lane, t0 == 0);
                if (!JNN) acc_p = chain_superblock(add[JNN ? 0 : 1], ntiles, acc_p, lane, t0 == 0);
            }
            store_moments<JNN>(out, r, pass, acc_r, acc_p, nf, mean_r, mean_p, lane == 0);
        }
    }
}

// ---- role 2: one CTA of CW warps per read of at least `cta_min` samples ---------------------------------------------
// (a 2,000,000-sample read is 1,954 superblocks: one warp would walk them one after the other.) The warps take CW
// consecutive superblocks per round. Every warp summarises its superblock in the binade the accumulator has at the
// start of the round (summarise_superblock: what the superblock adds for an even and an odd incoming mantissa), every
// thread composes the CW summaries in order, and the first superblock that cannot be summarised or would carry the
// accumulator out of the binade is added up by its own warp from the accumulator it now knows (chain_superblock);
// the warps after it summarise again in the new binade. The accumulator leaves a binade ~log2 times per read, so
// nearly every round is one summarise + one barrier + one compose. Bit-identical to the sequential loop for the same
// reason the one-warp role is.
template <bool JNN>
__device__ __forceinline__ void moments_by_cta(const DevBatch& b, float* __restrict__ out, uint32_t cta_min,
                                               float (*add)[32 * SB_STRIDE], uint32_t cta, uint32_t n_ctas, int lane, int warp) {
    constexpr int CH = JNN ? 1 : 2;
    __shared__ uint32_t sum_u[2][CH][CW][2];         // [round parity][channel][warp][parity of the incoming mantissa]
    __shared__ uint32_t sum_ok[2][CH][CW];
    __shared__ float s_bcast[CH];
    for (uint32_t r = cta; r < b.n_reads; r += n_ctas) {
        if (b.read_len[r] < cta_min) continue;       // (the same for every thread of the CTA)
        const int16_t* __restrict__ raw = b.samples + b.read_off[r];
        const int n = (int)b.read_len[r];
        const float off = JNN ? 0.0f : b.offset[r], unit = JNN ? 0.0f : b.unit[r];
        const float nf = (float)n;
        const uint4* __restrict__ src = reinterpret_cast<const uint4*>(raw);
        const int n_words = (n + 7) >> 3;
        float mean_r = 0.0f, mean_p = 0.0f;
        uint4 cur[4], nxt[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int w = ((warp * SB) >> 3) + q * 32 + lane;
            cur[q] = w < n_words ? __ldg(src + w) : make_uint4(0, 0, 0, 0);
        }
        int rp = 0;
        __syncthreads();                             // the previous read's last summaries have been read
        for (int pass = 0; pass < 2; pass++) {
            float acc[2] = {0.0f, 0.0f};             // (every thread holds the same values)
            for (int round0 = 0; round0 < n; round0 += CW * SB, rp ^= 1) {
                const int t0 = round0 + warp * SB;
                const int ntiles = t0 < n ? (min(SB, n - t0) + 31) >> 5 : 0;
                const int active = min(CW, (n - round0 + SB - 1) / SB);
                {   // the next round's samples (after the last round: the first one again, for pass 2)
                    const int tn = (round0 + CW * SB < n ? round0 + CW * SB : 0) + warp * SB;
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        const int w = (tn >> 3) + q * 32 + lane;
                        nxt[q] = w < n_words ? __ldg(src + w) : make_uint4(0, 0, 0, 0);
                    }
                }
                __syncwarp();                        // this warp's readers of the previous round's addends are done
                if (ntiles) fill_addends<JNN>(cur, t0, n, lane, pass, mean_r, mean_p, off, unit, add);
#pragma unroll
                for (int q = 0; q < 4; q++) cur[q] = nxt[q];
                __syncwarp();
                int start[2] = {0, CH == 2 ? 0 : active};    // first superblock of the round not yet added, per channel
                while (start[0] < active || start[1] < active) {
                    bool binade[2] = {false, false};
#pragma unroll
                    for (int ch = 0; ch < CH; ch++) {
                        if (start[ch] >= active) continue;
                        binade[ch] = summable(acc[ch]) && !(round0 == 0 && start[ch] == 0);
                        if (binade[ch] && warp >= start[ch] && warp < active) {
                            uint32_t U0, U1;
                            const bool ok = summarise_superblock(add[ch], ntiles, acc[ch], lane, U0, U1);
                            if (lane == 0) { sum_u[rp][ch][warp][0] = U0; sum_u[rp][ch][warp][1] = U1; sum_ok[rp][ch][warp] = ok ? 1u : 0u; }
                        }
                    }
                    __syncthreads();
                    int fail[2] = {active, active};
                    bool any_fail = false;
#pragma unroll
                    for (int ch = 0; ch < CH; ch++) {
                        if (start[ch] >= active) continue;
                        fail[ch] = start[ch];
                        if (binade[ch]) {
                            const uint32_t sb = __float_as_uint(acc[ch]);
                            uint32_t S = (sb & 0x7fffffu) | 0x800000u;
                            uint32_t u[CW][2], okw[CW];  // (loaded up front: the walk below is a chain of selects)
#pragma unroll
                            for (int w = 0; w < CW; w++) {
                                u[w][0] = sum_u[rp][ch][w][0]; u[w][1] = sum_u[rp][ch][w][1]; okw[w] = sum_ok[rp][ch][w];
                            }
                            bool go = true;
#pragma unroll
                            for (int w = 0; w < CW; w++) {
                                const uint32_t inc = (S & 1u) ? u[w][1] : u[w][0];
                                go = go && (w < start[ch] || (w < active && okw[w] && inc < 0x1000000u && S + inc < 0x1000000u));
                                if (go && w >= start[ch]) { S += inc; fail[ch] = w + 1; }
                            }
                            acc[ch] = __uint_as_float((sb & 0x7f800000u) | (S & 0x7fffffu));
                        }
                        if (fail[ch] < active) {     // this superblock by its own warp, from the accumulator it meets
                            any_fail = true;
                            if (warp == fail[ch]) {
                                const float s = chain_superblock(add[ch], ntiles, acc[ch], lane, round0 == 0 && fail[ch] == 0);
                                if (lane == 0) s_bcast[ch] = s;
                            }
                        }
                    }
                    if (any_fail) {
                        __syncthreads();
#pragma unroll
                        for (int ch = 0; ch < CH; ch++)
                            if (fail[ch] < active) acc[ch] = s_bcast[ch];
                    }
#pragma unroll
                    for (int ch = 0; ch < CH; ch++)
                        if (start[ch] < active) start[ch] = fail[ch] < active ? fail[ch] + 1 : active;
                }
            }
            store_moments<JNN>(out, r, pass, acc[0], acc[1], nf, mean_r, mean_p, threadIdx.x == 0);
        }
    }
}

// The first `cta_blocks` CTAs take the long reads (they start first), the others the short ones, a warp each.
template <bool JNN>
__global__ void __launch_bounds__(CW * 32, 3) stat_moments_kernel(DevBatch b, float* __restrict__ out, uint32_t cta_min,
                                                                  uint32_t cta_blocks) {
    extern __shared__ float moments_add[];           // [CW][channels][32 * SB_STRIDE]: every warp's addends of one superblock
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float (*add)[32 * SB_STRIDE] =
        reinterpret_cast<float (*)[32 * SB_STRIDE]>(moments_add + (size_t)warp * (JNN ? 1 : 2) * 32 * SB_STRIDE);
    if (blockIdx.x < cta_blocks)
        moments_by_cta<JNN>(b, out, cta_min, add, blockIdx.x, cta_blocks, lane, warp);
    else
        moments_by_warp<JNN>(b, out, cta_min, add, (blockIdx.x - cta_blocks) * CW + warp, (gridDim.x - cta_blocks) * CW, lane);
}

// reads of lo <= n < hi samples, one CTA of NT threads each (256 for most reads, 1,024 for the long ones: a
// 2,000,000-sample read is two passes over 4 MB)
template <int NT>
__global__ void __launch_bounds__(NT) stat_median_kernel(DevBatch b, float* __restrict__ out, uint32_t lo, uint32_t hi) {
    __shared__ uint32_t hist[MED_BINS];
    __shared__ uint32_t part[256];
    __shared__ uint32_t sh[4];
    for (uint32_t r = blockIdx.x; r < b.n_reads; r += gridDim.x) {
        const int16_t* __restrict__ raw = b.samples + b.read_off[r];
        const uint32_t n = b.read_len[r];
        if (n < lo || n >= hi) continue;
        if (n == 0) {  // an empty record: defined values instead of the previous batch's
            if (threadIdx.x == 0) { out[(size_t)r * 6 + 4] = 0.0f; out[(size_t)r * 6 + 5] = 0.0f; }
            continue;
        }
        const uint32_t rank = (uint32_t)((int)n / 2);  // ks_ksmall(n, copy, n/2), stat.h:60,70
        const int med_r = select_rank_i16<true>(raw, n, rank, hist, part, sh);
        const float off = b.offset[r], unit = b.unit[r];
        // pA is non-decreasing in raw for unit >= 0 and non-increasing for unit < 0
        int med_for_pa = med_r;
        if (unit < 0.0f) med_for_pa = select_rank_i16<true>(raw, n, n - 1 - rank, hist, part, sh);
        if (threadIdx.x == 0) {
            float* o = out + (size_t)r * 6;
            o[4] = (float)med_r;
            o[5] = pa_of((int16_t)med_for_pa, off, unit);
        }
    }
}

// reads of at least `cta_min` samples get a CTA each, the others a warp each: one launch
template <bool JNN>
static int launch_moments(const DevBatch& b, float* out, uint32_t cta_min, int sm_count, cudaStream_t st) {
    if (b.n_reads == 0) return 0;
    constexpr size_t smem = moments_smem(JNN);
    cudaFuncSetAttribute(stat_moments_kernel<JNN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);  // per device
    uint32_t g2 = b.n_reads < (uint32_t)sm_count * 2u ? b.n_reads : (uint32_t)sm_count * 2u;
    uint32_t g1 = (b.n_reads + CW - 1) / CW;         // one warp per read
    if (g1 > (uint32_t)sm_count * 8u) g1 = (uint32_t)sm_count * 8u;
    stat_moments_kernel<JNN><<<g2 + g1, CW * 32, smem, st>>>(b, out, cta_min, g2);
    return 1;
}

int launch_stat_moments(const DevBatch& b, float* stat6, uint32_t cta_min, int sm_count, cudaStream_t st) {
    return launch_moments<false>(b, stat6, cta_min, sm_count, st);
}

int launch_stat_median(const DevBatch& b, float* stat6, uint32_t cta_min, int sm_count, cudaStream_t st) {
    if (b.n_reads == 0) return 0;
    int g = (int)b.n_reads;
    stat_median_kernel<1024><<<g > sm_count * 2 ? sm_count * 2 : g, 1024, 0, st>>>(b, stat6, cta_min, 0xffffffffu);
    stat_median_kernel<256><<<g > sm_count * 8 ? sm_count * 8 : g, 256, 0, st>>>(b, stat6, 0u, cta_min);
    return 2;
}

// ---- the statistics of the caller's pA floats: meanf, stdvf, medianf of every record ----------------------------------
// The same two roles as stat_moments_kernel with one channel; a superblock of 1024 floats is 8 128-bit words per lane
// (lane L holds the words q*32 + L: floats q*128 + 4L .. +3). The first pass adds values of either sign
// (chain_superblock_signed / summarise_superblock_signed), the second the squared deviations, which are not negative.

// the addends of one superblock (floats t0 .. t0+1023 of the read) into the warp's shared rows; +0 past the read's end,
// whatever the padding holds
template <int PASS>
__device__ __forceinline__ void fill_pa_addends(const uint4 (&cur)[8], int t0, int n, int lane, float mean,
                                                float* __restrict__ add) {
#pragma unroll
    for (int q = 0; q < 8; q++) {
        const uint32_t wd[4] = {cur[q].x, cur[q].y, cur[q].z, cur[q].w};
#pragma unroll
        for (int h = 0; h < 4; h++) {
            const int j = q * 128 + lane * 4 + h;
            float a = 0.0f;
            if (t0 + j < n) {
                a = __uint_as_float(wd[h]);
                if (PASS) {
                    const float d = __fsub_rn(a, mean);
                    a = __fmul_rn(d, d);
                }
            }
            add[(j >> 5) * SB_STRIDE + (j & 31)] = a;
        }
    }
}

__device__ __forceinline__ void load_pa_superblock(const uint4* __restrict__ src, int t, int n_words, int lane,
                                                   uint4 (&q)[8]) {
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const int w = (t >> 2) + k * 32 + lane;
        q[k] = w < n_words ? __ldg(src + w) : make_uint4(0, 0, 0, 0);
    }
}

__device__ __forceinline__ void store_pa_moment(float* __restrict__ out, uint32_t r, int pass, float acc, float nf,
                                                float& mean, bool writer) {
    if (pass == 0) {
        mean = __fdiv_rn(acc, nf);
        if (writer) out[(size_t)r * 6 + 1] = mean;
    } else if (writer) {
        out[(size_t)r * 6 + 3] = __fsqrt_rn(__fdiv_rn(acc, nf));
    }
}

__device__ __forceinline__ void pa_moments_by_warp(const DevBatch& b, const float* __restrict__ pa,
                                                   float* __restrict__ out, uint32_t cta_min, float* __restrict__ add,
                                                   uint32_t warp, uint32_t n_warps, int lane) {
    for (uint32_t r = warp; r < b.n_reads; r += n_warps) {
        if (b.read_len[r] >= cta_min) continue;  // the CTA role's
        const uint4* __restrict__ src = reinterpret_cast<const uint4*>(pa + b.read_off[r]);
        const int n = (int)b.read_len[r];
        const int n_words = (n + 3) >> 2;
        const float nf = (float)n;
        float mean = 0.0f;
        uint4 cur[8], nxt[8];
        load_pa_superblock(src, 0, n_words, lane, cur);
        for (int pass = 0; pass < 2; pass++) {
            float acc = 0.0f;
            for (int t0 = 0; t0 < n; t0 += SB) {
                __syncwarp();  // the previous superblock's readers are done
                load_pa_superblock(src, t0 + SB < n ? t0 + SB : 0, n_words, lane, nxt);
                if (pass) fill_pa_addends<1>(cur, t0, n, lane, mean, add);
                else fill_pa_addends<0>(cur, t0, n, lane, mean, add);
#pragma unroll
                for (int q = 0; q < 8; q++) cur[q] = nxt[q];
                __syncwarp();
                const int ntiles = (min(SB, n - t0) + 31) >> 5;
                acc = pass ? chain_superblock(add, ntiles, acc, lane, t0 == 0)
                           : chain_superblock_signed(add, ntiles, acc, lane, t0 == 0);
            }
            store_pa_moment(out, r, pass, acc, nf, mean, lane == 0);
        }
    }
}

// as moments_by_cta: CW consecutive superblocks per round, summarised in the binade the accumulator has, composed in
// order by every thread; the first that cannot be composed is added up by its own warp
__device__ __forceinline__ void pa_moments_by_cta(const DevBatch& b, const float* __restrict__ pa,
                                                  float* __restrict__ out, uint32_t cta_min, float* __restrict__ add,
                                                  uint32_t cta, uint32_t n_ctas, int lane, int warp) {
    __shared__ SgnSum sum_s[2][CW];                  // [round parity][warp]: first pass
    __shared__ uint32_t sum_u[2][CW][2];             // second pass: [parity of the incoming mantissa]
    __shared__ uint32_t sum_ok[2][CW];
    __shared__ float s_bcast;
    for (uint32_t r = cta; r < b.n_reads; r += n_ctas) {
        if (b.read_len[r] < cta_min) continue;       // (the same for every thread of the CTA)
        const uint4* __restrict__ src = reinterpret_cast<const uint4*>(pa + b.read_off[r]);
        const int n = (int)b.read_len[r];
        const int n_words = (n + 3) >> 2;
        const float nf = (float)n;
        float mean = 0.0f;
        uint4 cur[8], nxt[8];
        load_pa_superblock(src, warp * SB, n_words, lane, cur);
        int rp = 0;
        __syncthreads();                             // the previous read's last summaries have been read
        for (int pass = 0; pass < 2; pass++) {
            float acc = 0.0f;                        // (every thread holds the same value)
            for (int round0 = 0; round0 < n; round0 += CW * SB, rp ^= 1) {
                const int t0 = round0 + warp * SB;
                const int ntiles = t0 < n ? (min(SB, n - t0) + 31) >> 5 : 0;
                const int active = min(CW, (n - round0 + SB - 1) / SB);
                load_pa_superblock(src, (round0 + CW * SB < n ? round0 + CW * SB : 0) + warp * SB, n_words, lane, nxt);
                __syncwarp();                        // this warp's readers of the previous round's addends are done
                if (ntiles) {
                    if (pass) fill_pa_addends<1>(cur, t0, n, lane, mean, add);
                    else fill_pa_addends<0>(cur, t0, n, lane, mean, add);
                }
#pragma unroll
                for (int q = 0; q < 8; q++) cur[q] = nxt[q];
                __syncwarp();
                int start = 0;                       // first superblock of the round not yet added
                while (start < active) {
                    const bool binade = (pass ? summable(acc) : summable_signed(acc)) && !(round0 == 0 && start == 0);
                    if (binade && warp >= start && warp < active) {
                        bool ok;
                        if (pass) {
                            uint32_t U0, U1;
                            ok = summarise_superblock(add, ntiles, acc, lane, U0, U1);
                            if (lane == 0) { sum_u[rp][warp][0] = U0; sum_u[rp][warp][1] = U1; }
                        } else {
                            SgnSum U;
                            ok = summarise_superblock_signed(add, ntiles, acc, lane, U);
                            if (lane == 0) sum_s[rp][warp] = U;
                        }
                        if (lane == 0) sum_ok[rp][warp] = ok ? 1u : 0u;
                    }
                    __syncthreads();
                    int fail = start;
                    if (binade) {
                        const uint32_t sb = __float_as_uint(acc);
                        uint32_t S = (sb & 0x7fffffu) | 0x800000u;
                        bool go = true;
                        for (int w = start; w < active && go; w++) {
                            uint32_t inc;
                            if (pass) {
                                inc = sum_u[rp][w][S & 1u];
                                go = sum_ok[rp][w] && inc < 0x1000000u && S + inc < 0x1000000u;
                            } else {
                                const SgnSum& u = sum_s[rp][w];
                                inc = (uint32_t)u.inc[S & 1u];
                                go = sum_ok[rp][w] && sgn_fits(u, S);
                            }
                            if (go) { S += inc; fail = w + 1; }
                        }
                        acc = __uint_as_float((sb & 0xff800000u) | (S & 0x7fffffu));
                    }
                    if (fail < active) {             // this superblock by its own warp, from the accumulator it meets
                        if (warp == fail) {
                            const bool first = round0 == 0 && fail == 0;
                            const float s = pass ? chain_superblock(add, ntiles, acc, lane, first)
                                                 : chain_superblock_signed(add, ntiles, acc, lane, first);
                            if (lane == 0) s_bcast = s;
                        }
                        __syncthreads();
                        acc = s_bcast;
                        start = fail + 1;
                    } else {
                        start = active;
                    }
                }
            }
            store_pa_moment(out, r, pass, acc, nf, mean, threadIdx.x == 0);
        }
    }
}

__global__ void __launch_bounds__(CW * 32, 2) stat_pa_moments_kernel(DevBatch b, const float* __restrict__ pa,
                                                                     float* __restrict__ out, uint32_t cta_min,
                                                                     uint32_t cta_blocks) {
    __shared__ float pa_add[CW][32 * SB_STRIDE];     // every warp's addends of one superblock
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (blockIdx.x < cta_blocks)
        pa_moments_by_cta(b, pa, out, cta_min, pa_add[warp], blockIdx.x, cta_blocks, lane, warp);
    else
        pa_moments_by_warp(b, pa, out, cta_min, pa_add[warp], (blockIdx.x - cta_blocks) * CW + warp,
                           (gridDim.x - cta_blocks) * CW, lane);
}

// Median of float records: a radix select over the order-preserving 32-bit key (-0 before +0, NaN outside +-inf), in
// three levels of 12, 12 and 8 bits; each level counts, among the read's values whose key starts with the bins chosen
// so far, the next bits into a shared-memory histogram. Only the read's n values are counted, never its padding.
__device__ __forceinline__ uint32_t f32_key(uint32_t bits) {
    return bits ^ ((bits & 0x80000000u) ? 0xffffffffu : 0x80000000u);
}

// the bin of hist[0 .. MED_BINS) that holds `rank` (0-based; fewer than the histogram's count): sh[0] = the bin,
// sh[1] = the rank within it. All threads of the CTA (256 or more) call it.
__device__ void rank_bin(const uint32_t* hist, uint32_t rank, uint32_t* part, uint32_t* sh) {
    if (threadIdx.x < 256) {   // 256 threads x 16 bins
        uint32_t sum = 0;
        for (int k = 0; k < MED_BINS / 256; k++) sum += hist[threadIdx.x * (MED_BINS / 256) + k];
        part[threadIdx.x] = sum;
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        uint32_t mine = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) mine += part[lane * 8 + k];
        uint32_t incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        const uint32_t owner = __ballot_sync(0xffffffffu, incl > rank);
        if (lane == __ffs(owner) - 1) {
            uint32_t seen = incl - mine, g = (uint32_t)lane * 8u;
            for (;; g++) {
                if (seen + part[g] > rank) break;
                seen += part[g];
            }
            uint32_t k = g * (MED_BINS / 256);
            for (;; k++) {
                if (seen + hist[k] > rank) break;
                seen += hist[k];
            }
            sh[0] = k;
            sh[1] = rank - seen;
        }
    }
    __syncthreads();
}

// one level: the keys with key >> MATCH == prefix (MATCH = 32: every key) into hist[(key >> BIN) & MASK]; returns
// whether this thread met a NaN. Four 128-bit loads in flight per thread.
template <int MATCH, int BIN, uint32_t MASK>
__device__ __forceinline__ bool count_keys(const uint4* __restrict__ src, uint32_t n, uint32_t prefix, uint32_t* hist) {
    const uint32_t n_words = (n + 3u) >> 2;
    bool nan = false;
    for (uint32_t w0 = threadIdx.x; w0 < n_words; w0 += 4u * blockDim.x) {
        uint4 q[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t w = w0 + (uint32_t)k * blockDim.x;
            q[k] = w < n_words ? __ldg(src + w) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t w = w0 + (uint32_t)k * blockDim.x;
            const uint32_t wd[4] = {q[k].x, q[k].y, q[k].z, q[k].w};
#pragma unroll
            for (int h = 0; h < 4; h++) {
                if (w >= n_words || w * 4u + (uint32_t)h >= n) continue;
                const uint32_t key = f32_key(wd[h]);
                if (MATCH == 32) nan |= (wd[h] & 0x7fffffffu) > 0x7f800000u;
                if (MATCH == 32 || (key >> (MATCH & 31)) == prefix) atomicAdd(&hist[(key >> BIN) & MASK], 1u);
            }
        }
    }
    return nan;
}

// the element of rank `rank` of x[0 .. n) (16-byte aligned), NaN when the read holds a NaN
__device__ float select_rank_f32(const float* __restrict__ x, uint32_t n, uint32_t rank, uint32_t* hist,
                                 uint32_t* part, uint32_t* sh) {
    const uint4* __restrict__ src = reinterpret_cast<const uint4*>(x);
    for (int k = threadIdx.x; k < MED_BINS; k += blockDim.x) hist[k] = 0;
    __syncthreads();
    if (__syncthreads_or(count_keys<32, 20, 0xfffu>(src, n, 0u, hist))) return __uint_as_float(0x7fc00000u);
    rank_bin(hist, rank, part, sh);
    const uint32_t b1 = sh[0], r1 = sh[1];
    for (int k = threadIdx.x; k < MED_BINS; k += blockDim.x) hist[k] = 0;
    __syncthreads();
    count_keys<20, 8, 0xfffu>(src, n, b1, hist);
    __syncthreads();
    rank_bin(hist, r1, part, sh);
    const uint32_t p2 = (b1 << 12) | sh[0], r2 = sh[1];
    for (int k = threadIdx.x; k < MED_BINS; k += blockDim.x) hist[k] = 0;
    __syncthreads();
    count_keys<8, 0, 0xffu>(src, n, p2, hist);
    __syncthreads();
    rank_bin(hist, r2, part, sh);
    const uint32_t key = (p2 << 8) | sh[0];
    __syncthreads();                                 // sh and hist are free again
    return __uint_as_float(key ^ ((key & 0x80000000u) ? 0x80000000u : 0xffffffffu));
}

// reads of lo <= n < hi floats, one CTA of NT threads each; also the raw columns (NaN: there is no raw signal)
template <int NT>
__global__ void __launch_bounds__(NT) stat_pa_median_kernel(DevBatch b, const float* __restrict__ pa,
                                                            float* __restrict__ out, uint32_t lo, uint32_t hi) {
    __shared__ uint32_t hist[MED_BINS];
    __shared__ uint32_t part[256];
    __shared__ uint32_t sh[4];
    for (uint32_t r = blockIdx.x; r < b.n_reads; r += gridDim.x) {
        const uint32_t n = b.read_len[r];
        if (n < lo || n >= hi) continue;
        // ks_ksmall(n, copy, n/2), stat.h:56-64; an empty record: 0, as for int16 records
        const float med = n ? select_rank_f32(pa + b.read_off[r], n, (uint32_t)((int)n / 2), hist, part, sh) : 0.0f;
        if (threadIdx.x == 0) {
            float* o = out + (size_t)r * 6;
            const float nan = __uint_as_float(0x7fc00000u);
            o[0] = nan; o[2] = nan; o[4] = nan;
            o[5] = med;
        }
    }
}

int launch_stat_pa_moments(const DevBatch& b, const float* pa, float* stat6, uint32_t cta_min, int sm_count,
                           cudaStream_t st) {
    if (b.n_reads == 0) return 0;
    uint32_t g2 = b.n_reads < (uint32_t)sm_count * 2u ? b.n_reads : (uint32_t)sm_count * 2u;
    uint32_t g1 = (b.n_reads + CW - 1) / CW;         // one warp per read
    if (g1 > (uint32_t)sm_count * 8u) g1 = (uint32_t)sm_count * 8u;
    stat_pa_moments_kernel<<<g2 + g1, CW * 32, 0, st>>>(b, pa, stat6, cta_min, g2);
    return 1;
}

int launch_stat_pa_median(const DevBatch& b, const float* pa, float* stat6, uint32_t cta_min, int sm_count,
                          cudaStream_t st) {
    if (b.n_reads == 0) return 0;
    int g = (int)b.n_reads;
    stat_pa_median_kernel<1024><<<g > sm_count * 2 ? sm_count * 2 : g, 1024, 0, st>>>(b, pa, stat6, cta_min, 0xffffffffu);
    stat_pa_median_kernel<256><<<g > sm_count * 8 ? sm_count * 8 : g, 256, 0, st>>>(b, pa, stat6, 0u, cta_min);
    return 2;
}

// mean and standard deviation (float, in the reference's summation order) of the samples clamped to [0, 1200]:
// what jnn_core derives its band from (jnn.c:58-75, 181-185). moments2 = [n_reads][2].
int launch_jnn_moments(const DevBatch& b, float* moments2, uint32_t cta_min, int sm_count, cudaStream_t st) {
    return launch_moments<true>(b, moments2, cta_min, sm_count, st);
}

}  // namespace sgpu
