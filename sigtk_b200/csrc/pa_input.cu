// pa_input.cu -- event detection on the caller's own pA floats: getevents(n, pa, rna) (events.c:553-573).
//
// The chunk walker (walk.cu) cannot take floats: it places int16 bits under a float exponent and its test of the long
// window works on exact integer sums of raw - pivot (oracle/proofs/long_filter.md covers int16 input only). A pA batch
// therefore runs on the sequential-order kernels of generic.cu, which are exact for any input, with their serial part
// -- the two chains of FP64 additions of compute_sum_sumsq (events.c:293-303), one lane per read -- replaced by a
// parallel scan wherever the scan provably gives the same bits:
//
//   pa_init_kernel   tiles per read, the work list of all reads (scratch base = the read's own offset)
//   pa_tile_kernel   per tile of PT samples (several CTAs share a long read): the tile's sums of x and of fl(x*x) in
//                    FP64, and the exactness witness: the smallest nonzero |x| and fl(x*x), and upper bounds of
//                    sum |x| and sum fl(x*x) (additions rounded upwards)
//   pa_read_kernel   one warp per read: exclusive scan of its tile sums, the witness (below); a read that fails it
//                    goes to the list of gen_prefix_pa_kernel (the reference's own order) and seq_order[r] = 1
//   pa_scan_kernel   per tile of a read that passed: Sinc / Qinc = tile prefix + CTA scan of the tile's samples
//
// Witness: every value is a multiple of 2^k, k the smallest ulp exponent over the nonzero x (over the nonzero
// fl(x*x) for Q). If sum |x| < 2^(k+53), every partial sum of any grouping is a multiple of 2^k below 2^(k+53) in
// magnitude, i.e. a double: no FP64 addition rounds, and the reference's S[i] equals the scan's (DESIGN §3, point 1).
// A NaN or an infinity makes the bound NaN or infinite and fails the test; so does an fl(x*x) that overflows.
//
// Batches of int16 records (and decoded svb-zd streams) whose detector is the caller's set (sgpu_set_detector) take
// the same route: the tile and scan kernels are templates on the sample type, and an int16 instantiation forms the pA
// of every sample (misc.c:28) where it loads it, so no pA array is stored.
#include <type_traits>

#include "kernels.cuh"

namespace sgpu {

constexpr int PT = 4096;          // samples per tile
constexpr int PT_THREADS = 256;   // 16 samples per thread

// ulp exponent of a positive finite float given by its bits: 2^(e-150) for a normal, 2^-149 for a subnormal
__device__ __forceinline__ int ulp_exp(uint32_t bits) {
    const int e = (int)(bits >> 23);
    return (e ? e : 1) - 150;
}
__device__ __forceinline__ double pow2(int e) {  // 2^e for -1022 <= e <= 1023
    return __longlong_as_double((long long)(e + 1023) << 52);
}
// sum < 2^(ulp exponent of the smallest nonzero addend + 53); false for a NaN sum
__device__ __forceinline__ bool sum_exact(double bound, uint32_t min_bits) {
    return min_bits == 0xffffffffu ? bound == 0.0 : bound < pow2(ulp_exp(min_bits) + 53);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_sum_up(double v) {  // rounded upwards: an upper bound whatever the order
#pragma unroll
    for (int o = 16; o; o >>= 1) v = __dadd_ru(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ uint32_t warp_min(uint32_t v) { return __reduce_min_sync(0xffffffffu, v); }

// the reference's floats of values i .. i+3 of a read (i a multiple of 4; reads start on 8 samples): the caller's pA
// as it is, or int16 samples through the read's calibration
__device__ __forceinline__ float4 load4(const float* __restrict__ p, uint64_t i, float, float) {
    return __ldg(reinterpret_cast<const float4*>(p + i));
}
__device__ __forceinline__ float4 load4(const int16_t* __restrict__ p, uint64_t i, float off, float unit) {
    const uint2 v = __ldg(reinterpret_cast<const uint2*>(p + i));
    return make_float4(pa_of((int16_t)(uint16_t)v.x, off, unit), pa_of((int16_t)(uint16_t)(v.x >> 16), off, unit),
                       pa_of((int16_t)(uint16_t)v.y, off, unit), pa_of((int16_t)(uint16_t)(v.y >> 16), off, unit));
}
template <typename T>
__device__ __forceinline__ void calibration(const DevBatch& b, uint32_t r, float& off, float& unit) {
    off = 0.0f; unit = 0.0f;
    if constexpr (std::is_same_v<T, int16_t>) { off = b.offset[r]; unit = b.unit[r]; }
}

// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pa_init_kernel(DevBatch b, uint32_t* __restrict__ tile_cnt,
                                                      uint32_t* __restrict__ fixups, uint32_t* __restrict__ all_list,
                                                      uint64_t* __restrict__ all_sbase, uint32_t* __restrict__ all_count,
                                                      uint32_t* __restrict__ ord_count) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g == 0) { *all_count = b.n_reads; *ord_count = 0u; }
    for (uint32_t r = g; r < b.n_reads; r += gridDim.x * blockDim.x) {
        tile_cnt[r] = (b.read_len[r] + (PT - 1u)) / PT;
        fixups[r] = 0u;
        all_list[r] = r;
        all_sbase[r] = b.read_off[r];  // the scratch holds the whole span (capi.cu grows it on demand)
    }
}

// ---------------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(PT_THREADS) pa_tile_kernel(DevBatch b, const T* __restrict__ pa,
                                                             const uint64_t* __restrict__ tile_base,
                                                             double* __restrict__ tS, double* __restrict__ tQ,
                                                             double* __restrict__ tA, double* __restrict__ tB,
                                                             uint2* __restrict__ tmin) {
    __shared__ double sh[4][PT_THREADS / 32];
    __shared__ uint32_t shm[2][PT_THREADS / 32];
    const uint64_t n_tiles = tile_base[b.n_reads];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (uint64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const uint32_t r = find_read(tile_base, b.n_reads, t);
        const uint32_t i0 = (uint32_t)(t - tile_base[r]) * PT, n = b.read_len[r];
        const uint64_t src = b.read_off[r] + i0;
        float off, unit;
        calibration<T>(b, r, off, unit);
        // the order of the additions does not matter here (only exact sums are used): coalesced 4-value loads
        float4 v[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t i = 4u * (k * PT_THREADS + threadIdx.x);   // reads are padded to 8 samples
            v[k] = i0 + i < n ? load4(pa, src + i, off, unit) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        double s = 0.0, q = 0.0, a = 0.0, bq = 0.0;
        uint32_t mx = 0xffffffffu, mq = 0xffffffffu;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const float e[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
#pragma unroll
            for (int m = 0; m < 4; m++) {
                const float x = i0 + 4u * (k * PT_THREADS + threadIdx.x) + m < n ? e[m] : 0.0f;
                const float xq = __fmul_rn(x, x);  // events.c:301: float product, widened afterwards
                s = __dadd_rn(s, (double)x);
                q = __dadd_rn(q, (double)xq);
                a = __dadd_ru(a, fabs((double)x));
                bq = __dadd_ru(bq, (double)xq);
                const uint32_t ux = __float_as_uint(x) & 0x7fffffffu, uq = __float_as_uint(xq) & 0x7fffffffu;
                if (ux) mx = min(mx, ux);
                if (uq) mq = min(mq, uq);
            }
        }
        s = warp_sum(s); q = warp_sum(q); a = warp_sum_up(a); bq = warp_sum_up(bq);
        mx = warp_min(mx); mq = warp_min(mq);
        if (lane == 0) { sh[0][wid] = s; sh[1][wid] = q; sh[2][wid] = a; sh[3][wid] = bq; shm[0][wid] = mx; shm[1][wid] = mq; }
        __syncthreads();
        if (wid == 0) {
            const bool on = lane < PT_THREADS / 32;
            s = warp_sum(on ? sh[0][lane] : 0.0);
            q = warp_sum(on ? sh[1][lane] : 0.0);
            a = warp_sum_up(on ? sh[2][lane] : 0.0);
            bq = warp_sum_up(on ? sh[3][lane] : 0.0);
            mx = warp_min(on ? shm[0][lane] : 0xffffffffu);
            mq = warp_min(on ? shm[1][lane] : 0xffffffffu);
            if (lane == 0) { tS[t] = s; tQ[t] = q; tA[t] = a; tB[t] = bq; tmin[t] = make_uint2(mx, mq); }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) pa_read_kernel(DevBatch b, const uint64_t* __restrict__ tile_base,
                                                      double* __restrict__ tS, double* __restrict__ tQ,
                                                      const double* __restrict__ tA, const double* __restrict__ tB,
                                                      const uint2* __restrict__ tmin, int force_all,
                                                      uint32_t* __restrict__ seq_flag, uint32_t* __restrict__ ord_list,
                                                      uint64_t* __restrict__ ord_sbase, uint32_t* __restrict__ ord_count,
                                                      unsigned long long* __restrict__ counters) {
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t r = warp; r < b.n_reads; r += n_warps) {
        const uint64_t t0 = tile_base[r], t1 = tile_base[r + 1];
        double cs = 0.0, cq = 0.0, a = 0.0, bq = 0.0;   // running prefix of the tile sums; bounds
        uint32_t mx = 0xffffffffu, mq = 0xffffffffu;
        for (uint64_t g = t0; g < t1; g += 32) {
            const uint64_t t = g + lane;
            const bool on = t < t1;
            const double s = on ? tS[t] : 0.0, q = on ? tQ[t] : 0.0;
            a = __dadd_ru(a, on ? tA[t] : 0.0);
            bq = __dadd_ru(bq, on ? tB[t] : 0.0);
            const uint2 m = on ? tmin[t] : make_uint2(0xffffffffu, 0xffffffffu);
            mx = min(mx, m.x); mq = min(mq, m.y);
            double is = s, iq = q;   // inclusive scan over the lanes (exact when the witness holds)
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const double us = __shfl_up_sync(0xffffffffu, is, o), uq = __shfl_up_sync(0xffffffffu, iq, o);
                if (lane >= o) { is = __dadd_rn(is, us); iq = __dadd_rn(iq, uq); }
            }
            if (on) { tS[t] = __dadd_rn(cs, __dsub_rn(is, s)); tQ[t] = __dadd_rn(cq, __dsub_rn(iq, q)); }
            cs = __dadd_rn(cs, __shfl_sync(0xffffffffu, is, 31));
            cq = __dadd_rn(cq, __shfl_sync(0xffffffffu, iq, 31));
        }
        a = warp_sum_up(a); bq = warp_sum_up(bq);
        mx = warp_min(mx); mq = warp_min(mq);
        if (lane == 0) {
            const bool ordered = b.read_len[r] != 0 && (force_all || !(sum_exact(a, mx) && sum_exact(bq, mq)));
            seq_flag[r] = ordered ? 1u : 0u;
            if (ordered) {
                const uint32_t k = atomicAdd(ord_count, 1u);
                ord_list[k] = r;
                ord_sbase[k] = b.read_off[r];
                atomicAdd(&counters[1], 1ull);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// CTA-wide inclusive scan of (s, q) over the threads; returns the CTA's totals in (ts, tq)
__device__ __forceinline__ void cta_scan2(double& s, double& q, double& ts, double& tq, double (*sh)[PT_THREADS / 32]) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double us = __shfl_up_sync(0xffffffffu, s, o), uq = __shfl_up_sync(0xffffffffu, q, o);
        if (lane >= o) { s = __dadd_rn(s, us); q = __dadd_rn(q, uq); }
    }
    if (lane == 31) { sh[0][wid] = s; sh[1][wid] = q; }
    __syncthreads();
    double es = 0.0, eq = 0.0;
    ts = 0.0; tq = 0.0;
#pragma unroll
    for (int w = 0; w < PT_THREADS / 32; w++) {
        const double vs = sh[0][w], vq = sh[1][w];
        if (w < wid) { es = __dadd_rn(es, vs); eq = __dadd_rn(eq, vq); }
        ts = __dadd_rn(ts, vs); tq = __dadd_rn(tq, vq);
    }
    s = __dadd_rn(s, es); q = __dadd_rn(q, eq);
    __syncthreads();
}

template <typename T>
__global__ void __launch_bounds__(PT_THREADS) pa_scan_kernel(DevBatch b, const T* __restrict__ pa,
                                                             const uint64_t* __restrict__ tile_base,
                                                             const double* __restrict__ tS, const double* __restrict__ tQ,
                                                             const uint32_t* __restrict__ seq_flag,
                                                             double* __restrict__ Sinc, double* __restrict__ Qinc) {
    __shared__ double sh[2][PT_THREADS / 32];
    const uint64_t n_tiles = tile_base[b.n_reads];
    for (uint64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const uint32_t r = find_read(tile_base, b.n_reads, t);
        if (seq_flag[r]) continue;   // (the whole CTA) the read is summed in the reference's order
        const uint32_t i0 = (uint32_t)(t - tile_base[r]) * PT, n = b.read_len[r];
        const uint64_t base = b.read_off[r];   // = the read's scratch base
        double cs = tS[t], cq = tQ[t];         // S[i0], Q[i0]
        float off, unit;
        calibration<T>(b, r, off, unit);
        // 1,024 samples per round, four consecutive ones per thread; the next round's loads in flight
        const uint64_t src = base + i0 + 4u * threadIdx.x;
        float4 nxt = i0 + 4u * threadIdx.x < n ? load4(pa, src, off, unit) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
        for (int k = 0; k < PT / (4 * PT_THREADS); k++) {
            const uint32_t i = i0 + (uint32_t)(k * 4 * PT_THREADS) + 4u * threadIdx.x;
            const float4 v = nxt;
            const uint32_t ni = i + 4u * PT_THREADS;
            nxt = (k + 1 < PT / (4 * PT_THREADS) && ni < n) ? load4(pa, src + (uint64_t)(k + 1) * 4 * PT_THREADS, off, unit)
                                                              : make_float4(0.f, 0.f, 0.f, 0.f);
            const float e[4] = {v.x, v.y, v.z, v.w};
            double ps[4], pq[4], s = 0.0, q = 0.0;
#pragma unroll
            for (int m = 0; m < 4; m++) {
                const float x = i + m < n ? e[m] : 0.0f;
                s = __dadd_rn(s, (double)x);
                q = __dadd_rn(q, (double)__fmul_rn(x, x));
                ps[m] = s; pq[m] = q;
            }
            double ts, tq, es = s, eq = q;
            cta_scan2(es, eq, ts, tq, sh);
            es = __dadd_rn(cs, __dsub_rn(es, s));   // S just before this thread's first sample
            eq = __dadd_rn(cq, __dsub_rn(eq, q));
#pragma unroll
            for (int m = 0; m < 4; m++) { ps[m] = __dadd_rn(es, ps[m]); pq[m] = __dadd_rn(eq, pq[m]); }
            if (i + 3u < n) {   // 32-byte aligned: the read starts on 8 samples, i on 4
                double2* ds = reinterpret_cast<double2*>(Sinc + base + i);
                double2* dq = reinterpret_cast<double2*>(Qinc + base + i);
                ds[0] = make_double2(ps[0], ps[1]); ds[1] = make_double2(ps[2], ps[3]);
                dq[0] = make_double2(pq[0], pq[1]); dq[1] = make_double2(pq[2], pq[3]);
            } else {
#pragma unroll
                for (int m = 0; m < 4; m++)
                    if (i + m < n) { Sinc[base + i + m] = ps[m]; Qinc[base + i + m] = pq[m]; }
            }
            cs = __dadd_rn(cs, ts); cq = __dadd_rn(cq, tq);
            if (i0 + (uint32_t)((k + 1) * 4 * PT_THREADS) >= n) break;   // (uniform over the CTA)
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
uint64_t pa_tile_capacity(uint64_t max_samples, uint32_t max_reads) { return max_samples / PT + max_reads + 1; }

template <typename T>
static void launch_tiles_and_scan(const DevBatch& b, const T* src, PaScratch& w, Scratch& sc, uint32_t* seq_flag,
                                  int force_all, int sm_count, cudaStream_t st) {
    const uint64_t tiles = b.span / PT + b.n_reads;   // at least the batch's tiles
    pa_tile_kernel<T><<<grid_cap(tiles, 1, sm_count * 8), PT_THREADS, 0, st>>>(b, src, w.tile_base, w.tS, w.tQ, w.tA,
                                                                             w.tB, w.tmin);
    pa_read_kernel<<<grid_cap((uint64_t)b.n_reads * 32, 128, sm_count * 8), 128, 0, st>>>(
        b, w.tile_base, w.tS, w.tQ, w.tA, w.tB, w.tmin, force_all, seq_flag, w.ord_list, w.ord_sbase, w.ord_count,
        sc.counters);
    pa_scan_kernel<T><<<grid_cap(tiles, 1, sm_count * 8), PT_THREADS, 0, st>>>(b, src, w.tile_base, w.tS, w.tQ,
                                                                             seq_flag, sc.Sinc, sc.Qinc);
}

int launch_pa_prefix(const DevBatch& b, const float* pa, PaScratch& w, Scratch& sc, uint32_t* seq_flag,
                     uint32_t* fixups, int force_all, int sm_count, cudaStream_t st) {
    pa_init_kernel<<<grid_cap(b.n_reads, 256, sm_count), 256, 0, st>>>(b, w.tile_cnt, fixups, sc.seq_list, sc.seq_sbase,
                                                                       sc.seq_count, w.ord_count);
    int n = 1 + launch_scan_u32(w.tile_cnt, b.n_reads, w.tile_base, nullptr, sc, st);
    if (pa) launch_tiles_and_scan(b, pa, w, sc, seq_flag, force_all, sm_count, st);
    else    launch_tiles_and_scan(b, b.samples, w, sc, seq_flag, force_all, sm_count, st);
    return n + 4;
}

}  // namespace sgpu
