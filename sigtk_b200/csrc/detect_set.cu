// detect_set.cu -- the detector of the sequential-order kernels (generic.cu) for a caller's parameter set
// (sgpu_set_detector). It is a translation unit of its own so that the compile-time instantiations of generic.cu for
// the reference's sets keep their code.
#include "kernels.cuh"

namespace sgpu {

// The warp-chunked detector for a caller's parameter set (sgpu_set_detector): the chunks, cold warm-up and boundary
// check of detect_read_chunked, stepped with det_step -- the reference's own comparisons with the set's windows,
// thresholds and height at run time. Being the reference's step it needs no NaN rule (a NaN t-statistic does to the
// state what it does in the reference's order) and holds for every peak_height, where the branch-free step of
// walk_core.cuh assumes height >= 0. The canonical state at boundary b is the whole DetState of both detectors, with
// the long one's masked_to folded to 0 when it no longer masks a step >= b. Returns the read's mismatched chunks.
constexpr uint32_t SET_WARMUP = 384;  // the RNA default's warm-up (its long window, 14, is the largest a set may have)
__device__ __forceinline__ void set_canon(const DetState& s, const DetState& l, uint32_t b, uint32_t (&v)[7]) {
    v[0] = __float_as_uint(s.peak_value); v[1] = (uint32_t)s.peak_pos; v[2] = (uint32_t)s.valid;
    v[3] = __float_as_uint(l.peak_value); v[4] = (uint32_t)l.peak_pos; v[5] = (uint32_t)l.valid;
    v[6] = l.masked_to >= b ? l.masked_to : 0u;
}
__device__ uint32_t detect_read_chunked_set(const float* __restrict__ t1, const float* __restrict__ t2, uint64_t base,
                                            uint64_t foff, uint32_t n, uint32_t* __restrict__ bitmap, int lane,
                                            const DetParams& p) {
    if (lane == 0) {
        clear_read_bits(bitmap, foff, foff + n);
        atomicOr(&bitmap[foff >> 5], 1u << (foff & 31));  // event 0 starts at the first sample
    }
    __syncwarp();
    const uint32_t n_chunks = (n + GD_CHUNK - 1) / GD_CHUNK;
    uint32_t n_bad = 0;
    uint32_t carry[7] = {};  // end state of the previous group's last chunk
    for (uint32_t c0 = 0; c0 < n_chunks; c0 += 32) {
        const uint32_t c = c0 + lane;
        const bool have = c < n_chunks;
        const uint32_t s0 = c * GD_CHUNK, s1 = min(n, s0 + GD_CHUNK);
        uint32_t begin[7] = {}, end[7] = {};
        if (have) {
            DetState s, l;
            det_reset(s);
            det_reset(l);
            uint32_t i = (c == 0) ? 1u : s0 - SET_WARMUP;  // position 0 is never stepped (masked_to = 0, events.c:387)
            for (; i < s0; i++) {  // warm-up: nothing is recorded
                det_step(s, &l, true, i, __ldg(t1 + base + i), p.thr1, p.w1, p.height);
                det_step(l, nullptr, false, i, __ldg(t2 + base + i), p.thr2, p.w2, p.height);
            }
            set_canon(s, l, s0, begin);
            for (; i < s1; i++) {
                const int32_t ps = det_step(s, &l, true, i, __ldg(t1 + base + i), p.thr1, p.w1, p.height);
                if (ps > 0) { const uint64_t f = foff + (uint32_t)ps; atomicOr(&bitmap[f >> 5], 1u << (f & 31)); }
                const int32_t pl = det_step(l, nullptr, false, i, __ldg(t2 + base + i), p.thr2, p.w2, p.height);
                if (pl > 0) { const uint64_t f = foff + (uint32_t)pl; atomicOr(&bitmap[f >> 5], 1u << (f & 31)); }
            }
            set_canon(s, l, s1, end);
        }
        // chunk c must have reached the state chunk c-1 ended in
        bool same = true;
#pragma unroll
        for (int q = 0; q < 7; q++) {
            uint32_t prev = __shfl_up_sync(0xffffffffu, end[q], 1);
            if (lane == 0) prev = carry[q];
            same = same && (prev == begin[q]);
        }
        if (have && c > 0 && !same) n_bad++;
        const int last = (int)min(31u, n_chunks - 1u - c0);
#pragma unroll
        for (int q = 0; q < 7; q++) carry[q] = __shfl_sync(0xffffffffu, end[q], last);
    }
    if (__any_sync(0xffffffffu, n_bad != 0)) {
        __syncwarp();
        if (lane == 0) detect_read_in_order(p, t1, t2, base, foff, n, bitmap);
    }
    return __reduce_add_sync(0xffffffffu, n_bad);
}

// fixups[r] = the read's mismatched chunks
__global__ void __launch_bounds__(128) gen_detect_set_kernel(DevBatch b, WorkList wl, const float* __restrict__ t1,
                                                             const float* __restrict__ t2, uint32_t* __restrict__ bitmap,
                                                             uint32_t* __restrict__ fixups, DetParams p) {
    const uint32_t n_list = *wl.count;
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t j = warp; j < n_list; j += n_warps) {
        const uint32_t r = wl.list[j];
        const uint32_t n = b.read_len[r];
        if (n == 0) continue;
        const uint32_t n_bad = detect_read_chunked_set(t1, t2, wl.sbase[j], b.read_off[r], n, bitmap, lane, p);
        if (lane == 0) fixups[r] = n_bad;
    }
}

int launch_detect_set(const DevBatch& b, const WorkList& wl, Scratch& sc, uint32_t* fixups, const DetParams& set,
                      int sm_count, cudaStream_t st) {
    gen_detect_set_kernel<<<sm_count * 8, 128, 0, st>>>(b, wl, sc.t1, sc.t2, sc.bitmap, fixups, set);
    return 1;
}

}  // namespace sgpu
