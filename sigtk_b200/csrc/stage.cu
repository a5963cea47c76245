// stage.cu -- reads at any sample offset (sgpu_run_device_at, sgpu_run_device_pa_at): a gather that stages the
// caller's reads into the aligned layout every other kernel reads, so that none of them has to load unaligned reads.
//
//   stage_count_kernel    refuses reads past the caller's array (empty records, status SGPU_E_INVAL) and counts the
//                         8-sample groups of the others
//   scan_counts_kernel    (generic.cu) their exclusive scan
//   stage_offsets_kernel  staged offsets in samples; reads whose staged end passes the span become empty records
//                         (status SGPU_E_TOOBIG)
//   stage_gather_kernel   copies every 8-sample group of the staged layout from the caller's array
//
// The gather is bandwidth-bound work. A warp takes 32 x STAGE_IT consecutive groups of the staged layout per step, so
// one long read and many short ones fill the GPU alike. Each group is stored with aligned 128-bit stores (two for
// floats); its 8 elements are cut from the aligned 16-byte words that cover them, shifted into place by whole 32-bit
// words and, for int16 samples at an odd position, a 16-bit funnel shift. A word is loaded only when it holds one of
// the group's samples, so no load touches a 16-byte word outside the caller's array. Padding up to the next group is
// written as zeros.
#include "kernels.cuh"

namespace sgpu {
namespace {

constexpr int STAGE_IT = 4;  // groups per lane and step (their loads are all in flight before the first store)

__global__ void __launch_bounds__(256) stage_count_kernel(StageSrc s, uint32_t* __restrict__ len, uint32_t* __restrict__ grp,
                                                          int* __restrict__ status) {
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < s.n_reads; r += gridDim.x * blockDim.x) {
        const uint64_t off = s.read_off[r];
        const uint32_t n = s.read_len[r];
        const bool ok = off <= s.n_elems && n <= s.n_elems - off;
        if (!ok) atomicExch(status, SGPU_DEV_E_INVAL);
        len[r] = ok ? n : 0u;
        grp[r] = ok ? (uint32_t)(((uint64_t)n + 7u) >> 3) : 0u;
    }
}

// off[r] = 8 goff[r], clamped to the span; a read that would end past it is staged as an empty record. (SGPU_E_INVAL of
// stage_count_kernel, already written, takes precedence.)
__global__ void __launch_bounds__(256) stage_offsets_kernel(const uint64_t* __restrict__ goff, uint32_t n_reads,
                                                            uint64_t span, uint64_t* __restrict__ off,
                                                            uint32_t* __restrict__ len, int* __restrict__ status) {
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r <= n_reads; r += gridDim.x * blockDim.x) {
        const uint64_t a = goff[r] << 3;
        if (r < n_reads && (goff[r + 1] << 3) > span) {
            len[r] = 0u;
            atomicCAS(status, 0, SGPU_DEV_E_TOOBIG);
        }
        off[r] = a < span ? a : span;
    }
}

// largest r in [lo, hi] with off[r] <= p (off[lo] <= p)
__device__ __forceinline__ uint32_t read_between(const uint64_t* __restrict__ off, uint32_t lo, uint32_t hi, uint64_t p) {
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if (off[mid] <= p) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// T: int16_t or float. A group is 8 elements: OUT = 2 sizeof(T) 32-bit words, cut from the IN / 4 16-byte source words
// that cover them at any 16-bit position.
template <typename T>
__global__ void __launch_bounds__(256) stage_gather_kernel(const T* __restrict__ src, const uint64_t* __restrict__ read_off,
                                                           const uint64_t* __restrict__ off, const uint32_t* __restrict__ len,
                                                           uint32_t n_reads, T* __restrict__ dst) {
    constexpr int OUT = 2 * (int)sizeof(T), IN = OUT + 4, NL = IN / 4;
    const uint64_t n_groups = off[n_reads] >> 3;
    const int lane = threadIdx.x & 31;
    const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uintptr_t base = reinterpret_cast<uintptr_t>(src);
    for (uint64_t c0 = warp * (32 * STAGE_IT); c0 < n_groups; c0 += n_warps * (32 * STAGE_IT)) {
        // the reads of the step's first and last groups bound every lane's search
        const uint64_t c1 = c0 + 32 * STAGE_IT - 1 < n_groups ? c0 + 32 * STAGE_IT - 1 : n_groups - 1;
        uint32_t r = 0;
        if (lane == 0) r = find_read(off, n_reads, c0 << 3);
        if (lane == 31) r = find_read(off, n_reads, c1 << 3);
        const uint32_t lo = __shfl_sync(0xffffffffu, r, 0), hi = __shfl_sync(0xffffffffu, r, 31);
        r = lo;
        uint32_t w[STAGE_IT][IN];
        uint32_t keep[STAGE_IT];  // 16-bit halves of the group that hold samples (the rest is padding)
        uint32_t shift[STAGE_IT];  // the group's position in its first source word, in 16-bit units
#pragma unroll
        for (int it = 0; it < STAGE_IT; it++) {
            const uint64_t g = c0 + (uint64_t)it * 32 + lane;
            keep[it] = 0u;
            shift[it] = 0u;
#pragma unroll
            for (int k = 0; k < IN; k++) w[it][k] = 0u;
            if (g >= n_groups) continue;
            const uint64_t p = g << 3;
            r = read_between(off, r, hi, p);
            const uint64_t q = p - off[r];  // (a multiple of 8)
            const uint32_t n = len[r];
            if (q >= n) continue;           // padding of an empty record: zeros
            const uint32_t m = n - q < 8u ? (uint32_t)(n - q) : 8u;
            const uintptr_t a = base + (read_off[r] + q) * sizeof(T);
            const uintptr_t a0 = a & ~(uintptr_t)15, end = a + m * sizeof(T);
            shift[it] = (uint32_t)(a & 15) >> 1;
            keep[it] = m * (uint32_t)(sizeof(T) / 2);
#pragma unroll
            for (int k = 0; k < NL; k++) {
                if (a0 + 16u * k >= end) break;  // a word holds none of the group's samples: never loaded
                const int4 v = __ldg(reinterpret_cast<const int4*>(a0 + 16u * k));
                w[it][4 * k] = (uint32_t)v.x; w[it][4 * k + 1] = (uint32_t)v.y;
                w[it][4 * k + 2] = (uint32_t)v.z; w[it][4 * k + 3] = (uint32_t)v.w;
            }
        }
#pragma unroll
        for (int it = 0; it < STAGE_IT; it++) {
            const uint64_t g = c0 + (uint64_t)it * 32 + lane;
            if (g >= n_groups) continue;
            const uint32_t h = shift[it];
            uint32_t t[IN];
#pragma unroll
            for (int k = 0; k < IN; k++) t[k] = w[it][k];
            // shift down by h 16-bit units: 2 words, 1 word, then 16 bits (odd h: int16 only)
#pragma unroll
            for (int k = 0; k < IN - 2; k++) t[k] = (h & 4u) ? t[k + 2] : t[k];
#pragma unroll
            for (int k = 0; k < IN - 3; k++) t[k] = (h & 2u) ? t[k + 1] : t[k];
            uint32_t o[OUT];
#pragma unroll
            for (int j = 0; j < OUT; j++) {
                const uint32_t v = (sizeof(T) == 2 && (h & 1u)) ? __funnelshift_r(t[j], t[j + 1], 16) : t[j];
                const uint32_t mask = 2u * j + 1u < keep[it] ? 0xffffffffu : (2u * j < keep[it] ? 0x0000ffffu : 0u);
                o[j] = v & mask;
            }
            int4* d = reinterpret_cast<int4*>(dst + (g << 3));
#pragma unroll
            for (int j = 0; j < OUT / 4; j++)
                d[j] = make_int4((int)o[4 * j], (int)o[4 * j + 1], (int)o[4 * j + 2], (int)o[4 * j + 3]);
        }
    }
}

}  // namespace

int launch_stage_reads(const StageSrc& s, bool f32, StageScratch& w, Scratch& sc, int sm_count, cudaStream_t st) {
    if (s.n_reads == 0) {
        cudaMemsetAsync(w.off, 0, sizeof(uint64_t), st);
        return 0;
    }
    stage_count_kernel<<<grid_cap(s.n_reads, 256, sm_count * 8), 256, 0, st>>>(s, w.len, w.grp, sc.status);
    int n = 1 + launch_scan_u32(w.grp, s.n_reads, w.goff, nullptr, sc, st);
    stage_offsets_kernel<<<grid_cap((uint64_t)s.n_reads + 1, 256, sm_count * 8), 256, 0, st>>>(
        w.goff, s.n_reads, s.span, w.off, w.len, sc.status);
    const int grid = grid_cap(((s.span >> 3) + STAGE_IT - 1) / STAGE_IT, 256, sm_count * 16);
    if (f32)
        stage_gather_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(s.src), s.read_off, w.off, w.len,
                                                         s.n_reads, w.f32);
    else
        stage_gather_kernel<int16_t><<<grid, 256, 0, st>>>(static_cast<const int16_t*>(s.src), s.read_off, w.off,
                                                           w.len, s.n_reads, w.i16);
    return n + 2;
}

}  // namespace sgpu
