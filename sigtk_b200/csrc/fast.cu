// fast.cu -- the small kernels around the chunk walker (walk.cu) and the event emitter (emit.cu):
//
//   init_reads_kernel      resets the per-read witness / flags, first read of every 2048-sample bitmap tile
//   build_seq_list_kernel  evaluates the exact-sum witness per read and compacts the list of reads that need the
//                          sequential-order kernels (generic.cu)
//   count_tile_bits_kernel / read_event_offsets_kernel   ranks of event starts (ev_off)
//
// Why the fast path is bit-identical to the reference although the sums are formed in another order: the
// reference's S[i], Q[i] (double) are exact (no rounding happened) whenever every value is a multiple of 2^k and
// the sum of magnitudes stays below 2^(k+53); then ANY grouping of the same additions is exact too, and every
// window / event difference S[b]-S[a] equals the exact sum of the samples in [a,b).  The witness checks that
// sufficient condition per read from the smallest nonzero and the largest |pA|; reads that fail it
// are recomputed in the reference's own order by generic.cu.
#include "kernels.cuh"

namespace sgpu {
constexpr int T = FAST_TILE;  // samples per tile of the event-start bitmap
}

namespace sgpu {

// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool sums_exact(uint32_t e_min, uint32_t e_max, uint32_t log2n) {
    // every value is a multiple of 2^(e_min-150) and the sum of magnitudes is below 2^(e_max+1-127+log2n)
    return e_min != 0u && e_max < 255u && (e_max + 1u + log2n <= e_min + 30u);
}

__global__ void __launch_bounds__(256) build_seq_list_kernel(DevBatch b, const uint32_t* __restrict__ wit_min,
                                                             const uint32_t* __restrict__ wit_max,
                                                             uint32_t* __restrict__ seq_flag, int force_all,
                                                             uint32_t* __restrict__ seq_list,
                                                             uint64_t* __restrict__ seq_sbase,
                                                             uint32_t* __restrict__ seq_count,
                                                             unsigned long long* __restrict__ cursor, uint64_t gen_cap,
                                                             int* __restrict__ status,
                                                             unsigned long long* __restrict__ counters) {
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < b.n_reads; r += gridDim.x * blockDim.x) {
        const uint32_t n = b.read_len[r];
        bool flag = force_all || seq_flag[r] != 0u;
        // the walker's unguarded shortcuts need unit > 0 (no -0 sums) and 32-bit positions with headroom
        const float unit = b.unit[r];
        if (!(unit > 0.0f && unit <= FLT_MAX) || n >= (1u << 30) - 64u) flag = true;
        if (!flag && n > 0) {
            const uint32_t mn = wit_min[r], mx = wit_max[r];
            // every nonzero |pA| must be in [2^-60, 2^20) (the range of the walker's shortcuts) ...
            if (mn < 0x21800000u || mn > mx || mx >= 0x49800000u) flag = true;
            else {  // ... and the sums of x and x*x must be exact whatever the order
                const uint32_t log2n = n > 1 ? 32u - __clz(n - 1) : 0u;
                const float fmn = __uint_as_float(mn), fmx = __uint_as_float(mx);
                const uint32_t qmn = __float_as_uint(__fmul_rn(fmn, fmn)), qmx = __float_as_uint(__fmul_rn(fmx, fmx));
                if (!(sums_exact(mn >> 23, mx >> 23, log2n) && sums_exact(qmn >> 23, qmx >> 23, log2n))) flag = true;
            }
        }
        if (n == 0) flag = false;
        seq_flag[r] = flag ? 1u : 0u;
        if (flag) {
            const uint64_t need = ((uint64_t)n + 7u) & ~7ull;
            const unsigned long long base = atomicAdd(cursor, (unsigned long long)need);
            if (base + need > gen_cap) { atomicExch(status, SGPU_DEV_E_SCRATCH); continue; }
            const uint32_t k = atomicAdd(seq_count, 1u);
            seq_list[k] = r;
            seq_sbase[k] = base;
            atomicAdd(&counters[1], 1ull);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) count_tile_bits_kernel(const uint32_t* __restrict__ bitmap, uint32_t n_tiles,
                                                              uint32_t* __restrict__ tile_cnt) {
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t t = warp; t < n_tiles; t += n_warps) {
        const uint2 v = reinterpret_cast<const uint2*>(bitmap + (size_t)t * (T / 32))[lane];
        uint32_t c = __popc(v.x) + __popc(v.y);
        for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        if (lane == 0) tile_cnt[t] = c;
    }
}

// number of event starts before flat position p
__device__ __forceinline__ uint64_t rank_before(const uint32_t* __restrict__ bitmap, const uint64_t* __restrict__ tile_base,
                                                uint64_t p) {
    const uint64_t t = p / T;
    const uint32_t u = (uint32_t)(p - t * T);
    uint64_t k = tile_base[t];
    const uint32_t* w = bitmap + t * (T / 32);
    for (uint32_t j = 0; j < (u >> 5); j++) k += __popc(w[j]);
    if (u & 31) k += __popc(w[u >> 5] & ((1u << (u & 31)) - 1u));
    return k;
}

__global__ void __launch_bounds__(256) read_event_offsets_kernel(DevBatch b, const uint32_t* __restrict__ bitmap,
                                                                 const uint64_t* __restrict__ tile_base,
                                                                 uint32_t n_tiles, uint64_t* __restrict__ ev_off) {
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r <= b.n_reads; r += gridDim.x * blockDim.x) {
        if (r == b.n_reads) { ev_off[r] = tile_base[n_tiles]; continue; }
        const uint64_t p = b.read_off[r];
        ev_off[r] = (p >= b.span) ? tile_base[n_tiles] : rank_before(bitmap, tile_base, p);
    }
}

// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) init_reads_kernel(DevBatch b, uint32_t n_tiles, uint32_t* __restrict__ wit_min,
                                                         uint32_t* __restrict__ wit_max, uint32_t* __restrict__ seq_flag,
                                                         uint32_t* __restrict__ fixups, uint32_t* __restrict__ seq_count,
                                                         unsigned long long* __restrict__ cursor,
                                                         uint32_t* __restrict__ tile_read0) {
    const uint32_t n_reads = b.n_reads;
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g == 0) { *seq_count = 0u; *cursor = 0ull; }
    // first read that can intersect the staged region of every tile (the region starts at most 160 samples early)
    for (uint32_t t = g; t < n_tiles; t += gridDim.x * blockDim.x) {
        const long long p = (long long)t * T - 160;
        tile_read0[t] = find_read(b.read_off, n_reads, (uint64_t)(p < 0 ? 0 : p));
    }
    for (uint32_t r = g; r < n_reads; r += gridDim.x * blockDim.x) {
        wit_min[r] = 0xffffffffu;
        wit_max[r] = 0u;
        seq_flag[r] = 0u;
        fixups[r] = 0u;
    }
}

uint32_t fast_tiles_for(uint64_t span) { return (uint32_t)((span + T - 1) / T); }

int launch_init_reads(const DevBatch& b, Scratch& sc, uint32_t* seq_flag, uint32_t* fixups, int sm_count,
                      cudaStream_t st) {
    const uint32_t n_tiles = fast_tiles_for(b.span);
    init_reads_kernel<<<grid_cap(max(b.n_reads, n_tiles), 256, sm_count * 8), 256, 0, st>>>(
        b, n_tiles, sc.wit_min, sc.wit_max, seq_flag, fixups, sc.seq_count, sc.cursor, sc.tile_read0);
    return 1;
}

int launch_build_seq_list(const DevBatch& b, Scratch& sc, uint32_t* seq_flag, int force_all, int sm_count,
                          cudaStream_t st) {
    build_seq_list_kernel<<<grid_cap(b.n_reads, 256, sm_count * 8), 256, 0, st>>>(
        b, sc.wit_min, sc.wit_max, seq_flag, force_all, sc.seq_list, sc.seq_sbase, sc.seq_count, sc.cursor, sc.gen_cap,
        sc.status, sc.counters);
    return 1;
}

int launch_rank_events(const DevBatch& b, Scratch& sc, uint64_t* ev_off, int sm_count, cudaStream_t st) {
    const uint32_t n_tiles = fast_tiles_for(b.span);
    count_tile_bits_kernel<<<grid_cap((uint64_t)n_tiles * 32, 256, sm_count * 8), 256, 0, st>>>(sc.bitmap, n_tiles,
                                                                                               sc.tile_cnt);
    int n = 1 + launch_scan_u32(sc.tile_cnt, n_tiles, sc.tile_base, reinterpret_cast<uint64_t*>(sc.counters.get()), sc,
                                st);
    read_event_offsets_kernel<<<grid_cap((uint64_t)b.n_reads + 1, 256, sm_count * 8), 256, 0, st>>>(
        b, sc.bitmap, sc.tile_base, n_tiles, ev_off);
    return n + 1;
}

}  // namespace sgpu
