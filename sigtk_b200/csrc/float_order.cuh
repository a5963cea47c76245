// float_order.cuh -- sequential FLOAT accumulation (the reference's meanf / stdvf loops, stat.h:17-44) reproduced
// bit for bit by a whole warp: shared by stat.cu (`sigtk stat`, the jnn band) and prefix.cu (`sigtk prefix`).
#pragma once
#include "common.cuh"

namespace sgpu {

// ---- sequential float accumulation, in parallel ----------------------------------------------------------------------
// The reference adds in float, one value after the other: s <- fl(s + v). While s stays in one binade [2^e, 2^(e+1))
// every s is an integer multiple S of g = 2^(e-23), and for v >= 0
//     fl(s + v) = g * RNE(S + v/g) = g * (S + a + c),   v/g = a + f,  a = floor, 0 <= f < 1,
//     c = [f > 1/2], and on a tie (f == 1/2) c = parity of (S + a):
// the only thing the step needs to know about the running sum is the PARITY of S. So a run of values is summarised by
// two integers -- the total increment for an even and for an odd incoming S -- computed without knowing s, and runs
// compose. One warp takes 1024 values: every lane summarises 32 consecutive ones (both parities), a shuffle scan
// composes the 32 summaries (lane 0 used to walk them one by one: a quarter of the kernel's time). A tile that would carry S to 2^24 (the binade ends there), holds a negative value or meets s <= 0 is
// added value by value; the summaries after it are recomputed for the new binade. Bit-identical to the sequential
// loop by construction (tests: every stat of every parity test and of the fuzz reads against the oracle).
constexpr int SB = 1024;            // values per superblock
constexpr int SB_STRIDE = 33;       // shared-memory row stride of a 32-value tile (conflict-free both ways)

// one lane, one tile of 32 values (row), the accumulator's binade given as scale = 2^(23-e): the increment of the
// mantissa integer S for an even (u0) and for an odd (u1) incoming S; false when the tile cannot be summarised.
// Scaled by 2^(23-e) the accumulator is an integer-valued float in [2^23, 2^24), where one ulp is 1: the hardware's own
// float addition IS the recurrence (round to nearest, ties to even), so the run is simply added up twice, from the
// smallest even and the smallest odd accumulator of the binade. Both stay below 2^24 (checked at the end: the sums
// only grow), or the tile is handed to the value-by-value path.
__device__ __forceinline__ bool tile_summary(const float* __restrict__ row, float scale, uint32_t& u0, uint32_t& u1) {
    float acc0 = 8388608.0f, acc1 = 8388609.0f;
    uint32_t sign = 0u;
#pragma unroll 8
    for (int k = 0; k < 32; k++) {
        const float v = row[k];
        const float x = __fmul_rn(v, scale);          // exact: a power of two
        sign |= __float_as_uint(v);
        acc0 = __fadd_rn(acc0, x);
        acc1 = __fadd_rn(acc1, x);
    }
    u0 = __float_as_uint(acc0) - 0x4b000000u;         // mantissa integers: exact differences
    u1 = __float_as_uint(acc1) - 0x4b000001u;
    return ((sign >> 31) == 0u) && (acc0 < 16777216.0f) && (acc1 < 16777216.0f);  // (NaN / infinity: not ok)
}

// the summaries compose (the parity after a tile is the parity of S + its increment): an inclusive scan over the
// lanes gives the increment from the first summarised tile through every tile for either incoming parity.
// (32-bit wrap-around can only happen after the first tile that ends the binade, which is all that is used.)
__device__ __forceinline__ void compose_summaries(uint32_t& u0, uint32_t& u1, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t b0 = __shfl_up_sync(0xffffffffu, u0, d), b1 = __shfl_up_sync(0xffffffffu, u1, d);
        if (lane >= d) {
            const uint32_t n0 = b0 + ((b0 & 1u) ? u1 : u0);
            const uint32_t n1 = b1 + ((b1 & 1u) ? u0 : u1);
            u0 = n0; u1 = n1;
        }
    }
}

__device__ __forceinline__ bool summable(float s) {   // an accumulator whose binade can be worked in
    const int e = (int)((__float_as_uint(s) >> 23) & 0xffu) - 127;
    return s > 0.0f && e > -100 && e < 100;
}

__device__ __forceinline__ float chain_superblock(const float* __restrict__ A, int ntiles, float s, int lane, bool first) {
    int tile = 0;
    while (tile < ntiles) {  // (uniform across the warp)
        const uint32_t sb = __float_as_uint(s);
        const int e = (int)((sb >> 23) & 0xffu) - 127;
        const bool s_ok = !first && summable(s);  // the first superblock starts from 0: binades fly by
        int fail = tile;  // first tile that has to be added value by value
        uint32_t S = (sb & 0x7fffffu) | 0x800000u;
        if (s_ok) {
            const float scale = __uint_as_float((uint32_t)(127 + 23 - e) << 23);
            // every lane summarises one tile
            uint32_t u0 = 0u, u1 = 0u;  // lanes outside [tile, ntiles) are the identity
            bool ok = true;
            if (lane >= tile && lane < ntiles) ok = tile_summary(A + lane * SB_STRIDE, scale, u0, u1);
            compose_summaries(u0, u1, lane);
            const uint32_t S_after = S + ((S & 1u) ? u1 : u0);
            const uint32_t bad = __ballot_sync(0xffffffffu, !ok || S_after >= 0x1000000u);
            fail = bad ? __ffs(bad) - 1 : ntiles;  // the first tile that has to be added value by value
            if (fail > tile) S = __shfl_sync(0xffffffffu, S_after, fail - 1);
            s = __uint_as_float(((uint32_t)(e + 127) << 23) | (S & 0x7fffffu));
            __syncwarp();
        }
        if (fail < ntiles) {
            if (lane == 0) {
                const float* row = A + fail * SB_STRIDE;
#pragma unroll
                for (int k = 0; k < 32; k++) s = __fadd_rn(s, row[k]);
            }
            s = __shfl_sync(0xffffffffu, s, 0);
            tile = fail + 1;
        } else {
            tile = ntiles;
        }
    }
    return s;
}

// The summary of a whole superblock in the binade of `s` (summable(s) holds): what its tiles add to S for an even
// (U0) and an odd (U1) incoming S -- valid as long as S stays below 2^24 to the superblock's end (the values are
// non-negative, so S only grows: the caller checks the end). Superblocks summarised in the same binade compose like
// tiles do: several warps take consecutive superblocks of one long read (stat_moments_cta_kernel).
__device__ __forceinline__ bool summarise_superblock(const float* __restrict__ A, int ntiles, float s, int lane,
                                                     uint32_t& U0, uint32_t& U1) {
    const int e = (int)((__float_as_uint(s) >> 23) & 0xffu) - 127;
    const float scale = __uint_as_float((uint32_t)(127 + 23 - e) << 23);
    uint32_t u0 = 0u, u1 = 0u;
    bool ok = true;
    if (lane < ntiles) ok = tile_summary(A + lane * SB_STRIDE, scale, u0, u1);
    compose_summaries(u0, u1, lane);
    U0 = __shfl_sync(0xffffffffu, u0, 31);   // lanes past the last tile are the identity
    U1 = __shfl_sync(0xffffffffu, u1, 31);
    return __ballot_sync(0xffffffffu, !ok) == 0u;
}


// ---- signed values: the first pass over the caller's pA floats ---------------------------------------------------------
// Values of either sign, accumulators of either sign. fl(s + v) = -fl(-s - v), so an accumulator s < 0 is worked as -s
// with every value negated (the scale carries the sign). Inside the binade of |s| the step is the same integer
// recurrence as above, S <- RNE(S + x) with x = v * scale, now with x of either sign, and it still depends on nothing
// but the parity of S -- as long as every exact S + x lies in [2^23, 2^24]. A run can no longer be checked by where it
// ends (S goes down as well as up), so a summary also carries the lowest (lo) and highest (hi) point of the path
// relative to its start. The run is added up by the hardware from the middle of the binade, P = 1.5 * 2^23 (even) and
// P + 1 (odd): while every rounded point of that path lies strictly inside (2^23, 2^24) each exact sum lay in
// [2^23, 2^24) (rounding is monotone and both ends are floats), where float rounding is the integer recurrence. The
// path from the real S follows it shifted by S - P; it is exact while S + lo >= 2^23 + 1 and S + hi <= 2^24 - 1
// (every exact sum then lies within 1/2 of such a point, inside the binade). The path from P can reach 2^22 either
// way, so only a tile that moves the accumulator by more than a quarter of its magnitude, or that meets a NaN or an
// infinity, cannot be summarised; a run that would leave the binade of S (zero, a power of two) is added value by value.
constexpr int SGN_FAR = 1 << 28;    // lo of a run without a point (the identity); larger than any summarised path

struct SgnSum { int inc[2], lo[2], hi[2]; };  // [parity of the incoming S]: increment, lowest and highest point

__device__ __forceinline__ SgnSum sgn_identity() { return SgnSum{{0, 0}, {SGN_FAR, SGN_FAR}, {-SGN_FAR, -SGN_FAR}}; }

// one lane, one tile of 32 values; scale = +-2^(23-e) (the sign of the accumulator); false when it cannot be summarised
__device__ __forceinline__ bool tile_summary_signed(const float* __restrict__ row, float scale, SgnSum& u) {
    constexpr float P = 12582912.0f;                  // 1.5 * 2^23
    float acc0 = P, acc1 = P + 1.0f;
    float lo0 = 16777216.0f, lo1 = 16777216.0f, hi0 = 8388608.0f, hi1 = 8388608.0f;
#pragma unroll 8
    for (int k = 0; k < 32; k++) {
        const float x = __fmul_rn(row[k], scale);     // exact, or below 2^-126: too small to move S either way
        acc0 = __fadd_rn(acc0, x);
        acc1 = __fadd_rn(acc1, x);
        lo0 = fminf(lo0, acc0); hi0 = fmaxf(hi0, acc0);
        lo1 = fminf(lo1, acc1); hi1 = fmaxf(hi1, acc1);
    }
    // (a NaN stays NaN to the end and fails the first two tests; an infinity fails the bounds)
    const bool ok = acc0 > 8388608.0f && acc1 > 8388608.0f && lo0 > 8388608.0f && lo1 > 8388608.0f &&
                    hi0 < 16777216.0f && hi1 < 16777216.0f;
    if (!ok) { u = sgn_identity(); return false; }
    u.inc[0] = (int)acc0 - 12582912; u.lo[0] = (int)lo0 - 12582912; u.hi[0] = (int)hi0 - 12582912;
    u.inc[1] = (int)acc1 - 12582913; u.lo[1] = (int)lo1 - 12582913; u.hi[1] = (int)hi1 - 12582913;
    return true;
}

// b after a: the run of a, then the run of b from the parity a leaves
__device__ __forceinline__ SgnSum sgn_then(const SgnSum& a, const SgnSum& b) {
    SgnSum c;
#pragma unroll
    for (int p = 0; p < 2; p++) {
        const int d = a.inc[p], q = (p ^ d) & 1;
        c.inc[p] = d + b.inc[q];
        c.lo[p] = min(a.lo[p], d + b.lo[q]);
        c.hi[p] = max(a.hi[p], d + b.hi[q]);
    }
    return c;
}

// whether the run u keeps the path from S strictly inside the binade
__device__ __forceinline__ bool sgn_fits(const SgnSum& u, uint32_t S) {
    const int p = (int)(S & 1u);
    return (int)S + u.lo[p] >= 0x800001 && (int)S + u.hi[p] <= 0xffffff;
}

__device__ __forceinline__ void compose_signed(SgnSum& u, int lane) {   // inclusive scan over the lanes
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        SgnSum a;
#pragma unroll
        for (int p = 0; p < 2; p++) {
            a.inc[p] = __shfl_up_sync(0xffffffffu, u.inc[p], d);
            a.lo[p] = __shfl_up_sync(0xffffffffu, u.lo[p], d);
            a.hi[p] = __shfl_up_sync(0xffffffffu, u.hi[p], d);
        }
        if (lane >= d) u = sgn_then(a, u);
    }
}

__device__ __forceinline__ bool summable_signed(float s) { return summable(fabsf(s)); }

// the scale of the binade of s, negative for s < 0
__device__ __forceinline__ float signed_scale(float s) {
    const uint32_t sb = __float_as_uint(s);
    const int e = (int)((sb >> 23) & 0xffu) - 127;
    return __uint_as_float(((uint32_t)(127 + 23 - e) << 23) | (sb & 0x80000000u));
}

// chain_superblock for addends of either sign
__device__ __forceinline__ float chain_superblock_signed(const float* __restrict__ A, int ntiles, float s, int lane,
                                                        bool first) {
    int tile = 0;
    while (tile < ntiles) {  // (uniform across the warp)
        int fail = tile;
        if (!first && summable_signed(s)) {
            const uint32_t sb = __float_as_uint(s);
            uint32_t S = (sb & 0x7fffffu) | 0x800000u;
            SgnSum u = sgn_identity();  // lanes outside [tile, ntiles) are the identity
            bool ok = true;
            if (lane >= tile && lane < ntiles) ok = tile_summary_signed(A + lane * SB_STRIDE, signed_scale(s), u);
            compose_signed(u, lane);
            const uint32_t S_after = S + (uint32_t)u.inc[S & 1u];
            const uint32_t bad = __ballot_sync(0xffffffffu, !ok || !sgn_fits(u, S));
            fail = bad ? __ffs(bad) - 1 : ntiles;
            if (fail > tile) S = __shfl_sync(0xffffffffu, S_after, fail - 1);
            s = __uint_as_float((sb & 0xff800000u) | (S & 0x7fffffu));
            __syncwarp();
        }
        if (fail < ntiles) {
            if (lane == 0) {
                const float* row = A + fail * SB_STRIDE;
#pragma unroll
                for (int k = 0; k < 32; k++) s = __fadd_rn(s, row[k]);
            }
            s = __shfl_sync(0xffffffffu, s, 0);
            tile = fail + 1;
        } else {
            tile = ntiles;
        }
    }
    return s;
}

// summarise_superblock for addends of either sign (summable_signed(s) holds); the caller checks sgn_fits
__device__ __forceinline__ bool summarise_superblock_signed(const float* __restrict__ A, int ntiles, float s, int lane,
                                                            SgnSum& U) {
    SgnSum u = sgn_identity();
    bool ok = true;
    if (lane < ntiles) ok = tile_summary_signed(A + lane * SB_STRIDE, signed_scale(s), u);
    compose_signed(u, lane);
#pragma unroll
    for (int p = 0; p < 2; p++) {
        U.inc[p] = __shfl_sync(0xffffffffu, u.inc[p], 31);
        U.lo[p] = __shfl_sync(0xffffffffu, u.lo[p], 31);
        U.hi[p] = __shfl_sync(0xffffffffu, u.hi[p], 31);
    }
    return __ballot_sync(0xffffffffu, !ok) == 0u;
}


constexpr int MED_BINS = 4096;
// element of rank `rank` (0-based, ascending) of the int16 samples raw[0..n); all threads of the CTA (256 or more) call it.
// ALIGNED: raw is 16-byte aligned (a read's first sample: 128-bit loads); otherwise any sub-range of a read.
// Two levels over the order-preserving key raw + 32768: the upper 12 bits (4096 bins: the ~1,000 ADC units a signal
// spans spread over ~60 bins, so the shared-memory atomics of a warp rarely meet; with 256 bins they met on 2-4 bins),
// then the lower 4 bits among the samples of the selected bin. 128-bit loads (the read starts 16-byte aligned).
// one 128-bit word (8 samples, `cnt` of them inside the read) into the level-1 histogram: two keys per register,
// key = raw + 32768 = raw ^ 0x8000 as 16 bits, bin = key >> 4
__device__ __forceinline__ void med_count_word(const uint4& q, uint32_t cnt, uint32_t* hist) {
    const uint32_t wd[4] = {q.x, q.y, q.z, q.w};
    if (cnt >= 8u) {
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t x = wd[j] ^ 0x80008000u;
            atomicAdd(&hist[(x >> 4) & 0xfffu], 1u);
            atomicAdd(&hist[x >> 20], 1u);
        }
    } else {
#pragma unroll
        for (int h = 0; h < 8; h++) {
            const uint32_t key = ((wd[h >> 1] >> ((h & 1) * 16)) & 0xffffu) ^ 0x8000u;
            if ((uint32_t)h < cnt) atomicAdd(&hist[key >> 4], 1u);
        }
    }
}
// level 2: the low 4 bits of the samples whose upper 12 bits equal those of `pattern` (both halves hold the bin's
// first raw value). A register with no matching half -- nearly all of them -- is dismissed by one zero-halfword test.
__device__ __forceinline__ void med_match_word(const uint4& q, uint32_t cnt, uint32_t pattern, uint32_t* part) {
    const uint32_t wd[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const uint32_t x = wd[j] ^ pattern;
        const uint32_t m = x & 0xfff0fff0u;
        if (((m - 0x00010001u) & ~m & 0x80008000u) != 0u) {   // some halfword of m may be zero (exact test below)
            if ((m & 0xffffu) == 0u && (uint32_t)(2 * j) < cnt) atomicAdd(&part[x & 15u], 1u);
            if ((m >> 16) == 0u && (uint32_t)(2 * j + 1) < cnt) atomicAdd(&part[(x >> 16) & 15u], 1u);
        }
    }
}

template <bool ALIGNED>
__device__ int select_rank_i16(const int16_t* __restrict__ raw, uint32_t n, uint32_t rank, uint32_t* hist,
                               uint32_t* part, uint32_t* sh) {
    const uint4* __restrict__ src = reinterpret_cast<const uint4*>(raw);
    const uint32_t n_words = (n + 7u) >> 3;
    for (int k = threadIdx.x; k < MED_BINS; k += blockDim.x) hist[k] = 0;
    __syncthreads();
    if (ALIGNED) {
        // four 128-bit loads in flight per thread (a CTA's bandwidth is its bytes in flight over the load latency)
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
                if (w < n_words) med_count_word(q[k], n - w * 8u, hist);
            }
        }
    } else {
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x)
            atomicAdd(&hist[(uint32_t)((int)__ldg(raw + i) + 32768) >> 4], 1u);
    }
    __syncthreads();
    if (threadIdx.x < 256) {   // 256 threads x 16 bins
        uint32_t sum = 0;
        for (int k = 0; k < MED_BINS / 256; k++) sum += hist[threadIdx.x * (MED_BINS / 256) + k];
        part[threadIdx.x] = sum;
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        // the first warp finds the bin of the rank: every lane adds up 8 of the 256 partial sums, a shuffle scan
        // places the rank in one lane's group, and that lane walks its 8 partial sums and then the 16 bins
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
        const uint32_t owner = __ballot_sync(0xffffffffu, incl > rank);   // (rank < n: never empty)
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
    const uint32_t hi = sh[0], rank2 = sh[1];
    __syncthreads();
    // level 2: the low 4 bits among the samples whose upper 12 bits matched
    if (threadIdx.x < 16) part[threadIdx.x] = 0;
    __syncthreads();
    if (ALIGNED) {
        const uint32_t first = ((hi << 4) ^ 0x8000u) & 0xffffu;   // the bin's first raw value (16-bit pattern)
        const uint32_t pattern = first | (first << 16);
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
                if (w < n_words) med_match_word(q[k], n - w * 8u, pattern, part);
            }
        }
    } else {
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
            const uint32_t key = (uint32_t)((int)__ldg(raw + i) + 32768);
            if ((key >> 4) == hi) atomicAdd(&part[key & 15u], 1u);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t seen = 0, k = 0;
        for (; k < 16; k++) {
            if (seen + part[k] > rank2) break;
            seen += part[k];
        }
        sh[2] = k;
    }
    __syncthreads();
    const int med = (int)((hi << 4) | sh[2]) - 32768;
    __syncthreads();
    return med;
}


}  // namespace sgpu
