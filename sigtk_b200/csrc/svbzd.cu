// svbzd.cu -- svb-zd signal streams of BLOW5 records decoded in HBM (SURVEY 8f rank 1), so that only the compressed
// bytes cross PCIe. Replaces, per batch, what slow5lib does per record on the CPU:
//   ptr_depress_svb_zd / ptr_depress_svb            /root/reference/slow5lib/src/slow5_press.c:1091-1150
//   svb_decode_scalar / _decode_data                 thirdparty/streamvbyte/src/streamvbyte_decode.c:30-83
//   __slow5_zigzag_delta_decode                      thirdparty/streamvbyte/src/streamvbyte_zigzag.c:27-47
//
// Stream of one read:  uint32 count | ceil(count/4) key bytes (2 bits per value, low bits first) | data bytes;
// value i takes code_i + 1 little-endian bytes and is zigzag(raw[i] - raw[i-1]) in 32-bit arithmetic, raw[-1] = 0.
// Both the position of a value's bytes (sum of the lengths before it) and the sample itself (sum of the deltas
// before it) are prefix sums over the read, so the decode is three streaming passes over BLOCKS of 1024 values
// (one warp per block, one lane per 32 values = 64 key bits):
//   1. svb_bytes_kernel   data bytes per block from the keys alone (popcounts)         -> scan -> block data offsets
//   2. svb_sums_kernel    every lane walks its 32 values: sum of its deltas; block sums -> scan -> block start values;
//                         the last block of a read checks the stream length (slow5_press.c:1103)
//   3. svb_write_kernel   every lane walks its 32 values again from its exact start value and writes 64 aligned bytes
// All arithmetic is integer: results are bit-identical by construction, and checked against the oracle and the
// reference's own slow5lib in tests/test_gpu_svbzd.py.
//
// The encoder (SGPU_WANT_SVBZD, sgpu_encode_svbzd_device) writes what slow5lib's ptr_compress_svb_zd (slow5_press.c;
// streamvbyte_encode.c, streamvbyte_zigzag.c) writes, on the same block map; every stream starts on a 16-byte boundary:
//   1. svbe_bytes_kernel  every lane forms the zigzag deltas of its 32 samples: data bytes per block -> scan
//   2. svbe_len_kernel    stream length per read, 4 + ceil(n/4) + data, in 16-byte units -> scan -> comp_off;
//      svbe_head_kernel   the count header and the zero padding up to the boundary
//   3. svbe_write_kernel  key bytes at fixed offsets, data bytes staged per block in shared memory and written as
//                         whole words inside the block's range (byte stores at its edges)
// Checked byte for byte against the reference's slow5lib in tests/test_gpu_svbzd_encode.py.
#include "kernels.cuh"

namespace sgpu {

namespace {

constexpr int SVB_BLOCK = 1024;  // values per warp block
constexpr int SVB_WARPS = 4;

struct SvbBlock {
    uint32_t r;        // read
    uint32_t k;        // block index inside the read
    uint32_t n;        // values in the read
    uint32_t nv;       // valid values of this lane (0..32)
    uint64_t keys64;   // this lane's 32 two-bit codes (invalid ones cleared)
    uint64_t stream;   // byte offset of the read's stream in the batch buffer
    uint64_t key_len;  // key bytes of the read
};

__device__ __forceinline__ uint32_t find_block_read(const uint64_t* __restrict__ base, uint32_t n_reads, uint64_t b) {
    uint32_t lo = 0, hi = n_reads;  // largest r with base[r] <= b (base[n_reads] > b)
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (base[mid] <= b) lo = mid; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ SvbBlock load_block(const SvbBatch& s, const uint64_t* __restrict__ base, uint64_t b, int lane,
                                               uint32_t r) {
    SvbBlock q;
    q.r = r;
    q.k = (uint32_t)(b - base[q.r]);
    q.n = s.read_len[q.r];
    q.stream = s.comp_off[q.r];
    q.key_len = ((uint64_t)q.n + 3u) >> 2;
    const uint64_t i0 = (uint64_t)q.k * SVB_BLOCK + (uint64_t)lane * 32u;
    q.nv = i0 >= q.n ? 0u : (q.n - i0 >= 32u ? 32u : (uint32_t)(q.n - i0));
    q.keys64 = 0;
    if (q.nv) {
        // the stream starts on a 16-byte boundary and the keys 4 bytes later: key words are aligned; a word that
        // straddles the end of the keys also holds data bytes (inside the stream or the buffer's slack), masked below
        const uint32_t* __restrict__ kw = reinterpret_cast<const uint32_t*>(s.bytes + q.stream + 4u) + (i0 >> 4);
        const uint32_t w0 = __ldg(kw), w1 = q.nv > 16u ? __ldg(kw + 1) : 0u;
        q.keys64 = (uint64_t)w0 | ((uint64_t)w1 << 32);
        if (q.nv < 32u) q.keys64 &= (1ull << (2u * q.nv)) - 1ull;
    }
    return q;
}

// data bytes of a lane's values: one byte each plus the sum of the codes
__device__ __forceinline__ uint32_t lane_bytes(const SvbBlock& q) {
    return q.nv + (uint32_t)__popcll(q.keys64 & 0x5555555555555555ull) +
           2u * (uint32_t)__popcll(q.keys64 & 0xaaaaaaaaaaaaaaaaull);
}

__device__ __forceinline__ uint32_t warp_excl_scan(uint32_t v, int lane, uint32_t* total) {
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    *total = __shfl_sync(0xffffffffu, inc, 31);
    return inc - v;
}

constexpr int SVB_STAGE_WORDS = SVB_BLOCK + 4;  // a block's data: at most 4 bytes per value, plus alignment slack

// copies the data bytes [start, start + n_bytes) of one block into the warp's shared-memory stage (aligned words,
// coalesced) and returns the byte offset of `start` inside the stage
__device__ __forceinline__ uint32_t stage_block(const SvbBatch& s, uint64_t start, uint32_t n_bytes, uint32_t* stage, int lane) {
    const uint32_t* __restrict__ words = reinterpret_cast<const uint32_t*>(s.bytes);
    const uint64_t last_word = (s.n_bytes >> 2) + 1u;  // the buffer carries 8 bytes of slack
    const uint64_t w0 = start >> 2;
    const uint32_t lead = (uint32_t)start & 3u;
    const uint32_t n_words = (lead + n_bytes + 3u) / 4u + 1u;  // one more: the last value's fetch reads a word pair
    __syncwarp();  // the previous block's readers are done
    for (uint32_t k = lane; k < n_words; k += 32) {
        uint64_t wi = w0 + k;
        if (wi > last_word) wi = last_word;  // malformed stream: stay inside the buffer (the length check reports it)
        stage[k] = __ldg(words + wi);
    }
    __syncwarp();
    return lead;
}

// walks the valid values of one lane from the staged bytes; f(j, delta) receives the zigzag-decoded delta of value j
template <class F>
__device__ __forceinline__ void walk_lane(const SvbBlock& q, const uint32_t* stage, uint32_t at, F f) {
    const uint32_t klo = (uint32_t)q.keys64, khi = (uint32_t)(q.keys64 >> 32);
#pragma unroll
    for (uint32_t j = 0; j < 32u; j++) {  // unrolled: every index below is static
        if (j >= q.nv) break;
        const uint32_t code = ((j < 16u ? klo : khi) >> (2u * (j & 15u))) & 3u;
        const uint32_t i = at >> 2;
        const uint32_t z = __funnelshift_r(stage[i], stage[i + 1], (at & 3u) * 8u) & (0xffffffffu >> (24u - 8u * code));
        f(j, (z >> 1) ^ (0u - (z & 1u)));  // streamvbyte_zigzag.c:27-29
        at += code + 1u;
    }
}

__global__ void __launch_bounds__(256) svb_count_kernel(const uint32_t* __restrict__ read_len, uint32_t n_reads,
                                                        uint32_t* __restrict__ cnt) {
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < n_reads; r += gridDim.x * blockDim.x)
        cnt[r] = (read_len[r] + SVB_BLOCK - 1) / SVB_BLOCK;
}

__global__ void __launch_bounds__(SVB_WARPS * 32) svb_bytes_kernel(SvbBatch s, const uint64_t* __restrict__ base,
                                                                   uint32_t* __restrict__ blk_bytes,
                                                                   uint32_t* __restrict__ blk_read) {
    const int lane = threadIdx.x & 31;
    const uint64_t n_blocks = base[s.n_reads];
    for (uint64_t b = (uint64_t)blockIdx.x * SVB_WARPS + (threadIdx.x >> 5); b < n_blocks; b += (uint64_t)gridDim.x * SVB_WARPS) {
        const SvbBlock q = load_block(s, base, b, lane, find_block_read(base, s.n_reads, b));
        const uint32_t tot = __reduce_add_sync(0xffffffffu, lane_bytes(q));
        if (lane == 0) { blk_bytes[b] = tot; blk_read[b] = q.r; }  // the later passes reuse the block -> read map
    }
}

__global__ void __launch_bounds__(SVB_WARPS * 32) svb_sums_kernel(SvbBatch s, const uint64_t* __restrict__ base,
                                                                  const uint64_t* __restrict__ blk_gpos,
                                                                  const uint32_t* __restrict__ blk_read,
                                                                  uint32_t* __restrict__ lane_sum,
                                                                  uint32_t* __restrict__ blk_sum, int* __restrict__ status) {
    __shared__ uint32_t stage_all[SVB_WARPS][SVB_STAGE_WORDS];
    uint32_t* stage = stage_all[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    const uint64_t n_blocks = base[s.n_reads];
    for (uint64_t b = (uint64_t)blockIdx.x * SVB_WARPS + (threadIdx.x >> 5); b < n_blocks; b += (uint64_t)gridDim.x * SVB_WARPS) {
        const SvbBlock q = load_block(s, base, b, lane, blk_read[b]);
        uint32_t blk_total;
        const uint32_t before = warp_excl_scan(lane_bytes(q), lane, &blk_total);
        const uint64_t boff = blk_gpos[b] - blk_gpos[base[q.r]];  // data bytes of the read before this block
        const uint32_t lead = stage_block(s, q.stream + 4u + q.key_len + boff, blk_total, stage, lane);
        uint32_t sum = 0;
        walk_lane(q, stage, lead + before, [&](uint32_t, uint32_t d) { sum += d; });
        lane_sum[b * 32 + lane] = sum;
        const uint32_t tot = __reduce_add_sync(0xffffffffu, sum);
        if (lane == 0) {
            blk_sum[b] = tot;
            // the stream must end exactly where its last value ends (slow5_press.c:1103)
            if ((uint64_t)(q.k + 1) * SVB_BLOCK >= q.n && 4u + q.key_len + boff + blk_total != s.comp_len[q.r])
                atomicExch(status, SGPU_DEV_E_STREAM);
        }
    }
}

__global__ void __launch_bounds__(SVB_WARPS * 32) svb_write_kernel(SvbBatch s, const uint64_t* __restrict__ base,
                                                                   const uint64_t* __restrict__ blk_gpos,
                                                                   const uint32_t* __restrict__ blk_read,
                                                                   const uint32_t* __restrict__ lane_sum,
                                                                   const uint64_t* __restrict__ blk_vpos,
                                                                   int16_t* __restrict__ samples) {
    __shared__ uint32_t stage_all[SVB_WARPS][SVB_STAGE_WORDS];
    uint32_t* stage = stage_all[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    const uint64_t n_blocks = base[s.n_reads];
    for (uint64_t b = (uint64_t)blockIdx.x * SVB_WARPS + (threadIdx.x >> 5); b < n_blocks; b += (uint64_t)gridDim.x * SVB_WARPS) {
        const SvbBlock q = load_block(s, base, b, lane, blk_read[b]);
        uint32_t blk_total, unused;
        const uint32_t before = warp_excl_scan(lane_bytes(q), lane, &blk_total);
        const uint32_t vbefore = warp_excl_scan(lane_sum[b * 32 + lane], lane, &unused);
        const uint64_t boff = blk_gpos[b] - blk_gpos[base[q.r]];
        // value of the sample before this lane's first one: 32-bit wrap-around like the reference's int32 `prev`
        uint32_t prev = (uint32_t)(blk_vpos[b] - blk_vpos[base[q.r]]) + vbefore;
        const uint32_t lead = stage_block(s, q.stream + 4u + q.key_len + boff, blk_total, stage, lane);
        uint32_t w[16];
#pragma unroll
        for (int t = 0; t < 16; t++) w[t] = 0u;
        walk_lane(q, stage, lead + before, [&](uint32_t j, uint32_t d) {
            prev += d;                                   // streamvbyte_zigzag.c:44-45; the int16 store truncates
            w[j >> 1] |= (prev & 0xffffu) << (16u * (j & 1u));   // j is a compile-time constant after unrolling
        });
        if (q.nv) {
            int16_t* dst = samples + s.read_off[q.r] + (uint64_t)q.k * SVB_BLOCK + (uint64_t)lane * 32u;
            if (q.nv == 32u) {  // read_off is a multiple of 8 samples: 16-byte aligned
                int4* d4 = reinterpret_cast<int4*>(dst);
#pragma unroll
                for (int t = 0; t < 4; t++) d4[t] = make_int4((int)w[4 * t], (int)w[4 * t + 1], (int)w[4 * t + 2], (int)w[4 * t + 3]);
            } else {
#pragma unroll
                for (uint32_t j = 0; j < 32u; j++)  // static indices keep w[] in registers
                    if (j < q.nv) dst[j] = (int16_t)(w[j >> 1] >> (16u * (j & 1u)));
            }
        }
    }
}

// ---- encoder: int16 samples -> the streams slow5lib stores, on the decoder's block map --------------------------------
// For int16 input |d| <= 65535, so z <= 131070 < 2^24: every value takes 1 to 3 bytes, never 4.

struct EncBlock {
    uint32_t r;   // read
    uint32_t k;   // block index inside the read
    uint32_t n;   // values in the read
    uint32_t nv;  // valid values of this lane (0..32)
};

__device__ __forceinline__ EncBlock enc_block(const DevBatch& b, const uint64_t* __restrict__ base, uint64_t blk, int lane,
                                              uint32_t r) {
    EncBlock q;
    q.r = r;
    q.k = (uint32_t)(blk - base[r]);
    q.n = b.read_len[r];
    const uint64_t i0 = (uint64_t)q.k * SVB_BLOCK + (uint64_t)lane * 32u;
    q.nv = i0 >= q.n ? 0u : (q.n - i0 >= 32u ? 32u : (uint32_t)(q.n - i0));
    return q;
}

// z[j] = zigzag(raw[i] - raw[i-1]) of the lane's value j in 32-bit arithmetic, raw[-1] = 0 (streamvbyte_zigzag.c:5-25);
// 0 past q.nv. Called by the whole warp.
__device__ __forceinline__ void lane_zigzag(const DevBatch& b, const EncBlock& q, int lane, uint32_t (&z)[32]) {
    const int16_t* __restrict__ src = b.samples + b.read_off[q.r] + (uint64_t)q.k * SVB_BLOCK + (uint64_t)lane * 32u;
    uint32_t w[16];
    // read_off is a multiple of 8 samples and a lane starts on a multiple of 32: aligned 16-byte loads, the last one
    // inside the read's padding to 8 samples
#pragma unroll
    for (int t = 0; t < 4; t++) {
        int4 v = make_int4(0, 0, 0, 0);
        if ((uint32_t)(8 * t) < q.nv) v = __ldg(reinterpret_cast<const int4*>(src) + t);
        w[4 * t] = (uint32_t)v.x; w[4 * t + 1] = (uint32_t)v.y; w[4 * t + 2] = (uint32_t)v.z; w[4 * t + 3] = (uint32_t)v.w;
    }
    // the sample before the lane's first: the previous lane's last (full whenever this lane has values), before the
    // block's first the previous block's last, 0 at the read's start
    int32_t prev = (int16_t)(__shfl_up_sync(0xffffffffu, w[15], 1) >> 16);
    if (lane == 0) prev = q.k ? (int32_t)src[-1] : 0;
#pragma unroll
    for (int j = 0; j < 32; j++) {
        const int32_t cur = (int16_t)(w[j >> 1] >> (16 * (j & 1)));
        const int32_t d = cur - prev;
        z[j] = (uint32_t)j < q.nv ? ((uint32_t)d << 1) ^ (uint32_t)(d >> 31) : 0u;
        prev = cur;
    }
}

__device__ __forceinline__ uint32_t zz_code(uint32_t z) { return (z > 0xffu) + (z > 0xffffu); }  // bytes - 1

// data bytes of a lane's values
__device__ __forceinline__ uint32_t lane_data_bytes(uint32_t nv, const uint32_t (&z)[32]) {
    uint32_t n = nv;
#pragma unroll
    for (int j = 0; j < 32; j++) n += zz_code(z[j]);
    return n;
}

// stores the low `n` bytes of v at p (4-byte aligned): one word when n == 4
__device__ __forceinline__ void store_key_word(uint8_t* p, uint32_t v, uint32_t n) {
    if (n >= 4u) {
        *reinterpret_cast<uint32_t*>(p) = v;
    } else {
        for (uint32_t t = 0; t < n; t++) p[t] = (uint8_t)(v >> (8u * t));
    }
}

// data bytes of every block (0 for the blocks between the batch's count and the host's bound max_blocks, which the
// scan covers) and the read of every block
__global__ void __launch_bounds__(SVB_WARPS * 32) svbe_bytes_kernel(DevBatch b, const uint64_t* __restrict__ base,
                                                                    uint64_t max_blocks, uint32_t* __restrict__ blk_bytes,
                                                                    uint32_t* __restrict__ blk_read) {
    const int lane = threadIdx.x & 31;
    const uint64_t n_blocks = base[b.n_reads];
    for (uint64_t k = (uint64_t)blockIdx.x * SVB_WARPS + (threadIdx.x >> 5); k < max_blocks; k += (uint64_t)gridDim.x * SVB_WARPS) {
        if (k >= n_blocks) {
            if (lane == 0) blk_bytes[k] = 0;
            continue;
        }
        const EncBlock q = enc_block(b, base, k, lane, find_block_read(base, b.n_reads, k));
        uint32_t z[32];
        lane_zigzag(b, q, lane, z);
        const uint32_t tot = __reduce_add_sync(0xffffffffu, lane_data_bytes(q.nv, z));
        if (lane == 0) { blk_bytes[k] = tot; blk_read[k] = q.r; }
    }
}

// every read's stream length 4 + ceil(n/4) + data (comp_len) and that length in 16-byte units (for the scan of comp_off)
__global__ void __launch_bounds__(256) svbe_len_kernel(DevBatch b, const uint64_t* __restrict__ base,
                                                       const uint64_t* __restrict__ blk_gpos, uint32_t* __restrict__ comp_len,
                                                       uint32_t* __restrict__ units) {
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < b.n_reads; r += gridDim.x * blockDim.x) {
        const uint64_t n = b.read_len[r];
        const uint64_t len = 4u + (n + 3u) / 4u + (blk_gpos[base[r + 1]] - blk_gpos[base[r]]);
        comp_len[r] = (uint32_t)len;  // < 2^32: the host refuses longer streams (svbzd_stream_fits)
        units[r] = (uint32_t)((len + 15u) >> 4);
    }
}

// every read: comp_off from 16-byte units to bytes, the count header, zeros from the stream's end to the boundary
__global__ void __launch_bounds__(256) svbe_head_kernel(DevBatch b, uint64_t* __restrict__ comp_off,
                                                        const uint32_t* __restrict__ comp_len, uint8_t* __restrict__ bytes) {
    for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < b.n_reads; r += gridDim.x * blockDim.x) {
        const uint64_t off = comp_off[r] << 4;
        comp_off[r] = off;
        if (r == b.n_reads - 1) comp_off[r + 1] <<= 4;
        *reinterpret_cast<uint32_t*>(bytes + off) = b.read_len[r];  // the original length leads the stream
        for (uint64_t p = off + comp_len[r]; p & 15u; p++) bytes[p] = 0;
    }
}

constexpr int SVBE_STAGE_WORDS = 3 * SVB_BLOCK / 4 + 2;  // a block's data: at most 3 bytes per value, plus alignment

// the key and data bytes of every block
__global__ void __launch_bounds__(SVB_WARPS * 32) svbe_write_kernel(DevBatch b, const uint64_t* __restrict__ base,
                                                                    const uint64_t* __restrict__ blk_gpos,
                                                                    const uint32_t* __restrict__ blk_read,
                                                                    const uint64_t* __restrict__ comp_off,
                                                                    uint8_t* __restrict__ bytes) {
    __shared__ uint32_t stage_all[SVB_WARPS][SVBE_STAGE_WORDS];
    uint32_t* stage = stage_all[threadIdx.x >> 5];
    uint8_t* sb = reinterpret_cast<uint8_t*>(stage);
    const int lane = threadIdx.x & 31;
    const uint64_t n_blocks = base[b.n_reads];
    for (uint64_t k = (uint64_t)blockIdx.x * SVB_WARPS + (threadIdx.x >> 5); k < n_blocks; k += (uint64_t)gridDim.x * SVB_WARPS) {
        const EncBlock q = enc_block(b, base, k, lane, blk_read[k]);
        uint32_t z[32];
        lane_zigzag(b, q, lane, z);
        uint32_t klo = 0, khi = 0;
#pragma unroll
        for (int j = 0; j < 32; j++) {
            if (j < 16) klo |= zz_code(z[j]) << (2 * j); else khi |= zz_code(z[j]) << (2 * (j - 16));
        }
        uint32_t blk_total;
        const uint32_t before = warp_excl_scan(lane_data_bytes(q.nv, z), lane, &blk_total);
        const uint64_t stream = comp_off[q.r];
        // keys: the lane's ceil(nv/4) key bytes, 4-byte aligned (the stream starts on a 16-byte boundary, its keys 4
        // bytes later); whole words only where every byte is one of them: the read's last key word may hold data bytes
        if (q.nv) {
            uint8_t* kp = bytes + stream + 4u + (uint64_t)q.k * (SVB_BLOCK / 4) + (uint32_t)lane * 8u;
            const uint32_t kb = (q.nv + 3u) >> 2;
            store_key_word(kp, klo, kb < 4u ? kb : 4u);
            store_key_word(kp + 4, khi, kb > 4u ? kb - 4u : 0u);
        }
        // data: staged in shared memory, then written as whole words where the block owns every byte, and byte by
        // byte in the two edge words it shares with the neighbouring block, the keys or the padding
        const uint64_t start = stream + 4u + ((uint64_t)q.n + 3u) / 4u + (blk_gpos[k] - blk_gpos[base[q.r]]);
        const uint32_t lead = (uint32_t)start & 3u;
        __syncwarp();  // the previous block's copy-out has read the stage
        uint32_t at = lead + before;
#pragma unroll
        for (uint32_t j = 0; j < 32u; j++) {
            if (j >= q.nv) break;
            const uint32_t c = zz_code(z[j]);
            sb[at] = (uint8_t)z[j];
            if (c >= 1u) sb[at + 1] = (uint8_t)(z[j] >> 8);
            if (c >= 2u) sb[at + 2] = (uint8_t)(z[j] >> 16);
            at += c + 1u;
        }
        __syncwarp();
        const uint32_t end = lead + blk_total;
        uint8_t* const dst = bytes + (start - lead);  // 4-byte aligned, stage byte t -> dst[t]
        for (uint32_t i = lane; i < (end + 3u) >> 2; i += 32) {
            if (4u * i >= lead && 4u * i + 4u <= end) {
                reinterpret_cast<uint32_t*>(dst)[i] = stage[i];
            } else {
                for (uint32_t t = 4u * i < lead ? lead : 4u * i; t < end && t < 4u * i + 4u; t++) dst[t] = sb[t];
            }
        }
    }
}

}  // namespace

uint64_t svbzd_max_blocks(uint64_t max_samples, uint32_t max_reads) { return max_samples / SVB_BLOCK + max_reads + 1; }

uint32_t svbzd_blocks_of(uint64_t n) { return (uint32_t)((n + SVB_BLOCK - 1) / SVB_BLOCK); }

int launch_svbzd_decode(const SvbBatch& s, SvbScratch& w, Scratch& sc, int16_t* samples, int sm_count, cudaStream_t st) {
    if (s.n_reads == 0 || s.n_blocks == 0) return 0;
    const uint64_t max_blocks = s.n_blocks;  // sum of ceil(read_len / 1024): the host knows every count
    svb_count_kernel<<<grid_cap(s.n_reads, 256, sm_count * 8), 256, 0, st>>>(s.read_len, s.n_reads, w.cnt);
    int n = 1 + launch_scan_u32(w.cnt, s.n_reads, w.base, nullptr, sc, st);
    const int grid = grid_cap(max_blocks, SVB_WARPS, sm_count * 16);
    svb_bytes_kernel<<<grid, SVB_WARPS * 32, 0, st>>>(s, w.base, w.blk_bytes, w.blk_read);
    n += 1 + launch_scan_u32(w.blk_bytes, (uint32_t)max_blocks, w.blk_gpos, nullptr, sc, st);
    svb_sums_kernel<<<grid, SVB_WARPS * 32, 0, st>>>(s, w.base, w.blk_gpos, w.blk_read, w.lane_sum, w.blk_sum, sc.status);
    n += 1 + launch_scan_u32(w.blk_sum, (uint32_t)max_blocks, w.blk_vpos, nullptr, sc, st);
    svb_write_kernel<<<grid, SVB_WARPS * 32, 0, st>>>(s, w.base, w.blk_gpos, w.blk_read, w.lane_sum, w.blk_vpos, samples);
    return n + 1;
}

// a read of n samples: align16(4 + ceil(n/4) + 3n) <= 3.25 n + 19.75 bytes; the 16 more give the buffer's 8 bytes of
// slack past the last stream
uint64_t svbzd_encode_capacity(uint64_t max_samples, uint32_t max_reads) {
    return (13 * max_samples + 3) / 4 + 20ull * max_reads + 16;
}

int launch_svbzd_encode(const DevBatch& b, uint8_t* bytes, uint64_t* comp_off, uint32_t* comp_len, SvbScratch& w,
                        Scratch& sc, int sm_count, cudaStream_t st) {
    if (b.n_reads == 0) {
        cudaMemsetAsync(comp_off, 0, sizeof(uint64_t), st);
        return 0;
    }
    const uint64_t max_blocks = b.span / SVB_BLOCK + b.n_reads;  // >= the batch's blocks, which only the device counts
    const int read_grid = grid_cap(b.n_reads, 256, sm_count * 8);
    const int grid = grid_cap(max_blocks, SVB_WARPS, sm_count * 16);
    svb_count_kernel<<<read_grid, 256, 0, st>>>(b.read_len, b.n_reads, w.cnt);
    int n = 1 + launch_scan_u32(w.cnt, b.n_reads, w.base, nullptr, sc, st);
    svbe_bytes_kernel<<<grid, SVB_WARPS * 32, 0, st>>>(b, w.base, max_blocks, w.blk_bytes, w.blk_read);
    n += 1 + launch_scan_u32(w.blk_bytes, (uint32_t)max_blocks, w.blk_gpos, nullptr, sc, st);
    svbe_len_kernel<<<read_grid, 256, 0, st>>>(b, w.base, w.blk_gpos, comp_len, w.cnt);  // (cnt: scanned already)
    n += 1 + launch_scan_u32(w.cnt, b.n_reads, comp_off, nullptr, sc, st);
    svbe_head_kernel<<<read_grid, 256, 0, st>>>(b, comp_off, comp_len, bytes);
    svbe_write_kernel<<<grid, SVB_WARPS * 32, 0, st>>>(b, w.base, w.blk_gpos, w.blk_read, comp_off, bytes);
    return n + 2;
}

}  // namespace sgpu
