// generic.cu -- the sequential-order ("reference-order") kernels.
//
// These kernels evaluate the reference's per-read pipeline in exactly the
// reference's operation order, so their results are bit-identical to
// src/events.c for ANY input (including reads whose FP64 prefix sums are not
// exactly representable and therefore depend on the summation order):
//
//   gen_prefix_kernel   compute_sum_sumsq          events.c:293-303  (one thread walks one read)
//   gen_tstat_kernel    compute_tstat (both w)     events.c:315-364  (one thread per sample)
//   gen_detect_kernel   short_long_peak_detector   events.c:371-443  (one thread walks one read)
//   gen_emit_kernel     create_events/create_event events.c:457-504  (one thread walks one read)
//
// They serve (a) reads that fail the exact-sum witness or the detector
// boundary-state check of the fast path (fast.cu), (b) SGPU_F_FORCE_GENERIC,
// (c) as the on-device cross-check of the fast path in the tests, and (d) batches of
// the caller's own pA floats (pa_input.cu: gen_prefix_pa_kernel, gen_detect_pa_kernel), and (e) batches with a
// caller's detector set (sgpu_set_detector: gen_detect_set_kernel, detect_set.cu).  The
// work list is built on the device (build_seq_list_kernel), so every kernel
// here is launched with a fixed grid and returns at once when the list is empty.  They keep S, Q (16 B/sample) and t1, t2 (8 B/sample) in
// an HBM scratch area, so they are NOT the roofline path.
#include "kernels.cuh"
#include "walk_core.cuh"

namespace sgpu {

// ---------------------------------------------------------------------------
// 8 consecutive samples of one read as the reference's floats: int16 raw samples through misc.c:28, or pA floats
// as the caller gave them (getevents(n, pa, rna) on the caller's own signal: pa_input.cu)
template <typename T> struct Samples8;
template <> struct Samples8<int16_t> {
    using Group = int4;  // 16 bytes
    static constexpr bool kRaw = true;
    static __device__ __forceinline__ Group zero() { return make_int4(0, 0, 0, 0); }
    static __device__ __forceinline__ Group load(const Group* p) { return __ldg(p); }
};
struct Float8 { float4 a, b; };
template <> struct Samples8<float> {
    using Group = Float8;  // 32 bytes
    static constexpr bool kRaw = false;
    static __device__ __forceinline__ Group zero() { return {make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f)}; }
    static __device__ __forceinline__ Group load(const Group* p) {
        const float4* q = reinterpret_cast<const float4*>(p);
        return {__ldg(q), __ldg(q + 1)};
    }
    static __device__ __forceinline__ void to_float(const Group& cur, float (&x)[8]) {
        x[0] = cur.a.x; x[1] = cur.a.y; x[2] = cur.a.z; x[3] = cur.a.w;
        x[4] = cur.b.x; x[5] = cur.b.y; x[6] = cur.b.z; x[7] = cur.b.w;
    }
};

// compute_sum_sumsq: Sinc[base+i] = S[i+1], Qinc[base+i] = Q[i+1]  (S[0]=Q[0]=0 implied)
// one WARP per read: lane 0 runs the two dependent chains of additions (the order IS the result), 32 samples at a
// time into shared memory (sS, sQ: [4][32]); all lanes then store the tile coalesced (32 lanes walking 32 reads would
// issue 64 store wavefronts per sample: measured 130 cycles per sample)
template <typename T>
__device__ __forceinline__ void gen_prefix_reads(const DevBatch& b, const T* samples, const WorkList& wl,
                                                 double* __restrict__ Sinc, double* __restrict__ Qinc,
                                                 double (&sS)[4][32], double (&sQ)[4][32], uint32_t n_list,
                                                 uint32_t tid) {
    using L = Samples8<T>;
    const int lane = tid & 31, wib = tid >> 5;
    const uint32_t warp = (blockIdx.x * blockDim.x + tid) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t j = warp; j < n_list; j += n_warps) {
        const uint32_t r = wl.list[j];
        const uint64_t base = wl.sbase[j];
        // reads start on 8-sample boundaries and the batch is padded to one: whole groups of 8 samples can be loaded
        const typename L::Group* __restrict__ raw8 = reinterpret_cast<const typename L::Group*>(samples + b.read_off[r]);
        const uint32_t n = b.read_len[r], n8 = (n + 7u) >> 3;
        float off = 0.0f, unit = 0.0f;
        if constexpr (L::kRaw) { off = b.offset[r]; unit = b.unit[r]; }
        double s = 0.0, q = 0.0;
        typename L::Group buf[4];  // the next tile's samples (lane 0)
        if (lane == 0) {
#pragma unroll
            for (int k = 0; k < 4; k++) buf[k] = (uint32_t)k < n8 ? L::load(raw8 + k) : L::zero();
        }
        for (uint32_t t0 = 0; t0 < n; t0 += 32) {
            if (lane == 0) {
                const uint32_t g0 = t0 >> 3;
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const typename L::Group cur = buf[k];
                    buf[k] = g0 + 4 + k < n8 ? L::load(raw8 + g0 + 4 + k) : L::zero();
                    // everything that does not depend on the running sums first (conversions pipeline), then the chain
                    float x[8];
                    if constexpr (L::kRaw) {
                        const int v[4] = {cur.x, cur.y, cur.z, cur.w};
                        walk::cvt8(v, off, unit, x);   // misc.c:28 per sample (float add, float multiply)
                    } else {
                        L::to_float(cur, x);
                    }
                    double xd[8], qd[8];
#pragma unroll
                    for (int m = 0; m < 8; m++) {
                        xd[m] = (double)x[m];
                        qd[m] = (double)__fmul_rn(x[m], x[m]);  // float product, widened afterwards (events.c:301)
                    }
#pragma unroll
                    for (int m = 0; m < 8; m++) {  // (samples past the read's end only feed values nobody stores)
                        s = __dadd_rn(s, xd[m]);
                        q = __dadd_rn(q, qd[m]);
                        sS[wib][8 * k + m] = s;
                        sQ[wib][8 * k + m] = q;
                    }
                }
            }
            __syncwarp();
            if (t0 + lane < n) {
                Sinc[base + t0 + lane] = sS[wib][lane];
                Qinc[base + t0 + lane] = sQ[wib][lane];
            }
            __syncwarp();
        }
    }
}

__global__ void __launch_bounds__(128) gen_prefix_kernel(DevBatch b, WorkList wl, double* __restrict__ Sinc,
                                                         double* __restrict__ Qinc) {
    __shared__ double sS[4][32], sQ[4][32];
    const uint32_t n_list = *wl.count;
    gen_prefix_reads<int16_t>(b, b.samples, wl, Sinc, Qinc, sS, sQ, n_list, threadIdx.x);  // (the thread index is read
                                                                                            // where its bound is known)
}

// the same on the caller's pA floats: the reads of a pA batch that fail the exact-sum witness (pa_input.cu)
__global__ void __launch_bounds__(128) gen_prefix_pa_kernel(DevBatch b, const float* __restrict__ pa, WorkList wl,
                                                            double* __restrict__ Sinc, double* __restrict__ Qinc) {
    __shared__ double sS[4][32], sQ[4][32];
    const uint32_t n_list = *wl.count;
    gen_prefix_reads<float>(b, pa, wl, Sinc, Qinc, sS, sQ, n_list, threadIdx.x);
}

// ---------------------------------------------------------------------------
__device__ __forceinline__ double prefix_at(const double* __restrict__ inc, uint64_t base, uint32_t k) {
    return k ? inc[base + k - 1] : 0.0;
}

__device__ __forceinline__ float tstat_at(const double* __restrict__ Sinc, const double* __restrict__ Qinc,
                                          uint64_t base, uint32_t n, uint32_t i, uint32_t w) {
    // events.c:328-338: zero unless w <= i <= n-w (and n >= 2w, w >= 2)
    if (n < 2u * w || w < 2u || i < w || i + w > n) return 0.0f;
    const double s_i = prefix_at(Sinc, base, i), q_i = prefix_at(Qinc, base, i);
    // i == w subtracts S[0] == 0.0, identical to the reference's "if (i > w)" branch
    const double sum1 = __dsub_rn(s_i, prefix_at(Sinc, base, i - w));
    const double ssq1 = __dsub_rn(q_i, prefix_at(Qinc, base, i - w));
    const double sum2 = __dsub_rn(prefix_at(Sinc, base, i + w), s_i);
    const double ssq2 = __dsub_rn(prefix_at(Qinc, base, i + w), q_i);
    return tstat_reference_chain(sum1, ssq1, sum2, ssq2, (float)w);
}

// p: the windows of the batch's detector (det_params(b.rna), or the caller's set: sgpu_set_detector)
__global__ void __launch_bounds__(256) gen_tstat_kernel(DevBatch b, WorkList wl, const double* __restrict__ Sinc,
                                                        const double* __restrict__ Qinc, float* __restrict__ t1,
                                                        float* __restrict__ t2, DetParams p) {
    const uint32_t n_list = *wl.count;
    for (uint32_t j = blockIdx.x; j < n_list; j += gridDim.x) {  // one CTA walks one read
        const uint32_t r = wl.list[j];
        const uint64_t base = wl.sbase[j];
        const uint32_t n = b.read_len[r];
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
            t1[base + i] = tstat_at(Sinc, Qinc, base, n, i, (uint32_t)p.w1);
            t2[base + i] = tstat_at(Sinc, Qinc, base, n, i, (uint32_t)p.w2);
        }
    }
}

// ---------------------------------------------------------------------------
// Clear the peak bits of one read (edge words are shared with neighbouring reads).
__device__ void clear_read_bits(uint32_t* __restrict__ bitmap, uint64_t p0, uint64_t p1) {
    if (p1 <= p0) return;
    const uint64_t w0 = p0 >> 5, w1 = (p1 - 1) >> 5;
    const uint32_t m0 = 0xffffffffu << (p0 & 31);
    const uint32_t m1 = 0xffffffffu >> (31 - ((p1 - 1) & 31));
    if (w0 == w1) { atomicAnd(&bitmap[w0], ~(m0 & m1)); return; }
    atomicAnd(&bitmap[w0], ~m0);
    for (uint64_t w = w0 + 1; w < w1; w++) bitmap[w] = 0u;
    atomicAnd(&bitmap[w1], ~m1);
}

// the detector of one read in the reference's own order (one thread): events.c:371-443
__device__ void detect_read_in_order(const DetParams& p, const float* __restrict__ t1, const float* __restrict__ t2,
                                     uint64_t base, uint64_t foff, uint32_t n, uint32_t* __restrict__ bitmap) {
    clear_read_bits(bitmap, foff, foff + n);  // drop whatever was found for this read so far
    atomicOr(&bitmap[foff >> 5], 1u << (foff & 31));  // event 0 starts at the first sample
    DetState s, l;
    det_reset(s);
    det_reset(l);
    // the detector is one dependent chain per read; its inputs are loaded 16 positions at a time, one group ahead
    // (the scratch holds whole groups: every read's share is padded to 8 samples and the arrays to 16)
    const float4* __restrict__ a1 = reinterpret_cast<const float4*>(t1 + base);
    const float4* __restrict__ a2 = reinterpret_cast<const float4*>(t2 + base);
    const uint32_t n4 = (n + 3u) >> 2;
    float4 c1[4], c2[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        c1[k] = (uint32_t)k < n4 ? __ldg(a1 + k) : make_float4(0.f, 0.f, 0.f, 0.f);
        c2[k] = (uint32_t)k < n4 ? __ldg(a2 + k) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (uint32_t g0 = 0; g0 < n4; g0 += 4) {
        float u1[16], u2[16];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            u1[4 * k] = c1[k].x; u1[4 * k + 1] = c1[k].y; u1[4 * k + 2] = c1[k].z; u1[4 * k + 3] = c1[k].w;
            u2[4 * k] = c2[k].x; u2[4 * k + 1] = c2[k].y; u2[4 * k + 2] = c2[k].z; u2[4 * k + 3] = c2[k].w;
            const uint32_t g = g0 + 4 + k;
            c1[k] = g < n4 ? __ldg(a1 + g) : make_float4(0.f, 0.f, 0.f, 0.f);
            c2[k] = g < n4 ? __ldg(a2 + g) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int m = 0; m < 16; m++) {
            const uint32_t i = g0 * 4u + m;
            if (i >= n) break;
            const int32_t ps = det_step(s, &l, true, i, u1[m], p.thr1, p.w1, p.height);
            if (ps > 0) { const uint64_t f = foff + (uint32_t)ps; atomicOr(&bitmap[f >> 5], 1u << (f & 31)); }
            const int32_t pl = det_step(l, nullptr, false, i, u2[m], p.thr2, p.w2, p.height);
            if (pl > 0) { const uint64_t f = foff + (uint32_t)pl; atomicOr(&bitmap[f >> 5], 1u << (f & 31)); }
        }
    }
}

// The detector over the stored t arrays, one WARP per read: the lanes walk 32 consecutive chunks of GD_CHUNK
// positions at once, each from a cold state W positions early (the walker's warm-up, walk.cu), with the branch-free
// detector step of walk_core.cuh; a chunk's state after its warm-up must equal its predecessor's end state
// (compared through a shuffle; the group's last state is carried to the next group). Peaks are owned by the step
// that emits them. Any mismatch in the read: lane 0 redoes the read in the reference's own order.
// PA (t arrays of a caller's pA signal, which may hold NaN): returns the number of mismatched chunks, and a NaN
// t-statistic anywhere in the read also sends it to the reference's order -- the branch-free step's fminf / fmaxf
// would take the other operand where the reference's comparisons keep a NaN running value (events.c:393-409).
template <int RNA, bool PA>
__device__ uint32_t detect_read_chunked(const float* __restrict__ t1, const float* __restrict__ t2, uint64_t base,
                                        uint64_t foff, uint32_t n, uint32_t W, uint32_t* __restrict__ bitmap, int lane,
                                        const DetParams& p) {
    using namespace walk;
    if (lane == 0) {
        clear_read_bits(bitmap, foff, foff + n);
        atomicOr(&bitmap[foff >> 5], 1u << (foff & 31));  // event 0 starts at the first sample
    }
    __syncwarp();
    const uint32_t n_chunks = (n + GD_CHUNK - 1) / GD_CHUNK;
    bool bad = false, nan = false;
    uint32_t n_bad = 0;
    Canon carry = {};  // end state of the previous group's last chunk
    auto on_emit = [&](int pos) { const uint64_t f = foff + (uint32_t)pos; atomicOr(&bitmap[f >> 5], 1u << (f & 31)); };
    for (uint32_t c0 = 0; c0 < n_chunks; c0 += 32) {
        const uint32_t c = c0 + lane;
        const bool have = c < n_chunks;
        const uint32_t s0 = c * GD_CHUNK, s1 = min(n, s0 + GD_CHUNK);
        DualDet d;
        Canon begin = {}, end = {};
        if (have) {
            uint32_t i = (c == 0) ? 1u : s0 - W;   // position 0 is never stepped (masked_to = 0, events.c:387)
            dual_cold(d, (int)i);
            for (; i < s0; i++) {   // warm-up: nothing is recorded
                const float c1 = __ldg(t1 + base + i), c2 = __ldg(t2 + base + i);
                if constexpr (PA) nan |= (c1 != c1) | (c2 != c2);
                dual_step<RNA>(d, (int)i, c1, c2, NoEmit());
            }
            begin = dual_canon(d, (int)s0);
            for (; i < s1; i++) {
                const float c1 = __ldg(t1 + base + i), c2 = __ldg(t2 + base + i);
                if constexpr (PA) nan |= (c1 != c1) | (c2 != c2);
                dual_step<RNA>(d, (int)i, c1, c2, on_emit);
            }
            end = dual_canon(d, (int)s1);
        }
        // chunk c must have reached the state chunk c-1 ended in
        bool same = true;
#pragma unroll
        for (int q = 0; q < 5; q++) {
            int prev = __shfl_up_sync(0xffffffffu, end.v[q], 1);
            if (lane == 0) prev = carry.v[q];
            same = same && (prev == begin.v[q]);
        }
        if (have && c > 0 && !same) { bad = true; n_bad++; }
        const int last = (int)min(31u, n_chunks - 1u - c0);
#pragma unroll
        for (int q = 0; q < 5; q++) carry.v[q] = __shfl_sync(0xffffffffu, end.v[q], last);
    }
    if (__any_sync(0xffffffffu, bad || nan)) {
        __syncwarp();
        if (lane == 0) detect_read_in_order(p, t1, t2, base, foff, n, bitmap);
    }
    if constexpr (PA) return __reduce_add_sync(0xffffffffu, n_bad);
    return 0u;
}

// PA: fixups[r] = the read's mismatched chunks
template <bool PA>
__device__ __forceinline__ void gen_detect_reads(const DevBatch& b, const WorkList& wl, const float* __restrict__ t1,
                                                 const float* __restrict__ t2, uint32_t* __restrict__ bitmap,
                                                 uint32_t W, uint32_t* __restrict__ fixups) {
    const uint32_t n_list = *wl.count;
    const DetParams p = det_params(b.rna);
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t j = warp; j < n_list; j += n_warps) {
        const uint32_t r = wl.list[j];
        const uint64_t base = wl.sbase[j];
        const uint64_t foff = b.read_off[r];
        const uint32_t n = b.read_len[r];
        if (n == 0) continue;
        if (n >= (1u << 30)) { if (lane == 0) detect_read_in_order(p, t1, t2, base, foff, n, bitmap); continue; }
        const uint32_t n_bad = b.rna ? detect_read_chunked<1, PA>(t1, t2, base, foff, n, W, bitmap, lane, p)
                                     : detect_read_chunked<0, PA>(t1, t2, base, foff, n, W, bitmap, lane, p);
        if constexpr (PA) { if (lane == 0) fixups[r] = n_bad; }
    }
}

__global__ void __launch_bounds__(128) gen_detect_kernel(DevBatch b, WorkList wl, const float* __restrict__ t1,
                                                         const float* __restrict__ t2, uint32_t* __restrict__ bitmap,
                                                         uint32_t W) {
    gen_detect_reads<false>(b, wl, t1, t2, bitmap, W, nullptr);
}

__global__ void __launch_bounds__(128) gen_detect_pa_kernel(DevBatch b, WorkList wl, const float* __restrict__ t1,
                                                            const float* __restrict__ t2, uint32_t* __restrict__ bitmap,
                                                            uint32_t W, uint32_t* __restrict__ fixups) {
    gen_detect_reads<true>(b, wl, t1, t2, bitmap, W, fixups);
}

// ---------------------------------------------------------------------------
// Exclusive scan cnt[u32] -> off[u64] (n+1 entries), single pass with
// decoupled look-back (tile status = 2 flag bits | 62-bit value).
static constexpr int SCAN_THREADS = 256;
static constexpr int SCAN_ITEMS = 8;
static constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;
static constexpr uint64_t ST_AGG = 1ull << 62, ST_INC = 2ull << 62, ST_MASK = (1ull << 62) - 1;

__global__ void __launch_bounds__(SCAN_THREADS) scan_counts_kernel(const uint32_t* __restrict__ cnt, uint32_t n,
                                                                   uint64_t* __restrict__ off,
                                                                   unsigned long long* __restrict__ status,
                                                                   uint32_t* __restrict__ ticket,
                                                                   uint64_t* __restrict__ total_out) {
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_warp[SCAN_THREADS / 32];
    __shared__ uint64_t s_prefix;
    if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint32_t base = tile * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    uint64_t v[SCAN_ITEMS];
    uint64_t sum = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        v[k] = (base + k < n) ? cnt[base + k] : 0u;
        sum += v[k];
    }
    // CTA-wide exclusive scan of the per-thread sums
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint64_t inc = sum;
    for (int o = 1; o < 32; o <<= 1) {
        const uint64_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (uint32_t)o) inc += t;
    }
    if (lane == 31) s_warp[wid] = inc;
    __syncthreads();
    uint64_t warp_excl = 0, cta_total = 0;
    for (int k = 0; k < SCAN_THREADS / 32; k++) {
        if (k < (int)wid) warp_excl += s_warp[k];
        cta_total += s_warp[k];
    }
    uint64_t excl = warp_excl + inc - sum;
    if (threadIdx.x == 0) {
        uint64_t prefix = 0;
        if (tile == 0) {
            __threadfence();
            atomicExch(&status[0], ST_INC | cta_total);
        } else {
            atomicExch(&status[tile], ST_AGG | cta_total);
            int64_t look = (int64_t)tile - 1;
            while (look >= 0) {
                unsigned long long st;
                do { st = atomicAdd(&status[look], 0ull); } while ((st >> 62) == 0);
                prefix += st & ST_MASK;
                if ((st >> 62) == 2) break;
                look--;
            }
            atomicExch(&status[tile], ST_INC | (prefix + cta_total));
        }
        s_prefix = prefix;
    }
    __syncthreads();
    excl += s_prefix;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        if (base + k < n) off[base + k] = excl;
        excl += v[k];
        if (base + k == n - 1) { off[n] = excl; if (total_out) *total_out = excl; }
    }
}

// ---------------------------------------------------------------------------
// create_events / create_event (events.c:457-504) from the sequential-order prefix sums.
__global__ void __launch_bounds__(128) gen_emit_kernel(DevBatch b, WorkList wl, const double* __restrict__ Sinc,
                                                       const double* __restrict__ Qinc,
                                                       const uint32_t* __restrict__ bitmap,
                                                       const uint64_t* __restrict__ ev_off, uint64_t ev_cap,
                                                       uint32_t* __restrict__ ev_start, float* __restrict__ ev_mean,
                                                       float* __restrict__ ev_stdv, int* __restrict__ status) {
    // one WARP per read: the lanes take consecutive bitmap words; a warp scan gives every event start its index
    // and the start before it (the statistics only need the two prefix-sum entries at an event's ends)
    const uint32_t n_list = *wl.count;
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t j = warp; j < n_list; j += n_warps) {
        const uint32_t r = wl.list[j];
        const uint64_t base = wl.sbase[j];
        const uint64_t p0 = b.read_off[r];
        const uint32_t n = b.read_len[r];
        if (ev_off[r + 1] > ev_cap) { if (lane == 0) atomicExch(status, SGPU_DEV_E_EVCAP); continue; }
        if (n == 0) continue;
        const uint64_t p1 = p0 + n;
        const uint64_t w_first = p0 >> 5, w_last = (p1 - 1) >> 5;
        uint64_t k = ev_off[r];  // index of the read's open event (starts at `a`)
        uint32_t a = 0;
        for (uint64_t w0 = w_first; w0 <= w_last; w0 += 32) {
            const uint64_t w = w0 + lane;
            uint32_t v = w <= w_last ? bitmap[w] : 0u;
            // peaks[i] > 0 && peaks[i] < nsample (events.c:482): drop the bits at or before p0 and at or after p1
            if (w == w_first) v &= (p0 & 31) == 31 ? 0u : (0xffffffffu << ((p0 & 31) + 1));
            if (w == w_last && ((p1 - 1) & 31) != 31) v &= 0xffffffffu >> (31 - ((p1 - 1) & 31));
            const uint32_t cnt = __popc(v);
            uint32_t inc = cnt;
            // the last event start at or before the end of this lane's word (0xffffffff: none yet in this group)
            uint32_t last = v ? (uint32_t)((w << 5) + (31 - __clz(v)) - p0) : 0xffffffffu;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
                const uint32_t tl = __shfl_up_sync(0xffffffffu, last, o);
                if (lane >= o) { inc += t; if (last == 0xffffffffu) last = tl; }
            }
            uint32_t prev = __shfl_up_sync(0xffffffffu, last, 1);  // the start before this lane's first bit
            if (lane == 0 || prev == 0xffffffffu) prev = a;
            uint64_t kk = k + (inc - cnt);
            while (v) {
                const int bit = __ffs(v) - 1;
                v &= v - 1;
                const uint32_t e = (uint32_t)((w << 5) + bit - p0);
                float m, sd;
                event_stats(__dsub_rn(prefix_at(Sinc, base, e), prefix_at(Sinc, base, prev)),
                            __dsub_rn(prefix_at(Qinc, base, e), prefix_at(Qinc, base, prev)), e - prev, &m, &sd);
                ev_start[kk] = prev; ev_mean[kk] = m; ev_stdv[kk] = sd;
                kk++;
                prev = e;
            }
            const uint32_t tot = __shfl_sync(0xffffffffu, inc, 31), tl = __shfl_sync(0xffffffffu, last, 31);
            k += tot;
            if (tl != 0xffffffffu) a = tl;
        }
        if (lane == 0) {  // last event ends at nsample (events.c:499-501)
            float m, sd;
            event_stats(__dsub_rn(prefix_at(Sinc, base, n), prefix_at(Sinc, base, a)),
                        __dsub_rn(prefix_at(Qinc, base, n), prefix_at(Qinc, base, a)), n - a, &m, &sd);
            ev_start[k] = a; ev_mean[k] = m; ev_stdv[k] = sd;
        }
    }
}

// ---------------------------------------------------------------------------
// signal_in_picoamps (misc.c:15-32) for a whole batch: one thread converts 16-byte groups of 8 samples (groups
// never straddle reads: read starts are 8-aligned). A warp takes PA_IT x 256 consecutive samples per step: ONE
// binary search for the read of its first group, a short forward walk per lane and group (reads are consecutive),
// all PA_IT 128-bit loads of a lane in flight before the first conversion. (One search per 256 samples made the
// kernel latency bound on batches of many reads: 51 % of the copy peak with 16,384 reads against 84 % with 320.)
constexpr int PA_IT = 8;
__global__ void __launch_bounds__(256) pa_kernel(DevBatch b, float* __restrict__ pa) {
    const uint64_t n_groups = b.span >> 3;
    const int lane = threadIdx.x & 31;
    const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t c0 = warp * (32 * PA_IT); c0 < n_groups; c0 += n_warps * (32 * PA_IT)) {
        uint32_t r = 0;
        if (lane == 0) r = find_read(b.read_off, b.n_reads, c0 << 3);
        r = __shfl_sync(0xffffffffu, r, 0);
        int4 raw[PA_IT];
        float off[PA_IT], unit[PA_IT];
        bool live[PA_IT];
#pragma unroll
        for (int it = 0; it < PA_IT; it++) {
            const uint64_t g = c0 + (uint64_t)it * 32 + lane;
            const uint64_t p = g << 3;
            live[it] = g < n_groups;
            if (live[it]) {
                while (r + 1 < b.n_reads && b.read_off[r + 1] <= p) r++;
                live[it] = p - b.read_off[r] < b.read_len[r];  // false in an alignment gap
            }
            if (live[it]) {
                off[it] = b.offset[r];
                unit[it] = b.unit[r];
                raw[it] = __ldg(reinterpret_cast<const int4*>(b.samples + p));
            }
        }
#pragma unroll
        for (int it = 0; it < PA_IT; it++) {
            if (!live[it]) continue;
            const uint64_t p = (c0 + (uint64_t)it * 32 + lane) << 3;
            const int v[4] = {raw[it].x, raw[it].y, raw[it].z, raw[it].w};
            float o[8];
            walk::cvt8(v, off[it], unit[it], o);   // misc.c:28 per sample: float add of the offset, float multiply by the unit
            float4* dst = reinterpret_cast<float4*>(pa + p);
            __stcs(dst, make_float4(o[0], o[1], o[2], o[3]));      // streaming stores: the output is not read again here
            __stcs(dst + 1, make_float4(o[4], o[5], o[6], o[7]));
        }
    }
}

// ---------------------------------------------------------------------------
// host-side launchers
int launch_generic_detect(const DevBatch& b, const WorkList& wl, Scratch& sc, int sm_count, cudaStream_t st) {
    gen_prefix_kernel<<<sm_count * 8, 128, 0, st>>>(b, wl, sc.Sinc, sc.Qinc);
    gen_tstat_kernel<<<sm_count * 8, 256, 0, st>>>(b, wl, sc.Sinc, sc.Qinc, sc.t1, sc.t2, det_params(b.rna));
    gen_detect_kernel<<<sm_count * 8, 128, 0, st>>>(b, wl, sc.t1, sc.t2, sc.bitmap, b.rna ? 384u : 64u);  // (its own warm-up, longer than the walker's)
    return 3;
}

// a batch on the general route (pa_input.cu): the prefix sums of the reads in `ordered` (those that failed the
// exact-sum witness) in the reference's order -- the others' were stored by pa_scan_kernel --, then t-statistics and
// detector for all reads (pa: the caller's floats, or nullptr: b's int16 samples; set: the caller's detector set, or
// nullptr: the reference's chosen by b.rna)
int launch_generic_detect_pa(const DevBatch& b, const float* pa, const DetParams* set, const WorkList& ordered,
                             const WorkList& all, Scratch& sc, uint32_t* fixups, int sm_count, cudaStream_t st) {
    if (pa) gen_prefix_pa_kernel<<<sm_count * 8, 128, 0, st>>>(b, pa, ordered, sc.Sinc, sc.Qinc);
    else    gen_prefix_kernel<<<sm_count * 8, 128, 0, st>>>(b, ordered, sc.Sinc, sc.Qinc);
    gen_tstat_kernel<<<sm_count * 8, 256, 0, st>>>(b, all, sc.Sinc, sc.Qinc, sc.t1, sc.t2, set ? *set : det_params(b.rna));
    if (set) launch_detect_set(b, all, sc, fixups, *set, sm_count, st);
    else     gen_detect_pa_kernel<<<sm_count * 8, 128, 0, st>>>(b, all, sc.t1, sc.t2, sc.bitmap, b.rna ? 384u : 64u, fixups);
    return 3;
}

int launch_scan_u32(const uint32_t* cnt, uint32_t n, uint64_t* off, uint64_t* total_out, Scratch& sc, cudaStream_t st) {
    const uint32_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    cudaMemsetAsync(sc.scan_status, 0, (size_t)(tiles + 1) * sizeof(unsigned long long), st);
    cudaMemsetAsync(sc.scan_ticket, 0, sizeof(uint32_t), st);
    scan_counts_kernel<<<tiles ? tiles : 1, SCAN_THREADS, 0, st>>>(cnt, n, off, sc.scan_status, sc.scan_ticket,
                                                                  total_out);
    return 1;
}

int launch_generic_emit(const DevBatch& b, const WorkList& wl, Scratch& sc, const uint64_t* ev_off, uint64_t ev_cap,
                        uint32_t* ev_start, float* ev_mean, float* ev_stdv, int sm_count, cudaStream_t st) {
    gen_emit_kernel<<<sm_count * 8, 128, 0, st>>>(b, wl, sc.Sinc, sc.Qinc, sc.bitmap, ev_off, ev_cap, ev_start,
                                                  ev_mean, ev_stdv, sc.status);
    return 1;
}

int launch_pa(const DevBatch& b, float* pa, int sm_count, cudaStream_t st) {
    pa_kernel<<<grid_cap(((b.span >> 3) + PA_IT - 1) / PA_IT, 256, sm_count * 16), 256, 0, st>>>(b, pa);
    return 1;
}

uint32_t scan_tiles_for(uint32_t n) { return (n + SCAN_TILE - 1) / SCAN_TILE + 1; }

}  // namespace sgpu
