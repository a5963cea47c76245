// live.cu -- getevents (events.c:553-573) on signal that arrives in chunks, channel by channel.
//
// A push is a batch of entries, at most one per channel. Each entry continues its channel's read from the state the
// channel carries in HBM (LiveChan): the prefix sums are one sequential double chain continued from the carried S, Q
// (so they have the reference's bits), the t-statistic of a position needs S, Q over [i-w2, i+w2] only (the carried
// tail), and the two peak detectors are stepped in the reference's order (short, then long; events.c:385-437) over
// every position whose right window [i, i+w2) is complete -- at END over the rest, whose long t-statistic is 0
// (events.c:328-338). A peak can be emitted long after its position, so the channel keeps the prefix sums at each
// detector's peak and at the open event's start. Every emitted peak p closes the event [a, p) (events.c:475-504).
//
//   live_kernel<PA>      one warp per entry, tiles of LIVE_TILE samples: pA by all lanes (misc.c:28 on int16 samples,
//                        or the caller's floats as they are), the S/Q chain by lane 0
//                        (the lane-0 chain of gen_prefix_reads), the t-statistics of the positions that became final
//                        one lane per position (tstat_reference_chain), the detector by lane 0 (det_step), events
//                        staged at live_stage_base of the entry
//   scan_counts_kernel   events per entry -> ev_off (launch_scan_u32)
//   live_compact_kernel  staged events -> the compact event table
//
// The S/Q chain is formed one sample after another in the reference's order whatever the input, so pA entries need no
// exactness witness (pa_input.cu): the floats go through the same chain as the pA of int16 samples. A read keeps the
// form of the entry that started it (LiveScratch::form); an entry of the other form that continues it is refused.
// Likewise it keeps the detector set in force for its START entry (sgpu_set_detector; LiveChan::custom, set), and a
// position is stepped once both of its right windows are complete: i <= n - max(w1, w2).
#include "../../include/sigtk_b200.h"
#include "kernels.cuh"

namespace sgpu {

constexpr int LIVE_WARPS = 4;    // warps per block
constexpr int LIVE_TILE = 256;   // samples per tile: bounded shared memory for any length of entry

struct LiveWarpSmem {
    double S[LIVE_TAIL + LIVE_TILE], Q[LIVE_TAIL + LIVE_TILE];  // S[jb + k] at k (jb = n - LIVE_TAIL + 1)
    float pa[LIVE_TILE];
    float t1[LIVE_TILE + 16], t2[LIVE_TILE + 16];                // positions [st, L): at most a tile + 13
};

// t-statistic of position i (buffer index ki) with window w once n samples of the read are known: zero unless
// w <= i <= n - w (events.c:328-338; the positions asked for never change their value when n grows)
__device__ __forceinline__ float live_tstat(const double* S, const double* Q, int64_t ki, uint64_t i, uint32_t w,
                                            uint64_t n) {
    if (i < w || i + w > n) return 0.0f;
    const double s_i = S[ki], q_i = Q[ki];
    return tstat_reference_chain(__dsub_rn(s_i, S[ki - w]), __dsub_rn(q_i, Q[ki - w]), __dsub_rn(S[ki + w], s_i),
                                 __dsub_rn(Q[ki + w], q_i), (float)w);
}

// PA: the entries are the caller's pA floats (b.pa), else int16 samples with the calibration given at START
template <bool PA>
__global__ void __launch_bounds__(LIVE_WARPS * 32)
live_kernel(LiveBatch b, LiveChan* __restrict__ chan, uint32_t* __restrict__ nopen, uint32_t* __restrict__ claim,
            uint32_t n_channels, uint32_t stamp, float thr_long, DetParams set, bool use_set, bool dense,
            uint32_t* __restrict__ cnt, uint32_t* __restrict__ s_start, uint32_t* __restrict__ s_len,
            float* __restrict__ s_mean, float* __restrict__ s_stdv, uint64_t ev_cap, int* __restrict__ status,
            uint8_t* __restrict__ form) {
    constexpr uint8_t my_form = PA ? LIVE_FORM_PA : LIVE_FORM_INT16;
    __shared__ LiveWarpSmem smem[LIVE_WARPS];
    LiveWarpSmem& sm = smem[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t e = warp; e < b.n_entries; e += n_warps) {
        const uint32_t c = b.channel[e], f = b.flags[e], len = b.read_len[e];
        const uint64_t off = b.read_off[e];
        const bool start = (f & SGPU_LIVE_START) != 0, end = (f & SGPU_LIVE_END) != 0;
        // the checks sgpu_submit makes against its mirror, for entries that come from device memory; an entry that
        // fails them leaves its channel as it was and reports no event
        int code = SGPU_DEV_OK;
        uint32_t no = 0;
        if (lane == 0) {
            if ((f & ~LIVE_FLAGS) || c >= n_channels || off + len > b.read_off[e + 1] || b.read_off[e + 1] > b.span)
                code = SGPU_DEV_E_INVAL;
            else if (atomicExch(&claim[c], stamp) == stamp)  // a second entry for the channel in this run
                code = SGPU_DEV_E_INVAL;
            else {
                no = nopen[c];
                if (!start && !(no & LIVE_OPEN) && (len || end)) code = SGPU_DEV_E_STATE;
                else if (!start && (no & LIVE_OPEN) && form[c] != my_form) code = SGPU_DEV_E_STATE;  // the other form
                else if ((start ? 0ull : (uint64_t)(no & ~LIVE_OPEN)) + len > 0x7fffffffull) code = SGPU_DEV_E_TOOBIG;
            }
            if (code) atomicExch(status, code);
        }
        code = __shfl_sync(0xffffffffu, code, 0);
        no = __shfl_sync(0xffffffffu, no, 0);
        if (code || (!start && !(no & LIVE_OPEN))) {  // refused, or an empty entry on a channel without a read
            if (lane == 0) cnt[e] = 0;
            continue;
        }
        LiveChan& ch = chan[c];
        const uint32_t rna = start ? ((f & SGPU_LIVE_RNA) ? 1u : 0u) : ch.rna;
        const float offv = PA ? 0.0f : (start ? b.offset[e] : ch.offset), unitv = PA ? 1.0f : (start ? b.unit[e] : ch.unit);
        // the read's detector: the caller's set in force at its START, else the reference's for rna with the long
        // threshold of the push (SGPU_PARAM_THR_LONG)
        const bool custom = start ? use_set : ch.custom != 0u;
        const DetParams p = custom ? (start ? set : ch.set) : det_params((int)rna);
        const float thr2 = custom ? p.thr2 : thr_long;
        const uint32_t w1 = (uint32_t)p.w1, w2 = (uint32_t)p.w2, wm = max(w1, w2);
        uint64_t n_cur = start ? 0 : (no & ~LIVE_OPEN);
        if (lane < LIVE_TAIL) {  // a new read: S[j] = Q[j] = 0 for every j <= 0
            sm.S[lane] = start ? 0.0 : ch.tS[lane];
            sm.Q[lane] = start ? 0.0 : ch.tQ[lane];
        }
        // the detector, its peaks' and the open event's prefix sums (lane 0)
        DetState ds, dl;
        double pS0 = 0.0, pQ0 = 0.0, pS1 = 0.0, pQ1 = 0.0, aS = 0.0, aQ = 0.0;
        uint32_t a = 0, n_ev = 0;
        if (lane == 0) {
            if (start) {
                det_reset(ds);
                det_reset(dl);
            } else {
                ds = ch.det[0]; dl = ch.det[1];
                pS0 = ch.pS[0]; pQ0 = ch.pQ[0]; pS1 = ch.pS[1]; pQ1 = ch.pQ[1];
                aS = ch.aS; aQ = ch.aQ; a = ch.a;
            }
        }
        const uint64_t sbase = live_stage_base(off, e, dense);
        auto emit = [&](uint32_t pk, double pks, double pkq) {  // peak pk closes the event [a, pk)
            const uint64_t k = sbase + n_ev;
            if (k >= ev_cap) { atomicExch(status, SGPU_DEV_E_EVCAP); return; }  // (cannot happen: live_stage_base)
            float mn, sd;
            event_stats(__dsub_rn(pks, aS), __dsub_rn(pkq, aQ), pk - a, &mn, &sd);
            s_start[k] = a; s_len[k] = pk - a; s_mean[k] = mn; s_stdv[k] = sd;
            n_ev++;
            a = pk; aS = pks; aQ = pkq;
        };
        uint64_t st = n_cur + 1 > wm ? n_cur + 1 - wm : 0;  // positions [0, st) have been stepped
        uint32_t t0 = 0;
        do {
            const uint32_t m = min((uint32_t)LIVE_TILE, len - t0);
            if constexpr (PA)
                for (uint32_t k = lane; k < m; k += 32) sm.pa[k] = b.pa[off + t0 + k];
            else
                for (uint32_t k = lane; k < m; k += 32) sm.pa[k] = pa_of(b.samples[off + t0 + k], offv, unitv);
            __syncwarp();
            if (lane == 0) {  // events.c:293-303: the order of the additions is the result
                double s = sm.S[LIVE_TAIL - 1], q = sm.Q[LIVE_TAIL - 1];
                for (uint32_t k = 0; k < m; k++) {
                    const float x = sm.pa[k];
                    s = __dadd_rn(s, (double)x);
                    q = __dadd_rn(q, (double)__fmul_rn(x, x));  // float product, widened afterwards (events.c:301)
                    sm.S[LIVE_TAIL + k] = s;
                    sm.Q[LIVE_TAIL + k] = q;
                }
            }
            __syncwarp();
            const uint64_t n_new = n_cur + m;
            uint64_t L = (end && t0 + m == len) ? n_new : (n_new + 1 > wm ? n_new + 1 - wm : 0);
            if (L < st) L = st;
            const int64_t jb = (int64_t)n_cur - (LIVE_TAIL - 1);
            for (uint64_t i = st + lane; i < L; i += 32) {
                const int64_t ki = (int64_t)i - jb;
                sm.t1[i - st] = live_tstat(sm.S, sm.Q, ki, i, w1, n_new);
                sm.t2[i - st] = live_tstat(sm.S, sm.Q, ki, i, w2, n_new);
            }
            __syncwarp();
            if (lane == 0) {
                for (uint64_t i = st; i < L; i++) {  // events.c:385-437, short then long
                    const uint32_t k = (uint32_t)(i - st), pos = (uint32_t)i;
                    const int64_t ki = (int64_t)i - jb;
                    const double si = sm.S[ki], qi = sm.Q[ki];
                    const double os = pS0, oq = pQ0;
                    const int32_t ps = det_step(ds, &dl, true, pos, sm.t1[k], p.thr1, p.w1, p.height);
                    if (ds.peak_pos == (int32_t)pos) { pS0 = si; pQ0 = qi; }
                    if (ps > 0) emit((uint32_t)ps, os, oq);  // peaks[i] > 0 (events.c:481-485)
                    const double ol = pS1, oql = pQ1;
                    const int32_t pl = det_step(dl, nullptr, false, pos, sm.t2[k], thr2, p.w2, p.height);
                    if (dl.peak_pos == (int32_t)pos) { pS1 = si; pQ1 = qi; }
                    if (pl > 0) emit((uint32_t)pl, ol, oql);
                }
            }
            st = L;
            double vS = 0.0, vQ = 0.0;  // the tail of S[.. n_new] moves to the front
            if (lane < LIVE_TAIL) { vS = sm.S[m + lane]; vQ = sm.Q[m + lane]; }
            __syncwarp();
            if (lane < LIVE_TAIL) { sm.S[lane] = vS; sm.Q[lane] = vQ; }
            __syncwarp();
            n_cur = n_new;
            t0 += m;
        } while (t0 < len);
        if (end) {
            if (lane == 0) {
                if (n_cur) emit((uint32_t)n_cur, sm.S[LIVE_TAIL - 1], sm.Q[LIVE_TAIL - 1]);  // [a, n) (events.c:499-501)
                nopen[c] = 0;
            }
        } else {
            if (lane < LIVE_TAIL) { ch.tS[lane] = sm.S[lane]; ch.tQ[lane] = sm.Q[lane]; }
            if (lane == 0) {
                ch.det[0] = ds; ch.det[1] = dl;
                ch.pS[0] = pS0; ch.pQ[0] = pQ0; ch.pS[1] = pS1; ch.pQ[1] = pQ1;
                ch.aS = aS; ch.aQ = aQ; ch.a = a;
                ch.offset = offv; ch.unit = unitv; ch.rna = rna;
                ch.custom = custom ? 1u : 0u; ch.set = p;
                nopen[c] = (uint32_t)n_cur | LIVE_OPEN;
                if (start) form[c] = my_form;
            }
        }
        if (lane == 0) cnt[e] = n_ev;
        __syncwarp();
    }
}

// the staged events of every entry to [ev_off[e], ev_off[e+1]), one warp per entry
__global__ void __launch_bounds__(256) live_compact_kernel(LiveBatch b, const uint32_t* __restrict__ cnt,
                                                           const uint64_t* __restrict__ ev_off,
                                                           const uint32_t* __restrict__ s_start,
                                                           const uint32_t* __restrict__ s_len,
                                                           const float* __restrict__ s_mean,
                                                           const float* __restrict__ s_stdv, bool dense,
                                                           uint32_t* __restrict__ start, uint32_t* __restrict__ len,
                                                           float* __restrict__ mean, float* __restrict__ stdv) {
    const int lane = threadIdx.x & 31;
    const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t e = warp; e < b.n_entries; e += n_warps) {
        const uint64_t src = live_stage_base(b.read_off[e], e, dense), dst = ev_off[e];
        for (uint32_t k = lane; k < cnt[e]; k += 32) {
            start[dst + k] = s_start[src + k];
            len[dst + k] = s_len[src + k];
            mean[dst + k] = s_mean[src + k];
            stdv[dst + k] = s_stdv[src + k];
        }
    }
}

int launch_live(const LiveBatch& b, bool pa, const DetParams* set, LiveScratch& w, Scratch& sc, uint64_t* ev_off,
                uint32_t* ev_start, uint32_t* ev_len, float* ev_mean, float* ev_stdv, int sm_count, cudaStream_t st) {
    if (++w.stamp == 0) w.stamp = 1;  // (claim[] starts at 0)
    auto* const kernel = pa ? live_kernel<true> : live_kernel<false>;
    kernel<<<grid_cap(b.n_entries, LIVE_WARPS, sm_count * 8), LIVE_WARPS * 32, 0, st>>>(
        b, w.chan, w.nopen, w.claim, w.n_channels, w.stamp, sc.tune_thr_long, set ? *set : DetParams{}, set != nullptr,
        w.dense, w.cnt, w.s_start, w.s_len, w.s_mean, w.s_stdv, w.ev_cap, sc.status, w.form);
    int n = 1 + launch_scan_u32(w.cnt, b.n_entries, ev_off, reinterpret_cast<uint64_t*>(sc.counters.get()), sc, st);
    live_compact_kernel<<<grid_cap(b.n_entries, 8, sm_count * 8), 256, 0, st>>>(
        b, w.cnt, ev_off, w.s_start, w.s_len, w.s_mean, w.s_stdv, w.dense, ev_start, ev_len, ev_mean, ev_stdv);
    return n + 1;
}

}  // namespace sgpu
