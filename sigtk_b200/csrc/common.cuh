// common.cuh -- shared device helpers for the sigtk B200 hot path (sm_100a).
//
// Every arithmetic step that the reference performs is written with an explicit
// round-to-nearest intrinsic so that nvcc can neither contract (no FMA: the
// reference is built -std=c99 => -ffp-contract=off, Makefile:5) nor reassociate.
// The translation unit is additionally compiled with --fmad=false.
#pragma once
#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

namespace sgpu {

// detector parameters, reference src/events.c:35-54
struct DetParams {
    int w1, w2;        // short / long window length
    float thr1, thr2;  // thresholds
    float height;      // peak_height
};

__host__ __device__ inline DetParams det_params(int rna) {
    DetParams p;
    if (rna) { p.w1 = 7; p.w2 = 14; p.thr1 = 2.5f; p.thr2 = 9.0f; p.height = 1.0f; }
    else     { p.w1 = 3; p.w2 = 6;  p.thr1 = 1.4f; p.thr2 = 9.0f; p.height = 0.2f; }
    return p;
}

// One batch of reads resident in HBM (see include/sigtk_b200.h for the layout).
struct DevBatch {
    const int16_t*  samples;
    const uint64_t* read_off;  // [n_reads+1]
    const uint32_t* read_len;  // [n_reads]
    const float*    offset;    // [n_reads] (float)rec->offset
    const float*    unit;      // [n_reads] (float)range/(float)digitisation
    uint32_t n_reads;
    int      rna;
    uint64_t span;             // read_off[n_reads]
};

// pA of one sample, reference src/misc.c:28: float add, then float multiply.
__device__ __forceinline__ float pa_of(int16_t raw, float off, float unit) {
    return __fmul_rn(__fadd_rn((float)raw, off), unit);
}

// The windowed t-statistic exactly as the reference evaluates it
// (src/events.c:338-361) given the four window sums in double:
//   sum1/ssq1 : left window  [i-w, i)   (kept in double)
//   sum2/ssq2 : right window [i, i+w)   (narrowed to float at once)
__device__ __forceinline__ float tstat_reference_chain(double sum1, double ssq1, double sum2d,
                                                       double ssq2d, float wf) {
    const double wd = (double)wf;
    const float sum2 = __double2float_rn(sum2d);
    const float ssq2 = __double2float_rn(ssq2d);
    const float mean1 = __double2float_rn(__ddiv_rn(sum1, wd));
    const float mean2 = __fdiv_rn(sum2, wf);
    const float m1sq = __fmul_rn(mean1, mean1);
    const float m2sq = __fmul_rn(mean2, mean2);
    const float v2 = __fdiv_rn(ssq2, wf);
    double acc = __ddiv_rn(ssq1, wd);
    acc = __dsub_rn(acc, (double)m1sq);
    acc = __dadd_rn(acc, (double)v2);
    acc = __dsub_rn(acc, (double)m2sq);
    const float cv = fmaxf(__double2float_rn(acc), FLT_MIN);
    const float delta = __fsub_rn(mean2, mean1);
    const float scaled = __fdiv_rn(cv, wf);
    return __double2float_rn(__ddiv_rn(fabs((double)delta), __dsqrt_rn((double)scaled)));
}

// (the exact shortcuts of the fast path -- FMA-corrected division by the window length, guarded rsqrt tail --
// live in walk_core.cuh; the sequential-order kernels use the reference chain above)

// Event statistics from the two prefix-sum differences (src/events.c:457-473).
__device__ __forceinline__ void event_stats(double dsum, double dssq, uint32_t len, float* mean,
                                            float* stdv) {
    const float lenf = (float)len;
    const float m = __fdiv_rn(__double2float_rn(dsum), lenf);
    const float ex2 = __fdiv_rn(__double2float_rn(dssq), lenf);
    const float var = __fsub_rn(ex2, __fmul_rn(m, m));
    *mean = m;
    *stdv = __fsqrt_rn(fmaxf(var, 0.0f));
}

// State of one peak detector between samples (src/events.c:269-281).
struct DetState {
    uint32_t masked_to;
    int32_t  peak_pos;   // -1 = none
    float    peak_value;
    int32_t  valid;
};

__device__ __forceinline__ void det_reset(DetState& d) {
    d.masked_to = 0; d.peak_pos = -1; d.peak_value = FLT_MAX; d.valid = 0;
}

// One step of one detector (events.c:387-437). Returns the emitted peak position or -1.
// `is_short` selects the masking of the long detector (414-422).
__device__ __forceinline__ int32_t det_step(DetState& d, DetState* other_long, bool is_short, uint32_t i,
                                            float cur, float thr, int w, float height) {
    if (d.masked_to >= i) return -1;
    if (d.peak_pos < 0) {  // CASE 1
        if (cur < d.peak_value) {
            d.peak_value = cur;
        } else if (__fsub_rn(cur, d.peak_value) > height) {
            d.peak_value = cur;
            d.peak_pos = (int32_t)i;
        }
        return -1;
    }
    // CASE 2
    if (cur > d.peak_value) { d.peak_value = cur; d.peak_pos = (int32_t)i; }
    if (is_short && d.peak_value > thr) {
        other_long->masked_to = (uint32_t)d.peak_pos + (uint32_t)w;
        other_long->peak_pos = -1;
        other_long->peak_value = FLT_MAX;
        other_long->valid = 0;
    }
    if (__fsub_rn(d.peak_value, cur) > height && d.peak_value > thr) d.valid = 1;
    if (d.valid && (i - (uint32_t)d.peak_pos) > (uint32_t)(w / 2)) {
        const int32_t out = d.peak_pos;
        d.peak_pos = -1;
        d.peak_value = cur;
        d.valid = 0;
        return out;
    }
    return -1;
}

// grid of a launch: enough blocks of `block` threads for `work` items, at least 1 and at most max_blocks
static inline int grid_cap(uint64_t work, int block, int max_blocks) {
    uint64_t g = (work + block - 1) / block;
    if (g < 1) g = 1;
    if (g > (uint64_t)max_blocks) g = max_blocks;
    return (int)g;
}

// index of the read containing flat position p: largest r with read_off[r] <= p
__device__ __forceinline__ uint32_t find_read(const uint64_t* __restrict__ off, uint32_t n, uint64_t p) {
    uint32_t lo = 0, hi = n;  // invariant: off[lo] <= p < off[hi] (off[n] = span)
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (off[mid] <= p) lo = mid; else hi = mid;
    }
    return lo;
}

}  // namespace sgpu
