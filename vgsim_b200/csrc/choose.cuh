// Cumulative search over a weight vector: the device counterpart of the reference's fastChoose / fastChoose_skip
// (src/fast_choose.pxi:18-52).  The reference walks the vector sequentially until the running total reaches the target;
// here a warp walks it 32 entries at a time with an inclusive shuffle scan and a ballot.  Contract (tested entry by
// entry against a restatement of the reference through vgsim_test_choose):
//   * the pick is the FIRST index whose inclusive prefix sum is >= x and whose weight is positive;
//   * if rounding leaves x above the total, the LAST positive weight is the catch-all (the reference's loop bound);
//   * an entry with zero weight is never picked (the reference would print "0-weight sampled" and exit, :29-30);
//     all weights zero -> index -1, which the callers turn into the sticky ERR_ZERO_WEIGHT bit;
//   * `skip` leaves one index out of the walk (fastChoose_skip);
//   * the caller gets the weight and the cumulative weight BEFORE the pick, from which both forms of the next level's
//     target follow: the reference's residual (x - before) / w in [0, 1), or (x - before) itself when the next level's
//     total IS the picked weight (no division on the dependent chain of an event).
#pragma once
#include "common.cuh"

namespace vg {

struct Pick {
    int i;          // index, -1: every weight was zero
    double before;  // cumulative weight before the pick
    double w;       // its weight
    __device__ __forceinline__ double resid(double x) const {  // fastChoose's second return value
        const double r = (x - before) / w;
        return r < 0.0 ? 0.0 : (r >= 1.0 ? 0.9999999999999999 : r);
    }
    __device__ __forceinline__ double rest(double x) const {  // (x - before) clamped into [0, w)
        const double r = x - before;
        return r < 0.0 ? 0.0 : (r >= w ? w * 0.9999999999999999 : r);
    }
};

// sum over the lanes of a warp, every lane gets it; a butterfly, so the result is the same function of the 32 lane
// values in every lane and every call
__device__ __forceinline__ double warp_sum(double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// inclusive prefix sum over the lanes of a warp; lanes >= n must hold 0 (steps beyond n are skipped)
__device__ __forceinline__ double warp_scan_incl(double v, int n) {
    const int lane = threadIdx.x & 31;
#pragma unroll 1
    for (int o = 1; o < n && o < 32; o <<= 1) {
        const double t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
    }
    return v;
}

template <class WF>
__device__ __forceinline__ Pick warp_pick(WF wf, int n, double x, int skip = -1) {
    const int lane = threadIdx.x & 31;
    Pick out;
    out.i = -1;
    out.before = 0.0;
    out.w = 0.0;
    double base = 0.0;
#pragma unroll 1
    for (int off = 0; off < n; off += 32) {
        const int i = off + lane;
        const double w = (i < n && i != skip) ? wf(i) : 0.0;
        const double c = warp_scan_incl(w, n - off) + base;
        const unsigned hit = __ballot_sync(0xffffffffu, w > 0.0 && c >= x);
        if (hit) {
            const int l = __ffs(hit) - 1;
            out.w = __shfl_sync(0xffffffffu, w, l);
            out.before = __shfl_sync(0xffffffffu, c, l) - out.w;
            out.i = off + l;
            return out;
        }
        const unsigned pos = __ballot_sync(0xffffffffu, w > 0.0);
        if (pos) {  // remember the last positive weight: the catch-all
            const int l = 31 - __clz(pos);
            out.i = off + l;
            out.w = __shfl_sync(0xffffffffu, w, l);
            out.before = __shfl_sync(0xffffffffu, c, l) - out.w;
        }
        base = __shfl_sync(0xffffffffu, c, 31);
    }
    return out;
}

// the same search over a handful of weights, executed identically by every lane (no shuffles)
template <class WF>
__device__ __forceinline__ Pick small_pick(WF wf, int n, double x) {
    Pick out, last;
    out.i = last.i = -1;
    out.before = out.w = last.before = last.w = 0.0;
    double acc = 0.0;
#pragma unroll
    for (int i = 0; i < n; i++) {
        const double w = wf(i);
        if (w > 0.0) {
            last.i = i;
            last.w = w;
            last.before = acc;
        }
        acc += w;
        if (out.i < 0 && w > 0.0 && acc >= x) {
            out.i = i;
            out.w = w;
            out.before = acc - w;
        }
    }
    return out.i >= 0 ? out : last;
}

}  // namespace vg
