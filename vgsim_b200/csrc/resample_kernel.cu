// vgsim_resample: replicate r's whole run (state, counters, logs, archive, lockdown records) becomes the run of
// replicate source[r].  An HBM-bound gather of variable-length per-replicate segments: one CTA per (destination, array,
// 64 KB chunk) work item, 16-byte streaming loads and stores.
#include <algorithm>
#include "handle.h"

namespace vg {


enum { RS_THREADS = 256, RS_UNROLL = 8 };
static const long long RS_CHUNK = 2LL * RS_THREADS * RS_UNROLL * 16;  // bytes per work item: two rounds of 8 loads per thread

// How the used length of a source replicate's segment is found: rows(kind) * row bytes, or the whole row for SEG_FIXED.
enum { SEG_FIXED, SEG_EVENTS, SEG_LEAPS, SEG_DENSE, SEG_SPOFF, SEG_SPENT, SEG_LOC };
enum { RS_MAXSEG = 32 };

struct ResampleSeg {
    char *base;
    long long stride;  // bytes per replicate
    long long row;     // bytes per counted row
    int kind;
    int first_item, nitems;  // a SEG_FIXED segment with nitems == 0 is copied whole by work item 0 of its destination
};

struct ResampleArgs {
    const int2 *pairs;  // [ndst] (destination, source)
    int items;          // work items per destination
    int nseg;
    ResampleSeg seg[RS_MAXSEG];
};

static __device__ __forceinline__ long long clampll(long long v, long long hi) { return v < 0 ? 0 : v > hi ? hi : v; }

static __device__ long long used_bytes(const DevState &st, const ResampleSeg &g, int s) {
    const long long *c = st.counters + (size_t)s * NCOUNT;
    switch (g.kind) {
        case SEG_EVENTS: return clampll(c[C_EVPTR], st.ev_cap) * g.row;
        case SEG_LEAPS: return clampll(c[C_LEAPS], st.leap_cap) * g.row;
        case SEG_DENSE: return clampll(c[C_LEAPS] - st.dense_base[s], st.dense_cap) * g.row;
        case SEG_SPOFF: return (clampll(st.dense_base[s], st.leap_cap) + 1) * g.row;  // offsets of leaps 0..dense_base
        case SEG_SPENT: return clampll(st.sp_n[s], st.sp_cap) * g.row;
        case SEG_LOC: return clampll(st.loc_n[s], st.loc_cap) * g.row;
        default: return g.stride;
    }
}

// bytes [lo, hi) of one segment; lo is a multiple of 16, every length a multiple of 4 (4- and 8-byte elements)
static __device__ __forceinline__ void copy_range(char *dst, const char *src, long long lo, long long hi) {
    if (hi <= lo) return;
    dst += lo;
    src += lo;
    const long long n = hi - lo;
    long long done = 0;
    if ((((uintptr_t)dst | (uintptr_t)src) & 15) == 0) {
        const long long n16 = n >> 4;
        const uint4 *s4 = (const uint4 *)src;
        uint4 *d4 = (uint4 *)dst;
        for (long long i0 = threadIdx.x; i0 < n16; i0 += RS_THREADS * RS_UNROLL) {
            uint4 v[RS_UNROLL];
#pragma unroll
            for (int u = 0; u < RS_UNROLL; u++)
                if (i0 + u * RS_THREADS < n16) v[u] = __ldcs(s4 + i0 + u * RS_THREADS);
#pragma unroll
            for (int u = 0; u < RS_UNROLL; u++)
                if (i0 + u * RS_THREADS < n16) __stcs(d4 + i0 + u * RS_THREADS, v[u]);
        }
        done = n16 << 4;
    }
    // the tail, or a segment whose source and destination rows are not both 16-byte aligned (rows of a few int32)
    const int *s1 = (const int *)(src + done);
    int *d1 = (int *)(dst + done);
    for (long long i = threadIdx.x; i < (n - done) >> 2; i += RS_THREADS) __stcs(d1 + i, __ldcs(s1 + i));
}

__global__ void __launch_bounds__(RS_THREADS) resample_kernel(const DevState st, const ResampleArgs a) {
    const long long b = blockIdx.x;
    const int d = (int)(b / a.items), item = (int)(b - (long long)d * a.items);
    const int2 p = a.pairs[d];
    const int r = p.x, s = p.y;
    if (item == 0) {
        for (int k = 0; k < a.nseg; k++) {
            const ResampleSeg &g = a.seg[k];
            if (g.kind == SEG_FIXED && g.nitems == 0) copy_range(g.base + r * g.stride, g.base + s * g.stride, 0, g.stride);
        }
        return;
    }
    int k = 0;
    while (k < a.nseg && !(a.seg[k].nitems && item >= a.seg[k].first_item && item < a.seg[k].first_item + a.seg[k].nitems))
        k++;
    if (k == a.nseg) return;
    const ResampleSeg &g = a.seg[k];
    const long long lo = (item - g.first_item) * RS_CHUNK;
    const long long used = used_bytes(st, g, s);
    if (lo >= used) return;  // a chunk beyond this source's log: the host bound is a maximum over replicates
    copy_range(g.base + r * g.stride, g.base + s * g.stride, lo, lo + RS_CHUNK < used ? lo + RS_CHUNK : used);
}

cudaError_t launch_resample(const DevState &st, const int2 *pairs, int ndst, long long ev_bound, long long leap_bound,
                            long long dense_bound, cudaStream_t stream, int *nlaunch) {
    *nlaunch = 0;
    if (ndst <= 0) return cudaSuccess;
    const Dims &D = st.D;
    const long long K = D.K, KH = (long long)D.K * D.H, KS = (long long)D.K * D.S;
    ResampleArgs a;
    a.pairs = pairs;
    a.nseg = 0;
    a.items = 1;
    // bound: the largest used length of any replicate (bytes); fixed segments are always whole
    auto add = [&](void *base, long long stride, long long row, int kind, long long bound) {
        if (!base || stride <= 0) return;
        ResampleSeg &g = a.seg[a.nseg++];
        g.base = (char *)base;
        g.stride = stride;
        g.row = row;
        g.kind = kind;
        g.first_item = a.items;
        g.nitems = kind == SEG_FIXED && stride <= RS_CHUNK ? 0 : (int)((bound + RS_CHUNK - 1) / RS_CHUNK);
        a.items += g.nitems;
    };
    auto fixed = [&](void *base, long long bytes) { add(base, bytes, bytes, SEG_FIXED, bytes); };
    fixed(st.I, KH * 8);
    fixed(st.Sx, KS * 8);
    fixed(st.initI, KH * 8);
    fixed(st.initSx, KS * 8);
    fixed(st.cd, K * 8);
    fixed(st.lock, K * 4);
    fixed(st.eff, K * K * 8);
    fixed(st.ceff, K * 8);
    fixed(st.maxEBM, K * 8);
    fixed(st.time, 8);
    fixed(st.rate_tot, 16);
    fixed(st.counters, NCOUNT * 8);
    fixed(st.epoch, 4);
    fixed(st.err, 4);
    fixed(st.ev_base, 8);
    fixed(st.dense_base, 8);
    fixed(st.sp_n, 4);
    fixed(st.loc_n, 4);
    const long long ev = std::min(ev_bound, st.ev_cap), lp = std::min(leap_bound, st.leap_cap);
    add(st.ev_time, st.ev_cap * 8, 8, SEG_EVENTS, ev * 8);
    add(st.ev_desc, st.ev_cap * 8, 8, SEG_EVENTS, ev * 8);
    add(st.tau_tt, st.leap_cap * 16, 16, SEG_LEAPS, lp * 16);
    add(st.tau_counts, st.dense_cap * D.Pp * 4, (long long)D.Pp * 4, SEG_DENSE, std::min(dense_bound, st.dense_cap) * D.Pp * 4);
    add(st.sp_off, (st.leap_cap + 1) * 4, 4, SEG_SPOFF, (lp + 1) * 4);
    add(st.sp_ent, st.sp_cap * 8, 8, SEG_SPENT, st.sp_cap * 8);
    add(st.loc_sp, (long long)st.loc_cap * 4, 4, SEG_LOC, (long long)st.loc_cap * 4);
    add(st.loc_t, (long long)st.loc_cap * 8, 8, SEG_LOC, (long long)st.loc_cap * 8);
    // one launch unless the grid would pass 2^31 - 1 CTAs, then consecutive slices of the destination list
    const int per = (int)std::min<long long>(ndst, 2147483647LL / a.items);
    for (int d0 = 0; d0 < ndst; d0 += per) {
        const int nd = std::min(per, ndst - d0);
        a.pairs = pairs + d0;
        resample_kernel<<<(unsigned)((long long)nd * a.items), RS_THREADS, 0, stream>>>(st, a);
        ++*nlaunch;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

}  // namespace vg
