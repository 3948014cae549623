// Epidemic curves of every compartment of every replicate in ONE pass over the event logs.
//
// Replaces the reference's get_data_infectious / get_data_susceptible (src/_BirthDeath.pyx:1967-2045), which walk
// the whole log in a Python-level loop once per (deme, haplotype) query -- O(K*H) passes to draw one figure, and the
// consumer of the "epidemic curves" statistics of the distribution match (SURVEY §8d config 2, §8f rank 2).
//
// One warp per replicate.  The replicate's compartment counts live in the warp's slice of shared memory (int64):
// infectious I[K*H], susceptible S[K*S], and two cumulative tallies per infectious cell that the reference's
// curves expose through an operator-precedence quirk (removed = recoveries + samplings, sampled = samplings; see
// _engine.py get_data_infectious).  The log is read forward exactly once:
//   * direct-method rows: 16 B each (fp64 time + packed descriptor), 32 rows per warp load; rows are applied in
//     order by the lanes that hold them (the updates commute, only the grid crossings are ordered);
//   * MULTITYPE rows: the leap's dense row int32[P] is scanned with 16-byte loads, 8 in flight per lane (4 KB per
//     warp); the ~1 % non-zero counts are compacted into a per-warp queue (three ballots per round) and decoded
//     (logrec.cuh) and applied with shared-memory atomics 32 at a time, every lane busy.
// Grid: t_j = j * currentTime / step_num, j = 0..step_num (the reference's time_points).  The value at j is the
// state after every log row with time <= t_j; whenever the next row's time exceeds t_j the warp writes the
// snapshot of point j with coalesced 8-byte stores.  Points after the last row repeat the final state; the index
// of the point that holds the last row is returned so that the host wrapper can reproduce the reference's
// behaviour for them (it leaves them zero).
//
// Roofline: HBM read of the log (B_leap = 4P + 16 bytes per leap, 16 B per direct event) + the snapshot writes
// 8 * (3 K H + K S) * (step_num + 1) bytes per replicate.
//
// Trajectories (trajectories_kernel, TRAJ): the same walk on a grid the caller gives in absolute time, shared by every
// replicate, with a snapshot of marginals instead of every cell: infectious per deme and per haplotype, cumulative
// samplings per deme and per haplotype (2K + 2H int64 per point).  The slice holds I[K*H] and the K + H sampling
// counters (no susceptible counts, no per-cell tallies); a point after the replicate's currentTime was not simulated
// and is written as -1.  Roofline: the log once + 8 * (2K + 2H) * T bytes per replicate.
#include "common.cuh"
#include "handle.h"
#include "logrec.cuh"

namespace vg {

extern __shared__ __align__(16) unsigned char curves_smem[];

#define CURVE_QCAP 256  // >= 128 (one round of 32 int4 can add that many) 

struct CurveArgs {
    int rep_first, rep_count, step_num;
    long long *inf, *sus, *removed, *sampled;  // [rep_count][step_num+1][KH | KS | KH | KH], any may be null
    double *time_points;                       // [rep_count][step_num+1] or null
    int *last_point;                           // [rep_count] or null
};

struct TrajArgs {
    const double *times;  // [step_num + 1] the grid, absolute times, strictly increasing
    long long *out;       // [rep_count][step_num + 1][2K + 2H]
};

// TRAJ: no susceptible counts (Sx is not touched); rem = samplings per deme [K], smp = samplings per haplotype [H].
template <bool TRAJ>
__device__ __forceinline__ void curve_apply(int type, int hap, int pop, int nhap, int npop, long long n, int H, int S,
                                            unsigned long long *I, unsigned long long *Sx, unsigned long long *rem,
                                            unsigned long long *smp) {
    // unsigned wrap-around arithmetic == two's complement adds; the arrays are read back as signed
    const unsigned long long u = (unsigned long long)n, m = (unsigned long long)(-n);
    const int cell = pop * H + hap;
    if constexpr (TRAJ) {
        if (type == EV_BIRTH) {
            atomicAdd(&I[cell], u);
        } else if (type == EV_DEATH || type == EV_SAMPLING) {
            atomicAdd(&I[cell], m);
            if (type == EV_SAMPLING) {
                atomicAdd(&rem[pop], u);
                atomicAdd(&smp[hap], u);
            }
        } else if (type == EV_MUTATION) {
            atomicAdd(&I[cell], m);
            atomicAdd(&I[pop * H + nhap], u);
        } else if (type == EV_MIGRATION) {
            atomicAdd(&I[npop * H + hap], u);
        }
        return;
    }
    if (type == EV_BIRTH) {  // hap infects a susceptible of group nhap in deme pop
        atomicAdd(&I[cell], u);
        atomicAdd(&Sx[pop * S + nhap], m);
    } else if (type == EV_DEATH || type == EV_SAMPLING) {  // recovered go to group nhap = suscType[hap]
        atomicAdd(&I[cell], m);
        atomicAdd(&Sx[pop * S + nhap], u);
        if (rem) {  // the cumulative tallies exist only when one of them was asked for
            atomicAdd(&rem[cell], u);
            if (type == EV_SAMPLING) atomicAdd(&smp[cell], u);
        }
    } else if (type == EV_MUTATION) {
        atomicAdd(&I[cell], m);
        atomicAdd(&I[pop * H + nhap], u);
    } else if (type == EV_SUSCCHANGE) {  // group hap -> group nhap
        atomicAdd(&Sx[pop * S + hap], m);
        atomicAdd(&Sx[pop * S + nhap], u);
    } else if (type == EV_MIGRATION) {  // infection of a group-nhap susceptible of deme npop by haplotype hap of deme pop
        atomicAdd(&I[npop * H + hap], u);
        atomicAdd(&Sx[npop * S + nhap], m);
    }
}

// One trajectory point from the warp's slice: o[2K + 2H] = infectious per deme, per haplotype, samplings per deme, per
// haplotype (smp_deme and smp_hap are contiguous in the slice); every entry -1 for a point that was not simulated.
// Called by the whole warp.
__device__ __forceinline__ void traj_snapshot(const unsigned long long *I, const unsigned long long *smp, int K, int H,
                                              bool after_end, long long *o) {
    const int lane = threadIdx.x & 31;
    if (after_end) {
        for (int i = lane; i < 2 * (K + H); i += 32) o[i] = -1;
        return;
    }
    if (H >= 32) {  // a warp reduction per deme
        for (int p = 0; p < K; p++) {
            unsigned long long s = 0ull;
            for (int h = lane; h < H; h += 32) s += I[(size_t)p * H + h];
#pragma unroll
            for (int w = 16; w > 0; w >>= 1) s += __shfl_xor_sync(0xffffffffu, s, w);
            if (lane == 0) o[p] = (long long)s;
        }
    } else {  // a lane per deme
        for (int p = lane; p < K; p += 32) {
            unsigned long long s = 0ull;
            for (int h = 0; h < H; h++) s += I[p * H + h];
            o[p] = (long long)s;
        }
    }
    for (int h = lane; h < H; h += 32) {
        unsigned long long s = 0ull;
        for (int p = 0; p < K; p++) s += I[(size_t)p * H + h];
        o[K + h] = (long long)s;
    }
    for (int i = lane; i < K + H; i += 32) o[K + H + i] = (long long)smp[i];
}

// The replay; GSLICE: the warps' slices live in gslices (one per warp of the grid, curves_large_kernel: replicates whose
// counts do not fit one SM's shared memory), else in shared memory (curves_kernel).  TRAJ: the caller's grid ta.times
// and marginal snapshots into ta.out (trajectories_kernel); a.step_num is then the grid's last index.
template <bool GSLICE, bool TRAJ>
__device__ __forceinline__ void curves_body(const DevState &st, const CurveArgs &a, const TrajArgs &ta, int slice_bytes,
                                            unsigned char *gslices) {
    const Dims &D = st.D;
    const int K = D.K, H = D.H, S = D.S, KH = K * H, KS = K * S;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    unsigned long long *I = reinterpret_cast<unsigned long long *>(
        GSLICE ? gslices + (size_t)(blockIdx.x * nw + wid) * slice_bytes : curves_smem + (size_t)wid * slice_bytes);
    const bool tallies = !TRAJ && (a.removed != nullptr || a.sampled != nullptr);
    unsigned long long *Sx = I + KH, *rem = tallies ? Sx + KS : nullptr, *smp = tallies ? rem + KH : nullptr;
    // (channel, count) of the non-zero counts of the row being scanned
    int2 *queue = reinterpret_cast<int2 *>(tallies ? smp + KH : Sx + KS);
    if constexpr (TRAJ) {  // I[KH], samplings per deme [K] and per haplotype [H], queue
        Sx = nullptr;
        rem = I + KH;
        smp = rem + K;
        queue = reinterpret_cast<int2 *>(smp + H);
    }
    const int T = a.step_num;
    // the walk may snapshot every point of the caller's grid; the reference's last point (= currentTime) is never
    // crossed by a row and is written after the walk
    const int walk_end = TRAJ ? T + 1 : T;
    for (int q = blockIdx.x * nw + wid; q < a.rep_count; q += gridDim.x * nw) {
        const int r = a.rep_first + q;
        const double *pp = st.params + (size_t)st.rep_pp[r] * D.blob;
        const long long *I0 = (st.first_simulation ? st.initI : st.I) + (size_t)r * KH;
        const long long *S0 = (st.first_simulation ? st.initSx : st.Sx) + (size_t)r * KS;
        for (int i = lane; i < KH; i += 32) {
            I[i] = (unsigned long long)I0[i];
            if (tallies) {
                rem[i] = 0ull;
                smp[i] = 0ull;
            }
        }
        if constexpr (TRAJ)
            for (int i = lane; i < K + H; i += 32) rem[i] = 0ull;
        else
            for (int i = lane; i < KS; i += 32) Sx[i] = (unsigned long long)S0[i];
        __syncwarp();
        const long long n = st.counters[(size_t)r * NCOUNT + C_EVPTR];
        const double ct = st.time[r];
        const double *evt = st.ev_time + (size_t)r * st.ev_cap;
        const unsigned long long *evd = st.ev_desc + (size_t)r * st.ev_cap;
        if (a.time_points)
            for (int j = lane; j <= T; j += 32) a.time_points[(size_t)q * (T + 1) + j] = ((double)j * ct) / (double)T;
        int point = 0;
        auto grid = [&](int j) -> double {
            if constexpr (TRAJ)
                return ta.times[j];
            else
                return ((double)j * ct) / (double)T;
        };
        auto snapshot = [&](int j) {  // coalesced copy of the current state into point j
            __syncwarp();
            if constexpr (TRAJ) {
                traj_snapshot(I, rem, K, H, ta.times[j] > ct, ta.out + ((size_t)q * (T + 1) + j) * (2 * (K + H)));
                return;
            }
            const size_t o = (size_t)q * (T + 1) + j;
            if (a.inf)
                for (int i = lane; i < KH; i += 32) a.inf[o * KH + i] = (long long)I[i];
            if (a.removed)
                for (int i = lane; i < KH; i += 32) a.removed[o * KH + i] = (long long)rem[i];
            if (a.sampled)
                for (int i = lane; i < KH; i += 32) a.sampled[o * KH + i] = (long long)smp[i];
            if (a.sus)
                for (int i = lane; i < KS; i += 32) a.sus[o * KS + i] = (long long)Sx[i];
        };
        // point advances while time_points[point] < t (reference :1975-1978); the state before the row is point's value
        auto advance = [&](double t) {
            while (point != walk_end && grid(point) < t) {
                snapshot(point);
                point++;
            }
        };
        for (long long base = 0; base < n; base += 32) {
            if constexpr (TRAJ)
                if (point == walk_end) break;  // every grid point is written: the rest of the log is not needed
            const long long i = base + lane;
            double t = 0.0;
            unsigned long long d = 0ull;
            if (i < n) {
                t = evt[i];
                d = evd[i];
            }
            const int cnt = (int)((n - base < 32) ? n - base : 32);
            // does any row of this batch cross a grid point or carry a leap?  (times are non-decreasing)
            const double t_last = __shfl_sync(0xffffffffu, t, cnt - 1);
            const bool crosses = point != walk_end && grid(point) < t_last;
            const unsigned multi = __ballot_sync(0xffffffffu, i < n && (int)(d & 7) == EV_MULTITYPE);
            if (!crosses && multi == 0u) {  // fast path: 32 direct rows inside one grid interval, applied in parallel
                if (i < n) {
                    int ty, hp_, pp_, nh, np_;
                    unpack_event(d, ty, hp_, pp_, nh, np_);
                    curve_apply<TRAJ>(ty, hp_, pp_, nh, np_, 1, H, S, I, Sx, rem, smp);
                }
                continue;
            }
            for (int k = 0; k < cnt; k++) {  // ordered walk of the batch
                const double tk = __shfl_sync(0xffffffffu, t, k);
                const unsigned long long dk = __shfl_sync(0xffffffffu, d, k);
                advance(tk);
                const int ty = (int)(dk & 7);
                if (ty != EV_MULTITYPE) {
                    if (lane == 0) {
                        int t2, hp_, pp_, nh, np_;
                        unpack_event(dk, t2, hp_, pp_, nh, np_);
                        curve_apply<TRAJ>(t2, hp_, pp_, nh, np_, 1, H, S, I, Sx, rem, smp);
                    }
                    continue;
                }
                const long long leap = unpack_multi(dk), dbase = st.dense_base[r];
                if (leap < dbase) {  // archived leap: (channel, count) pairs, applied 32 at a time (order does not matter here)
                    const int *soff = st.sp_off + (size_t)r * (st.leap_cap + 1);
                    const int2 *ent = st.sp_ent + (size_t)r * st.sp_cap;
                    const int e1 = soff[leap + 1];
                    __syncwarp();
                    for (int e0 = soff[leap]; e0 < e1; e0 += 128) {  // four loads in flight per lane: one dependent 256-byte
                        int2 en[4];                                    // load per step made the walk latency-bound
#pragma unroll
                        for (int u = 0; u < 4; u++) {
                            const int e = e0 + u * 32 + lane;
                            en[u] = e < e1 ? __ldcs(ent + e) : make_int2(-1, 0);
                        }
#pragma unroll
                        for (int u = 0; u < 4; u++) {
                            if (en[u].x < 0) continue;
                            int mty, mh, mp, mnh, mnp;
                            decode_record(en[u].x, D, pp, mty, mh, mp, mnh, mnp);
                            curve_apply<TRAJ>(mty, mh, mp, mnh, mnp, (long long)en[u].y, H, S, I, Sx, rem, smp);
                        }
                    }
                    __syncwarp();
                    continue;
                }
                const int4 *row = reinterpret_cast<const int4 *>(st.tau_counts + ((size_t)r * st.dense_cap + (leap - dbase)) * D.Pp);
                const int n16 = D.Pp >> 2;
                int qn = 0;  // entries in the warp's queue (uniform)
                auto flush = [&]() {  // decode + apply the queued non-zero counts, 32 at a time with every lane busy
                    __syncwarp();
                    for (int e = lane; e < qn; e += 32) {
                        const int2 en = queue[e];
                        int mty, mh, mp, mnh, mnp;
                        decode_record(en.x, D, pp, mty, mh, mp, mnh, mnp);
                        curve_apply<TRAJ>(mty, mh, mp, mnh, mnp, (long long)en.y, H, S, I, Sx, rem, smp);
                    }
                    __syncwarp();
                    qn = 0;
                };
                const unsigned lt = (1u << lane) - 1u;
                int4 nxt[8];
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const int j = u * 32 + lane;
                    nxt[u] = j < n16 ? __ldcs(row + j) : make_int4(0, 0, 0, 0);  // streamed once: evict first
                }
                for (int b4 = 0; b4 < n16; b4 += 256) {
                    int4 v[8];
#pragma unroll
                    for (int u = 0; u < 8; u++) {  // this block arrives while the previous one was compacted
                        v[u] = nxt[u];
                        const int j = b4 + 256 + u * 32 + lane;
                        nxt[u] = j < n16 ? __ldcs(row + j) : make_int4(0, 0, 0, 0);
                    }
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        // compaction: a dense row holds ~1 % non-zero counts, decoding them where they lie would run the
                        // (division-heavy) decoder with one or two live lanes per pass
                        const int c0 = (b4 + u * 32 + lane) * 4;
                        const int cl = (v[u].x != 0) + (v[u].y != 0) + (v[u].z != 0) + (v[u].w != 0);
                        const unsigned b0 = __ballot_sync(0xffffffffu, cl & 1), b1 = __ballot_sync(0xffffffffu, cl & 2),
                                       b2 = __ballot_sync(0xffffffffu, cl & 4);
                        if ((b0 | b1 | b2) == 0u) continue;
                        const int tot = __popc(b0) + 2 * __popc(b1) + 4 * __popc(b2);
                        if (qn + tot > CURVE_QCAP) flush();
                        int pos = qn + __popc(b0 & lt) + 2 * __popc(b1 & lt) + 4 * __popc(b2 & lt);
                        if (v[u].x != 0) queue[pos++] = make_int2(c0, v[u].x);
                        if (v[u].y != 0) queue[pos++] = make_int2(c0 + 1, v[u].y);
                        if (v[u].z != 0) queue[pos++] = make_int2(c0 + 2, v[u].z);
                        if (v[u].w != 0) queue[pos++] = make_int2(c0 + 3, v[u].w);
                        qn += tot;
                    }
                }
                flush();
            }
        }
        __syncwarp();
        if (a.last_point && lane == 0) a.last_point[q] = point;
        for (int j = point; j <= T; j++) snapshot(j);
        __syncwarp();
    }
}

__global__ void __launch_bounds__(512, 1) curves_kernel(const DevState st, const CurveArgs a, int slice_bytes) {
    curves_body<false, false>(st, a, TrajArgs{}, slice_bytes, nullptr);
}

__global__ void __launch_bounds__(512, 1) curves_large_kernel(const DevState st, const CurveArgs a, int slice_bytes,
                                                               unsigned char *gslices) {
    curves_body<true, false>(st, a, TrajArgs{}, slice_bytes, gslices);
}

__global__ void __launch_bounds__(512, 1) trajectories_kernel(const DevState st, const CurveArgs a, const TrajArgs t,
                                                               int slice_bytes) {
    curves_body<false, true>(st, a, t, slice_bytes, nullptr);
}

__global__ void __launch_bounds__(512, 1) trajectories_large_kernel(const DevState st, const CurveArgs a, const TrajArgs t,
                                                                     int slice_bytes, unsigned char *gslices) {
    curves_body<true, true>(st, a, t, slice_bytes, gslices);
}

size_t curves_slice_bytes(const Dims &D, bool tallies) {
    const size_t ncell = tallies ? 3 : 1;  // I (+ removed, sampled) per infectious cell
    return ((ncell * D.K * D.H + (size_t)D.K * D.S) * 8 + CURVE_QCAP * 8 + 15) & ~(size_t)15;
}

size_t trajectories_slice_bytes(const Dims &D) {
    return (((size_t)D.K * D.H + D.K + D.H) * 8 + CURVE_QCAP * 8 + 15) & ~(size_t)15;
}

// One launch of the replay: shared-memory slices when one replicate's fits one SM, else the gslices scratch.
template <class Small, class Large, class... Extra>
static cudaError_t launch_replay(Small small, Large large, size_t slice_bytes, int rep_count, cudaStream_t stream,
                                 int num_sms, unsigned char *gslices, int nslices, const DevState &st, const CurveArgs &a,
                                 Extra... extra) {
    if (slice_bytes > 227 * 1024) {  // the state of one replicate does not fit one SM's shared memory
        if (!gslices || nslices < 1) return cudaErrorInvalidValue;
        int nw = (nslices + num_sms - 1) / num_sms;  // spread over the SMs, at most 16 warps per CTA
        if (nw > 16) nw = 16;
        int grid = nslices / nw;
        if (grid > (rep_count + nw - 1) / nw) grid = (rep_count + nw - 1) / nw;
        large<<<grid, nw * 32, 0, stream>>>(st, a, extra..., (int)slice_bytes, gslices);
        return cudaGetLastError();
    }
    const int slice = (int)slice_bytes;
    int nw = (227 * 1024) / slice;
    if (nw > 16) nw = 16;
    cudaError_t e = cudaFuncSetAttribute(small, cudaFuncAttributeMaxDynamicSharedMemorySize, nw * slice);
    if (e != cudaSuccess) return e;
    int per_sm = 1;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, small, nw * 32, (size_t)nw * slice);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    int grid = (rep_count + nw - 1) / nw;
    if (grid > num_sms * per_sm) grid = num_sms * per_sm;
    if (grid < 1) grid = 1;
    small<<<grid, nw * 32, (size_t)nw * slice, stream>>>(st, a, extra..., slice);
    return cudaGetLastError();
}

cudaError_t launch_curves(const DevState &st, int rep_first, int rep_count, int step_num, long long *inf, long long *sus,
                          long long *removed, long long *sampled, double *time_points, int *last_point,
                          cudaStream_t stream, int num_sms, unsigned char *gslices, int nslices) {
    CurveArgs a;
    a.rep_first = rep_first; a.rep_count = rep_count; a.step_num = step_num;
    a.inf = inf; a.sus = sus; a.removed = removed; a.sampled = sampled;
    a.time_points = time_points; a.last_point = last_point;
    return launch_replay(curves_kernel, curves_large_kernel, curves_slice_bytes(st.D, removed || sampled), rep_count,
                         stream, num_sms, gslices, nslices, st, a);
}

cudaError_t launch_trajectories(const DevState &st, const double *times, int npoints, long long *out, cudaStream_t stream,
                                int num_sms, unsigned char *gslices, int nslices) {
    CurveArgs a = {};
    a.rep_first = 0; a.rep_count = st.R; a.step_num = npoints - 1;
    TrajArgs t;
    t.times = times; t.out = out;
    return launch_replay(trajectories_kernel, trajectories_large_kernel, trajectories_slice_bytes(st.D), st.R, stream,
                         num_sms, gslices, nslices, st, a, t);
}

}  // namespace vg
