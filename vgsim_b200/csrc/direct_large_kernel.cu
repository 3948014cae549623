// Batched direct-method Gillespie for model shapes whose rate hierarchy does not fit one SM's shared memory
// (direct_kernel.cu holds every shape that does; launch_direct picks between the two).
//
// One WARP per replicate, replicates handed out through the same atomic work counter as direct_kernel.  The replicate's
// state lives in a per-warp slice of device memory (HBM / L2) that the handle owns, one slice per RESIDENT warp, so the
// scratch does not grow with R.  Nothing of size K*H is ever walked per event: the rates are factored so that an event
// touches O(1) cells and O(S) per-deme numbers.
//   birth weight of (p, h, s)   = c[p] Sx[p,s] * W_s[p,h],       W_s[p,h] = b[h] sigma[s,h] I[p,h]
//   non-birth weight of (p, h)  = N[p,h] = (d[h] + sr[h] sm[p] + tm[h]) I[p,h]
//   infectPopRate[p] = c[p] sum_s Sx[p,s] B[p,s] + N[p],  B[p,s] = sum_h W_s[p,h],  N[p] = sum_h N[p,h]
// Per deme there are S + 2 sum trees over h: the counts I (the migration source pick), N, and W_s for every group whose
// sigma row is not all zero (the others have B = 0 and are never built or read).  popRate[p] sits in one more tree over
// the demes; its root is totalRate, recomputed along one path per event (no drift).  Every tree is 32-ary: one level is
// one coalesced 256-byte warp load, a descent is one warp_pick per level carrying x - before down (Pick::rest), and an
// update recomputes each ancestor on the path as the warp_sum of its 32 children.  A node is therefore the same
// function of its leaves whatever the history, and a subtree of zero leaves sums to exactly 0 (never picked).
//
// An event: deme by popRate; immunity vs. infection as in direct_kernel; for an infection the class among
// [c Sx[p,s] B[p,s] ..., N[p]]; h by descent of that class's tree; for a non-birth death / sampling / mutation from the
// cell's three weights, then site and allele as direct_kernel does.  The joint law of (p, h, event, group) is the
// reference's (h first, then event, then group), so the two kernels agree in distribution, not draw for draw; each has
// its own Philox domain word.  Everything else (stop conditions, attempts / extinction retry / Restart, CheckLockdown,
// error bits, counters, the 32-event log bursts, the final rate_tot write) is direct_kernel's.
#include "common.cuh"
#include "handle.h"
#include "rates.cuh"
#include "choose.cuh"

namespace vg {

// ---------------------------------------------------------------------------------------------
// 32-ary sum tree over n leaves: level 0 holds the leaves, level l + 1 the sums of 32 consecutive nodes of level l, the
// top level has at most 32 nodes (their warp_sum is the root).  Every level starts on a 256-byte boundary.
__host__ __device__ inline Tree32 make_tree32(int n) {
    Tree32 T;
    int o = 0, l = 0;
    for (;;) {
        T.off[l] = o;
        T.n[l] = n;
        o += (n + 31) & ~31;
        l++;
        if (n <= 32) break;
        n = (n + 31) / 32;
    }
    T.depth = l;
    T.size = o;
    return T;
}

// Sets leaf i to v and recomputes its ancestors; returns the new root in every lane.  The siblings on the path are
// loaded up front (one memory latency), the path itself comes from the warp_sums.
__device__ __forceinline__ double tree_set(const Tree32 &T, double *t, int i, double v) {
    const int lane = threadIdx.x & 31;
    __syncwarp();  // an earlier update of this tree (same event, shared ancestors) is visible
    double sib[TREE32_MAXD];
#pragma unroll
    for (int l = 0; l < TREE32_MAXD; l++) {
        const int c = ((i >> (5 * l)) & ~31) + lane;
        sib[l] = (l < T.depth && c < T.n[l]) ? t[T.off[l] + c] : 0.0;
    }
#pragma unroll
    for (int l = 0; l < TREE32_MAXD; l++) {
        if (l < T.depth) {
            const int k = i >> (5 * l);
            if (lane == 0) t[T.off[l] + k] = v;
            v = warp_sum(lane == (k & 31) ? v : sib[l]);
        }
    }
    return v;
}

// Every level above the leaves from the leaves; returns the root in every lane.  32 nodes per round: lane j keeps node
// j of the round, so the loads of a round do not wait for stores.
__device__ __forceinline__ double tree_build(const Tree32 &T, double *t) {
    const int lane = threadIdx.x & 31;
#pragma unroll 1
    for (int l = 1; l < T.depth; l++) {
        const double *lo = t + T.off[l - 1];
        double *hi = t + T.off[l];
        const int n = T.n[l], nlo = T.n[l - 1];
        __syncwarp();
#pragma unroll 1
        for (int k0 = 0; k0 < n; k0 += 32) {
            double mine = 0.0;
#pragma unroll 8
            for (int j = 0; j < 32; j++) {
                const int c = (k0 + j) * 32 + lane;
                const double s = warp_sum(c < nlo ? lo[c] : 0.0);
                if (lane == j) mine = s;
            }
            if (k0 + lane < n) hi[k0 + lane] = mine;
        }
    }
    __syncwarp();
    const int top = T.depth - 1;
    return warp_sum(lane < T.n[top] ? t[T.off[top] + lane] : 0.0);
}

// The leaf that x in [0, root) falls into, by one warp_pick per level.  i = -1: every leaf is zero.
struct Leaf {
    int i;
    double z, w;  // the target inside the leaf, in [0, w), and the leaf's weight
    __device__ __forceinline__ double resid() const {  // fastChoose's residual of the pick
        const double r = z / w;
        return r < 0.0 ? 0.0 : (r >= 1.0 ? 0.9999999999999999 : r);
    }
};
__device__ __forceinline__ Leaf tree_pick(const Tree32 &T, const double *t, double x) {
    Leaf out;
    out.i = -1;
    out.z = out.w = 0.0;
    int k = 0;  // first node of the group searched at this level
#pragma unroll 1
    for (int l = T.depth - 1; l >= 0; l--) {
        const double *g = t + T.off[l] + k;
        const int n = T.n[l] - k < 32 ? T.n[l] - k : 32;
        const Pick pk = warp_pick([&](int i) { return g[i]; }, n, x);
        if (pk.i < 0) return out;
        x = pk.rest(x);
        if (l == 0) {
            out.i = k + pk.i;
            out.z = x;
            out.w = pk.w;
            return out;
        }
        k = (k + pk.i) * 32;
    }
    return out;
}

// ---------------------------------------------------------------------------------------------
// One warp's slice (doubles): K * nt haplotype trees, the deme tree, then the per-deme vectors.
DLLayout dl_layout(const Dims &D) {
    DLLayout L;
    L.th = make_tree32(D.H);
    L.tk = make_tree32(D.K);
    L.nt = D.S + 2;
    long long o = (long long)D.K * L.nt * L.th.size;
    auto take = [&](long long &f, long long n) {
        f = o;
        o += (n + 31) & ~31ll;
    };
    take(L.o_dtree, L.tk.size);
    take(L.o_tm, D.H);
    take(L.o_Sx, (long long)D.K * D.S);
    take(L.o_root, (long long)D.K * L.nt);
    take(L.o_totSus, D.K);
    take(L.o_imm, D.K);
    take(L.o_c, D.K);
    take(L.o_cd, D.K);
    take(L.o_maxEBM, D.K);
    take(L.o_lock, D.K);
    take(L.o_zs, D.S);
    L.slice = o;
    return L;
}

struct DLSlice {
    double *tree, *dtree, *tm, *Sx, *root, *totSus, *imm, *c, *cd, *maxEBM;
    int *lock, *zs;  // zs[s]: group s has a non-zero sigma row (its birth tree exists)
    __device__ __forceinline__ double *hap_tree(const DLLayout &L, int p, int j) const {
        return tree + ((size_t)p * L.nt + j) * L.th.size;
    }
};

__device__ __forceinline__ DLSlice dl_carve(const DLLayout &L, double *base) {
    DLSlice s;
    s.tree = base;
    s.dtree = base + L.o_dtree;
    s.tm = base + L.o_tm;
    s.Sx = base + L.o_Sx;
    s.root = base + L.o_root;
    s.totSus = base + L.o_totSus;
    s.imm = base + L.o_imm;
    s.c = base + L.o_c;
    s.cd = base + L.o_cd;
    s.maxEBM = base + L.o_maxEBM;
    s.lock = reinterpret_cast<int *>(base + L.o_lock);
    s.zs = reinterpret_cast<int *>(base + L.o_zs);
    return s;
}

// tree roots of deme p: j = 0 counts (totInf), 1 non-birth weights N, 2 + s birth weights B[p,s]
enum { TJ_I = 0, TJ_N = 1, TJ_W = 2 };

// popRate[p] = infectPopRate + immunePopRate from the roots (O(S)); imm: immunePopRate[p]
__device__ __forceinline__ double dl_pop_rate(const Dims &D, const DLLayout &L, const DLSlice &s, const double *pp, int p,
                                              double &imm) {
    const int S = D.S;
    const double *rt = s.root + (size_t)p * L.nt;
    double bs = 0.0, im = 0.0;
    for (int sn = 0; sn < S; sn++) {
        const double x = s.Sx[p * S + sn];
        bs += x * rt[TJ_W + sn];
        im += pp[D.o_Tc + sn] * x;
    }
    imm = im;
    return (s.c[p] * bs + rt[TJ_N]) + im;
}

// deme p's rates after a change of its cells or Sx: imm, the deme-tree leaf; returns totalRate (the new root)
__device__ __forceinline__ double dl_deme(const Dims &D, const DLLayout &L, const DLSlice &s, const double *pp, int p) {
    __syncwarp();  // roots written by lane 0
    double imm;
    const double pr = dl_pop_rate(D, L, s, pp, p, imm);
    if ((threadIdx.x & 31) == 0) s.imm[p] = imm;
    return tree_set(L.tk, s.dtree, p, pr);
}

// every deme's rates and the deme tree (after a lockdown flip changed c, or a rebuild); returns totalRate
__device__ __forceinline__ double dl_demes(const Dims &D, const DLLayout &L, const DLSlice &s, const double *pp) {
    __syncwarp();
    for (int p = threadIdx.x & 31; p < D.K; p += 32) {
        double imm;
        s.dtree[p] = dl_pop_rate(D, L, s, pp, p, imm);
        s.imm[p] = imm;
    }
    return tree_build(L.tk, s.dtree);
}

// cell (p, h) now holds In infectious: one leaf per tree of the deme, roots written by lane 0
__device__ __forceinline__ void dl_cell(const Dims &D, const DLLayout &L, const DLSlice &s, const double *pp, int p, int h,
                                        double In) {
    const bool l0 = (threadIdx.x & 31) == 0;
    double *rt = s.root + (size_t)p * L.nt;
    double v = tree_set(L.th, s.hap_tree(L, p, TJ_I), h, In);
    if (l0) rt[TJ_I] = v;
    const double base = pp[D.o_d + h] + pp[D.o_sr + h] * pp[D.o_sm + p] + s.tm[h];
    v = tree_set(L.th, s.hap_tree(L, p, TJ_N), h, base * In);
    if (l0) rt[TJ_N] = v;
    const double bI = pp[D.o_b + h] * In;
    for (int sn = 0; sn < D.S; sn++) {
        if (!s.zs[sn]) continue;
        v = tree_set(L.th, s.hap_tree(L, p, TJ_W + sn), h, bI * pp[D.o_sigT + sn * D.H + h]);
        if (l0) rt[TJ_W + sn] = v;
    }
}

// Every tree from the counts already in the count-tree leaves and the parameter point (state-independent rows first);
// returns totalRate.
__device__ __forceinline__ double dl_build(const Dims &D, const DLLayout &L, const DLSlice &s, const double *pp) {
    const int lane = threadIdx.x & 31, H = D.H, S = D.S, U = D.U;
    for (int h = lane; h < H; h += 32) {
        double m = 0.0;
        for (int u = 0; u < U; u++) m += pp[D.o_mu + h * U + u];  // tmRate (:306-308), direct_kernel's order
        s.tm[h] = m;
    }
    for (int sn = 0; sn < S; sn++) {
        int nz = 0;
        for (int h = lane; h < H; h += 32) nz |= pp[D.o_sigT + sn * H + h] != 0.0;
        nz = __any_sync(0xffffffffu, nz);
        if (lane == 0) s.zs[sn] = nz;
    }
    __syncwarp();
    for (int p = 0; p < D.K; p++) {
        const double *cnt = s.hap_tree(L, p, TJ_I);
        double *nt = s.hap_tree(L, p, TJ_N);
        const double smp = pp[D.o_sm + p];
        for (int h = lane; h < H; h += 32) {
            const double I = cnt[h];
            nt[h] = (pp[D.o_d + h] + pp[D.o_sr + h] * smp + s.tm[h]) * I;
            const double bI = pp[D.o_b + h] * I;
            for (int sn = 0; sn < S; sn++)
                if (s.zs[sn]) s.hap_tree(L, p, TJ_W + sn)[h] = bI * pp[D.o_sigT + sn * H + h];
        }
        double *rt = s.root + (size_t)p * L.nt;
        for (int j = 0; j < L.nt; j++) {
            const bool built = j < TJ_W || s.zs[j - TJ_W];
            const double v = built ? tree_build(L.th, s.hap_tree(L, p, j)) : 0.0;
            if (lane == 0) rt[j] = v;
        }
    }
    return dl_demes(D, L, s, pp);
}

// the two sums behind totalMigrationRate = G*A - B, and G (globalInfectious)
__device__ __forceinline__ void dl_mig_sums(const Dims &D, const DLLayout &L, const DLSlice &s, double &A, double &B,
                                            double &ginf) {
    __syncwarp();
    double a = 0.0, b = 0.0, g = 0.0;
    for (int q = threadIdx.x & 31; q < D.K; q += 32) {
        const double ti = s.root[(size_t)q * L.nt + TJ_I];
        const double ms = s.maxEBM[q] * s.totSus[q];
        a += ms;
        b += ms * ti;
        g += ti;
    }
    A = warp_sum(a);
    B = warp_sum(b);
    ginf = warp_sum(g);
}

// counts I of replicate r (or its Restart snapshot) into the count-tree leaves, Sx and its deme totals; returns whether a
// count does not fit int32
__device__ __forceinline__ bool dl_load_counts(const Dims &D, const DLLayout &L, const DLSlice &s, const long long *I,
                                               const long long *Sx) {
    const int lane = threadIdx.x & 31, H = D.H, S = D.S;
    int ovf = 0;
    for (int p = 0; p < D.K; p++) {
        double *cnt = s.hap_tree(L, p, TJ_I);
        for (int h = lane; h < H; h += 32) {
            const long long v = I[(size_t)p * H + h];
            if (v < 0 || v > 2147483647LL) ovf = 1;
            cnt[h] = (double)v;
        }
    }
    for (int i = lane; i < D.K * S; i += 32) {
        const long long v = Sx[i];
        if (v < 0 || v > 2147483647LL) ovf = 1;
        s.Sx[i] = (double)v;
    }
    __syncwarp();
    for (int p = lane; p < D.K; p += 32) {
        double ts = 0.0;
        for (int sn = 0; sn < S; sn++) ts += s.Sx[p * S + sn];
        s.totSus[p] = ts;
    }
    __syncwarp();
    return __any_sync(0xffffffffu, ovf) != 0;
}

__global__ void __launch_bounds__(512, 1) direct_large_kernel(const __grid_constant__ DevState st,
                                                               const __grid_constant__ SimArgs a,
                                                               const __grid_constant__ DLLayout L, double *slices, int *work) {
    const Dims &D = st.D;
    const int K = D.K, H = D.H, S = D.S, U = D.U;
    const int lane = threadIdx.x & 31;
    const DLSlice s = dl_carve(L, slices + (size_t)(blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * L.slice);

    for (;;) {
        int r = 0;
        if (lane == 0) r = atomicAdd(work, 1);
        r = __shfl_sync(0xffffffffu, r, 0);
        if (r >= st.R) break;
        const double *pp = st.params + (size_t)st.rep_pp[r] * D.blob;
        double *eff = st.eff + (size_t)r * K * K;
        long long *ctr = st.counters + (size_t)r * NCOUNT;
        const uint64_t seed = st.seeds[r];
        const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
        // ---- load and build
        __syncwarp();
        const bool ovf = dl_load_counts(D, L, s, st.I + (size_t)r * K * H, st.Sx + (size_t)r * K * S);
        for (int i = lane; i < K; i += 32) {
            s.cd[i] = st.cd[(size_t)r * K + i];
            s.c[i] = st.ceff[(size_t)r * K + i];
            s.maxEBM[i] = st.maxEBM[(size_t)r * K + i];
            s.lock[i] = st.lock[(size_t)r * K + i];
        }
        if (ovf) {
            if (lane == 0) st.err[r] |= ERR_COUNT_OVERFLOW;
            continue;
        }
        double Rt = dl_build(D, L, s, pp), mA, mB, ginf;
        dl_mig_sums(D, L, s, mA, mB, ginf);

        long long cB = ctr[C_B], cD = ctr[C_D], cS = ctr[C_S], cM = ctr[C_M], cI = ctr[C_I], cGp = ctr[C_MIGP],
                  cGn = ctr[C_MIGN];
        long long evptr = ctr[C_EVPTR], leaps = ctr[C_LEAPS], good_attempt = ctr[C_GOOD];
        int swaps = 0, errbits = 0;
        double t = st.time[r];
        unsigned epoch = st.epoch[r];
        const long long ev_limit = evptr + a.iterations < st.ev_cap ? evptr + a.iterations : st.ev_cap;
        const long long ev_base = st.ev_base[r];
        double *ev_time = st.ev_time + (size_t)r * st.ev_cap;
        unsigned long long *ev_desc = st.ev_desc + (size_t)r * st.ev_cap;
        int *loc_sp = st.loc_sp + (size_t)r * st.loc_cap;
        double *loc_t = st.loc_t + (size_t)r * st.loc_cap;
        double my_t = 0.0;
        unsigned long long my_d = 0ull;
        int nb = 0;
        auto flush_log = [&]() {
            if (lane < nb) {
                ev_time[evptr - nb + lane] = my_t;
                ev_desc[evptr - nb + lane] = my_d;
            }
            nb = 0;
        };
        auto totinf = [&](int q) { return s.root[(size_t)q * L.nt + TJ_I]; };
        // a lockdown flip changes c, eff and maxEBM: every deme's rate, no haplotype tree
        auto after_flip = [&]() {
            __syncwarp();
            update_contact_rates(WarpGroup(), D, pp, s.cd, eff, s.c, s.maxEBM);
            Rt = dl_demes(D, L, s, pp);
            dl_mig_sums(D, L, s, mA, mB, ginf);
        };

        for (long long attempt = 0; attempt < a.attempts; attempt++) {
            epoch++;
            unsigned long long iter = 0;
            double Rm = K > 1 ? fmax(ginf * mA - mB, 0.0) : 0.0;
            if (Rt + Rm != 0.0 && ginf != 0.0) {
                double Emine = 0.0, u2mine = 0.0;
                while (evptr < ev_limit && (a.sample_size == -1 || cS <= a.sample_size) && (!a.has_time || t < (double)a.time)) {
                    // ---- SampleTime + GenerateEvent (:476-512): two uniforms per iteration, iteration i on Philox block i
                    const int slot = (int)(iter & 31ull);
                    if (slot == 0) {
                        const unsigned long long it = iter + (unsigned)lane;
                        const uint4 w = philox4x32_10(make_uint4((uint32_t)it, (uint32_t)(it >> 32), epoch, 0x4C415247u), key);
                        double u1 = u53(w.x, w.y);
                        if (u1 <= 0.0) u1 = 1.0 / 9007199254740992.0;
                        Emine = -log(u1);
                        u2mine = u53(w.z, w.w);
                    }
                    const double E = __shfl_sync(0xffffffffu, Emine, slot);
                    const double u2 = __shfl_sync(0xffffffffu, u2mine, slot);
                    iter++;
                    if ((iter & 1023ull) == 0) {  // bound the drift of the incremental migration sums
                        dl_mig_sums(D, L, s, mA, mB, ginf);
                        Rm = K > 1 ? fmax(ginf * mA - mB, 0.0) : 0.0;
                    }
                    const double R = Rt + Rm;
                    t += E / R;
                    const double x = u2 * R;
                    int touched = -1;
                    double dS = 0.0, dI = 0.0;
                    bool logged = false;
                    unsigned long long desc = 0;
                    int ch = -1, ch2 = -1;  // haplotype of the changed cell(s) of deme `touched`
                    double In = 0.0, In2 = 0.0;  // their new counts
                    if (Rt > x) {
                        const Leaf pk = tree_pick(L.tk, s.dtree, x);
                        const int p = pk.i;
                        if (p < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                        double y = pk.z;  // in [0, popRate[p])
                        const double immp = s.imm[p];
                        if (immp > y) {
                            // ---- ImmunityTransition (:550-564)
                            const Pick ps = small_pick([&](int i) { return pp[D.o_Tc + i] * s.Sx[p * S + i]; }, S, y);
                            if (ps.i < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                            const int ssi = ps.i;
                            const double rn = ps.resid(y);
                            const Pick pt = small_pick([&](int i) { return pp[D.o_T + ssi * S + i]; }, S, rn * pp[D.o_Tc + ssi]);
                            if (pt.i < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                            const int tsi = pt.i;
                            if (lane == 0) {
                                s.Sx[p * S + ssi] -= 1.0;
                                s.Sx[p * S + tsi] += 1.0;
                            }
                            cI++;
                            desc = pack_event(EV_SUSCCHANGE, ssi, p, tsi, 0);
                        } else {
                            y -= immp;  // in [0, infectPopRate[p])
                            const double cp = s.c[p];
                            const double *rt = s.root + (size_t)p * L.nt;
                            // the class: birth into group 0..S-1, or S = one of the cell's other events
                            const Pick pc = small_pick([&](int i) { return i < S ? cp * s.Sx[p * S + i] * rt[TJ_W + i] : rt[TJ_N]; },
                                                       S + 1, y);
                            if (pc.i < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                            if (pc.i < S) {
                                // ---- Birth (:568-605) into group si, the haplotype by W_si[p,:]
                                const int si = pc.i;
                                const Leaf ph = tree_pick(L.th, s.hap_tree(L, p, TJ_W + si), pc.resid(y) * rt[TJ_W + si]);
                                const int h = ph.i;
                                if (h < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                                ch = h;
                                In = s.hap_tree(L, p, TJ_I)[h] + 1.0;
                                if (lane == 0) {
                                    s.Sx[p * S + si] -= 1.0;
                                    s.totSus[p] -= 1.0;
                                }
                                dS = -1.0;
                                dI = 1.0;
                                cB++;
                                desc = pack_event(EV_BIRTH, h, p, si, 0);
                            } else {
                                const Leaf ph = tree_pick(L.th, s.hap_tree(L, p, TJ_N), pc.rest(y));
                                const int h = ph.i;
                                if (h < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                                const double z = ph.z;  // in [0, N[p,h])
                                const double Ih = s.hap_tree(L, p, TJ_I)[h];
                                const double e1 = pp[D.o_d + h] * Ih, e2 = pp[D.o_sr + h] * pp[D.o_sm + p] * Ih,
                                             e3 = s.tm[h] * Ih;
                                // as direct_kernel: strict comparisons never pick a zero weight, a z past the total falls
                                // to the last positive one
                                const double c2 = e1 + e2;
                                int e = z < e1 ? 1 : z < c2 ? 2 : 3;
                                if (e == 3 && !(e3 > 0.0)) e = e2 > 0.0 ? 2 : 1;
                                Pick pe;
                                pe.i = e;
                                pe.before = e == 1 ? 0.0 : e == 2 ? e1 : c2;
                                pe.w = e == 1 ? e1 : e == 2 ? e2 : e3;
                                if (!(pe.w > 0.0)) { errbits |= ERR_ZERO_WEIGHT; break; }
                                ch = h;
                                if (e == 1 || e == 2) {
                                    // ---- Death / Sampling (:616-635)
                                    const int g = (int)pp[D.o_g + h];
                                    In = Ih - 1.0;
                                    if (lane == 0) {
                                        s.Sx[p * S + g] += 1.0;
                                        s.totSus[p] += 1.0;
                                    }
                                    dS = 1.0;
                                    dI = -1.0;
                                    if (e == 1) cD++; else cS++;
                                    desc = pack_event(e == 1 ? EV_DEATH : EV_SAMPLING, h, p, g, 0);
                                } else {
                                    // ---- Mutation (:640-667): site by mRate[h,:], then the allele by hapMutType[h,site,:]
                                    const double xm = pe.resid(z) * s.tm[h];
                                    const Pick pm = small_pick([&](int i) { return pp[D.o_mu + h * U + i]; }, U, xm);
                                    if (pm.i < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                                    const double *wv = pp + D.o_w + (h * U + pm.i) * 3;
                                    const Pick pa = small_pick([&](int i) { return wv[i]; }, 3, pm.resid(xm) * (wv[0] + wv[1] + wv[2]));
                                    if (pa.i < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                                    const int nh = mutate_hap(h, pm.i, pa.i, U);
                                    In = Ih - 1.0;
                                    ch2 = nh;
                                    In2 = s.hap_tree(L, p, TJ_I)[nh] + 1.0;
                                    cM++;
                                    desc = pack_event(EV_MUTATION, h, p, nh, 0);
                                }
                            }
                        }
                        logged = true;
                        touched = p;
                    } else {
                        // ---- GenerateMigration (:672-694): rejection-sampled cross-deme infection
                        auto mpw = [&](int i) { return s.maxEBM[i] * s.totSus[i] * (ginf - totinf(i)); };
                        double sum = 0.0;
                        for (int q = lane; q < K; q += 32) sum += mpw(q);
                        sum = warp_sum(sum);  // exact totalMigrationRate of the current state
                        double rn = (x - Rt) / Rm;
                        rn = rn < 0.0 ? 0.0 : (rn >= 1.0 ? 0.9999999999999999 : rn);
                        const double xm = rn * sum;
                        const Pick pt = warp_pick(mpw, K, xm);
                        const int tp = pt.i;
                        if (tp < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                        rn = pt.resid(xm);
                        const double xs = rn * (ginf - totinf(tp));
                        const Pick psrc = warp_pick(totinf, K, xs, tp);
                        const int sp = psrc.i;
                        if (sp < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                        rn = psrc.resid(xs);
                        const Leaf ph = tree_pick(L.th, s.hap_tree(L, sp, TJ_I), rn * totinf(sp));
                        const int h = ph.i;
                        if (h < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                        rn = ph.resid();
                        const double xg = rn * s.totSus[tp];
                        const Pick pg = small_pick([&](int i) { return s.Sx[tp * S + i]; }, S, xg);
                        const int si = pg.i;
                        if (si < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                        rn = pg.resid(xg);
                        const double p_accept = eff[sp * K + tp] * pp[D.o_b + h] * pp[D.o_sigT + si * H + h] / s.maxEBM[tp];
                        touched = tp;  // the reference runs CheckLockdown on the target deme either way (:694)
                        if (rn < p_accept) {
                            ch = h;
                            In = s.hap_tree(L, tp, TJ_I)[h] + 1.0;
                            if (lane == 0) {
                                s.Sx[tp * S + si] -= 1.0;
                                s.totSus[tp] -= 1.0;
                            }
                            dS = -1.0;
                            dI = 1.0;
                            cGp++;
                            desc = pack_event(EV_MIGRATION, h, sp, si, tp);
                            logged = true;
                        } else {
                            cGn++;
                        }
                    }
                    if (logged) {
                        if (lane == nb) {
                            my_t = t;
                            my_d = desc;
                        }
                        nb++;
                        evptr++;
                        if (nb == 32) flush_log();
                        // ---- UpdateRates (:516-546): the changed cells' leaves, the deme's O(S) combination, one path of
                        // the deme tree; the migration sums by increments
                        const int p = touched;
                        if (ch >= 0) dl_cell(D, L, s, pp, p, ch, In);
                        if (ch2 >= 0) dl_cell(D, L, s, pp, p, ch2, In2);
                        Rt = dl_deme(D, L, s, pp, p);
                        if (dI != 0.0) {
                            const double Sn = s.totSus[p], Ip = totinf(p);
                            const double m = s.maxEBM[p];
                            mA += m * dS;
                            mB += m * (Sn * Ip - (Sn - dS) * (Ip - dI));
                            ginf += dI;
                            Rm = K > 1 ? fmax(ginf * mA - mB, 0.0) : 0.0;
                        }
                        __syncwarp();
                        if (Rt <= 0.0 || ginf == 0.0) break;
                    }
                    // ---- CheckLockdown(pi) (:412, :698-710)
                    {
                        __syncwarp();
                        const double ti = totinf(touched);
                        const int lk = s.lock[touched];
                        if ((ti > pp[D.o_startN + touched] && lk == 0) || (ti < pp[D.o_endN + touched] && lk == 1)) {
                            int flips = 0;
                            if (lane == 0)
                                flips = check_lockdown(D, pp, touched, (long long)ti, s.cd, s.lock, t, &st.loc_n[r], loc_sp, loc_t,
                                                       st.loc_cap, &st.err[r]);
                            flips = __shfl_sync(0xffffffffu, flips, 0);
                            if (flips) {
                                swaps += flips;
                                after_flip();
                                Rm = K > 1 ? fmax(ginf * mA - mB, 0.0) : 0.0;
                            }
                        }
                    }
                }
            }
            if (errbits) break;
            // ---- extinction retry (:414-418) and Restart (:714-738)
            if (evptr + ev_base <= 100 && a.iterations > 100) {
                evptr = 0;
                nb = 0;
                leaps = 0;
                cB = cD = cS = cM = cI = cGp = cGn = 0;
                t = 0.0;
                __syncwarp();
                dl_load_counts(D, L, s, st.initI + (size_t)r * K * H, st.initSx + (size_t)r * K * S);
                Rt = dl_build(D, L, s, pp);
                dl_mig_sums(D, L, s, mA, mB, ginf);
                int flips = 0;
                if (lane == 0)
                    for (int p = 0; p < K; p++)
                        flips += check_lockdown(D, pp, p, (long long)totinf(p), s.cd, s.lock, t, &st.loc_n[r], loc_sp, loc_t,
                                                st.loc_cap, &st.err[r]);
                flips = __shfl_sync(0xffffffffu, flips, 0);
                if (flips) {
                    swaps += flips;
                    after_flip();
                }
                good_attempt = 0;
                if (lane == 0) {  // the tau log of the wiped run goes with it, as in the tau kernels
                    st.dense_base[r] = 0;
                    st.sp_n[r] = 0;
                }
            } else {
                good_attempt = attempt + 1;
                break;
            }
        }
        flush_log();

        // ---- commit
        __syncwarp();
        for (int p = 0; p < K; p++) {
            const double *cnt = s.hap_tree(L, p, TJ_I);
            for (int h = lane; h < H; h += 32) st.I[(size_t)r * K * H + (size_t)p * H + h] = (long long)cnt[h];
        }
        for (int i = lane; i < K * S; i += 32) st.Sx[(size_t)r * K * S + i] = (long long)s.Sx[i];
        for (int i = lane; i < K; i += 32) {
            st.cd[(size_t)r * K + i] = s.cd[i];
            st.ceff[(size_t)r * K + i] = s.c[i];
            st.maxEBM[(size_t)r * K + i] = s.maxEBM[i];
            st.lock[(size_t)r * K + i] = s.lock[i];
        }
        if (lane == 0) {
            ctr[C_B] = cB; ctr[C_D] = cD; ctr[C_S] = cS; ctr[C_M] = cM; ctr[C_I] = cI;
            ctr[C_MIGP] = cGp; ctr[C_MIGN] = cGn;
            ctr[C_SWAP] += swaps;
            ctr[C_GOOD] = good_attempt;
            ctr[C_EVPTR] = evptr;
            ctr[C_LEAPS] = leaps;
            ctr[C_GINF] = (long long)ginf;
            st.time[r] = t;
            st.epoch[r] = epoch;
            if (errbits) st.err[r] |= errbits;
            st.rate_tot[2 * (size_t)r] = Rt;
            st.rate_tot[2 * (size_t)r + 1] = K > 1 ? fmax(ginf * mA - mB, 0.0) : 0.0;
        }
        __syncwarp();
    }
}

// Deterministic parity tap on the factored rates: the trees of replicate r's current state, built as the kernel builds
// them, and the reference's rate hierarchy (UpdateAllRates, :279-351) from them.  hapPopRate[p,h] = c[p] sum_s Sx[p,s]
// W_s[p,h] + N[p,h]; popRate and totalRate are the deme tree's leaves and root.
__global__ void rates_large_kernel(const __grid_constant__ DevState st, const __grid_constant__ DLLayout L, double *slice,
                                   int r, double *ev, double *hp, double *popRate, double *migPop, double *totals) {
    const Dims &D = st.D;
    const int lane = threadIdx.x & 31, K = D.K, H = D.H, S = D.S;
    const DLSlice s = dl_carve(L, slice);
    const double *pp = st.params + (size_t)st.rep_pp[r] * D.blob;
    dl_load_counts(D, L, s, st.I + (size_t)r * K * H, st.Sx + (size_t)r * K * S);
    for (int i = lane; i < K; i += 32) {
        s.c[i] = st.ceff[(size_t)r * K + i];
        s.maxEBM[i] = st.maxEBM[(size_t)r * K + i];
    }
    __syncwarp();
    const double Rt = dl_build(D, L, s, pp);
    double A, B, ginf;
    dl_mig_sums(D, L, s, A, B, ginf);
    for (int p = 0; p < K; p++) {
        const double cp = s.c[p];
        const double *nt = s.hap_tree(L, p, TJ_N);
        for (int h = lane; h < H; h += 32) {
            const size_t i = (size_t)p * H + h;
            double Q = 0.0, bs = 0.0;
            for (int sn = 0; sn < S; sn++) {
                const double x = s.Sx[p * S + sn];
                Q += x * pp[D.o_sigT + sn * H + h];
                if (s.zs[sn]) bs += x * s.hap_tree(L, p, TJ_W + sn)[h];
            }
            ev[i * 4 + 0] = pp[D.o_b + h] * (Q * cp);
            ev[i * 4 + 1] = pp[D.o_d + h];
            ev[i * 4 + 2] = pp[D.o_sr + h] * pp[D.o_sm + p];
            ev[i * 4 + 3] = s.tm[h];
            hp[i] = cp * bs + nt[h];
        }
    }
    double y = 0.0;
    for (int p = lane; p < K; p += 32) {
        popRate[p] = s.dtree[p];
        const double m = s.maxEBM[p] * s.totSus[p] * (ginf - s.root[(size_t)p * L.nt + TJ_I]);
        migPop[p] = m;
        y += m;
    }
    y = warp_sum(y);
    if (lane == 0) {
        totals[0] = Rt;
        totals[1] = y;
    }
}

// nwarps: slices available; the warps are spread over the SMs, at most 16 per CTA (one CTA per SM)
cudaError_t launch_direct_large(const DevState &st, const SimArgs &a, const DLLayout &L, double *slices, int nwarps,
                                int num_sms, cudaStream_t stream, int *work) {
    if (nwarps < 1) return cudaErrorInvalidValue;
    int wpc = (nwarps + num_sms - 1) / num_sms;
    if (wpc > 16) wpc = 16;
    cudaError_t e = cudaMemsetAsync(work, 0, sizeof(int), stream);
    if (e != cudaSuccess) return e;
    direct_large_kernel<<<nwarps / wpc, wpc * 32, 0, stream>>>(st, a, L, slices, work);
    return cudaGetLastError();
}

cudaError_t launch_rates_large(const DevState &st, const DLLayout &L, double *slice, int r, double *ev, double *hp,
                               double *popRate, double *migPop, double *totals, cudaStream_t stream) {
    rates_large_kernel<<<1, 32, 0, stream>>>(st, L, slice, r, ev, hp, popRate, migPop, totals);
    return cudaGetLastError();
}

}  // namespace vg
