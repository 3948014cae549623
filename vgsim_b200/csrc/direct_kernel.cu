// Batched direct-method Gillespie (reference SimulatePopulation, src/_BirthDeath.pyx:396-738).
//
// One WARP per replicate; replicates are handed out through an atomic work counter (a batch ends with its LONGEST
// replicate -- epidemic sizes at a fixed time are heavy-tailed -- so what this kernel optimises is the length of the
// dependent chain of ONE event, and free warps pick up the next replicate instead of a fixed share).
//
// The rate hierarchy of the reference
//     totalRate -> popRate[p] -> {immunePopRate[p], infectPopRate[p]} -> hapPopRate[p,h] -> eventHapPopRate[p,h,0:4]
// lives in shared memory as fp64 (counts included: they are exact in fp64 and the chain needs no int<->double
// conversions); the parameter point is staged once per CTA.  An event is:
//   1. one Philox4x32-10 block = two 53-bit uniforms (time step, event choice), like SampleTime / GenerateEvent (:476-512);
//   2. the cumulative searches of fastChoose as lane-parallel scans (choose.cuh).  The reference recycles ONE uniform
//      through all levels by dividing the residual by the picked weight; where the next level's total IS the picked
//      weight the quotient cancels, so the hot levels carry (x - prefix) down instead -- the same draw without a
//      division on the chain.  Cold levels (mutation site / allele, immunity transition, migration) use the reference's
//      residual form;
//   3. the state change by one lane; the refresh of the touched deme (UpdateRates, :516-546) in O(H*S/32) with the
//      contact factor c[p] = sum_r m[p,r]^2 cd[r]/A[r] hoisted; the totals by increments:
//      totalRate += popRate'[p] - popRate[p], and totalMigrationRate = sum_q maxEBM[q] totSus[q] (G - totInf[q])
//      = G*A - B with A, B updated in O(1) (all recomputed from scratch every 1024 iterations to bound drift);
//   4. the 16-byte log record (fp64 time + packed descriptor) parked in a lane's registers -- event n of a burst in
//      lane n -- and written as 2 x 256-byte coalesced stores every 32 events.
#include "common.cuh"
#include "handle.h"
#include "rates.cuh"
#include "choose.cuh"

namespace vg {

struct DirLayout {
    int nwarps, par_shared, pp0;
    int o_par, par_bytes, o_warp0, warp_bytes, total_bytes;
    // parameter block (bytes)
    int p_b, p_d, p_sr, p_tm, p_sig, p_base, p_Tc, p_T, p_sm, p_startN, p_endN, p_g;
    // warp slice (bytes)
    int w_I, w_hp, w_Sx, w_inf, w_imm, w_pr, w_cd, w_c, w_maxEBM, w_totInf, w_totSus, w_lock;
};

inline DirLayout dir_layout(const Dims &D, bool par_shared, int pp0, int max_bytes, int max_warps) {
    DirLayout L;
    const int K = D.K, H = D.H, S = D.S;
    int o = 0;
    auto take = [&](int &f, int bytes) {
        o = (o + 7) & ~7;
        f = o;
        o += bytes;
    };
    take(L.p_b, H * 8); take(L.p_d, H * 8); take(L.p_sr, H * 8); take(L.p_tm, H * 8); take(L.p_sig, S * H * 8);
    take(L.p_base, K * H * 8); take(L.p_Tc, S * 8); take(L.p_T, S * S * 8); take(L.p_sm, K * 8);
    take(L.p_startN, K * 8); take(L.p_endN, K * 8); take(L.p_g, H * 4);
    L.par_bytes = (o + 15) & ~15;
    o = par_shared ? 0 : L.par_bytes;
    take(L.w_I, K * H * 8); take(L.w_hp, K * H * 8); take(L.w_Sx, K * S * 8); take(L.w_inf, K * 8); take(L.w_imm, K * 8);
    take(L.w_pr, K * 8); take(L.w_cd, K * 8); take(L.w_c, K * 8); take(L.w_maxEBM, K * 8); take(L.w_totInf, K * 8);
    take(L.w_totSus, K * 8); take(L.w_lock, K * 4);
    L.warp_bytes = (o + 15) & ~15;
    L.par_shared = par_shared ? 1 : 0;
    L.pp0 = pp0;
    L.o_par = 0;
    L.o_warp0 = par_shared ? L.par_bytes : 0;
    int nw = (max_bytes - L.o_warp0) / L.warp_bytes;
    if (nw > max_warps) nw = max_warps;
    L.nwarps = nw;
    L.total_bytes = L.o_warp0 + (nw > 0 ? nw : 0) * L.warp_bytes;
    return L;
}

struct DirShared {
    // parameter point
    const double *b, *d, *sr, *tm, *sig, *base, *Tc, *T, *sm, *startN, *endN;
    const int *g;
    // replicate
    double *I, *hp, *Sx, *inf, *imm, *pr, *cd, *c, *maxEBM, *totInf, *totSus;
    int *lock;
};

__device__ __forceinline__ void dir_carve(DirShared &s, const DirLayout &L, unsigned char *smem, int wib) {
    unsigned char *pb = smem + (L.par_shared ? L.o_par : L.o_warp0 + wib * L.warp_bytes);
    unsigned char *wb = smem + L.o_warp0 + wib * L.warp_bytes;
    auto P = [&](int o) { return reinterpret_cast<const double *>(pb + o); };
    auto W = [&](int o) { return reinterpret_cast<double *>(wb + o); };
    s.b = P(L.p_b); s.d = P(L.p_d); s.sr = P(L.p_sr); s.tm = P(L.p_tm); s.sig = P(L.p_sig); s.base = P(L.p_base);
    s.Tc = P(L.p_Tc); s.T = P(L.p_T); s.sm = P(L.p_sm); s.startN = P(L.p_startN); s.endN = P(L.p_endN);
    s.g = reinterpret_cast<const int *>(pb + L.p_g);
    s.I = W(L.w_I); s.hp = W(L.w_hp); s.Sx = W(L.w_Sx); s.inf = W(L.w_inf); s.imm = W(L.w_imm); s.pr = W(L.w_pr);
    s.cd = W(L.w_cd); s.c = W(L.w_c); s.maxEBM = W(L.w_maxEBM); s.totInf = W(L.w_totInf); s.totSus = W(L.w_totSus);
    s.lock = reinterpret_cast<int *>(wb + L.w_lock);
}

// stage one parameter point (blob layout of common.cuh); t / n: thread index / count of the staging group
__device__ __forceinline__ void dir_load_params(const Dims &D, const DirLayout &L, unsigned char *pb, const double *pp, int t,
                                                int n) {
    const int K = D.K, H = D.H, S = D.S, U = D.U;
    double *b = reinterpret_cast<double *>(pb + L.p_b), *d = reinterpret_cast<double *>(pb + L.p_d);
    double *sr = reinterpret_cast<double *>(pb + L.p_sr), *tm = reinterpret_cast<double *>(pb + L.p_tm);
    double *sig = reinterpret_cast<double *>(pb + L.p_sig), *base = reinterpret_cast<double *>(pb + L.p_base);
    double *Tc = reinterpret_cast<double *>(pb + L.p_Tc), *T = reinterpret_cast<double *>(pb + L.p_T);
    double *sm = reinterpret_cast<double *>(pb + L.p_sm), *startN = reinterpret_cast<double *>(pb + L.p_startN);
    double *endN = reinterpret_cast<double *>(pb + L.p_endN);
    int *g = reinterpret_cast<int *>(pb + L.p_g);
    for (int h = t; h < H; h += n) {
        b[h] = pp[D.o_b + h];
        d[h] = pp[D.o_d + h];
        sr[h] = pp[D.o_sr + h];
        g[h] = (int)pp[D.o_g + h];
        double m = 0.0;
        for (int u = 0; u < U; u++) m += pp[D.o_mu + h * U + u];  // tmRate (:306-308)
        tm[h] = m;
    }
    for (int i = t; i < S * H; i += n) sig[i] = pp[D.o_sigT + i];
    for (int i = t; i < S * S; i += n) T[i] = pp[D.o_T + i];
    for (int i = t; i < S; i += n) Tc[i] = pp[D.o_Tc + i];
    for (int i = t; i < K; i += n) {
        sm[i] = pp[D.o_sm + i];
        startN[i] = pp[D.o_startN + i];
        endN[i] = pp[D.o_endN + i];
    }
    // the state-independent part of tEventHapPopRate[p,h] (:310-314): death + sampling + mutation
    for (int i = t; i < K * H; i += n) {
        const int p = i / H, h = i - p * H;
        double m = 0.0;
        for (int u = 0; u < U; u++) m += pp[D.o_mu + h * U + u];
        base[i] = pp[D.o_d + h] + pp[D.o_sr + h] * pp[D.o_sm + p] + m;
    }
}

// Q[p,h] = sum_s Sx[p,s] sigma[s,h]: the susceptible pressure on haplotype h in deme p (inner sum of BirthRate, :382-392)
// SC: the number of susceptibility groups when it is a compile-time constant (1..4: the loops over groups unroll and
// their address arithmetic folds), 0: taken from D at run time.
template <int SC>
__device__ __forceinline__ double dir_Q(const Dims &D, const DirShared &s, int p, int h) {
    const int S = SC > 0 ? SC : D.S;
    double Q = 0.0;
#pragma unroll
    for (int sn = 0; sn < S; sn++) Q += s.Sx[p * S + sn] * s.sig[sn * D.H + h];
    return Q;
}

// hapPopRate[p,:] and its sum from the current compartments (UpdateRates(pi, infect=True), :516-546); every lane
// returns infectPopRate[p].  Ends without a barrier: the caller syncs before anyone reads hp.
template <int SC>
__device__ __forceinline__ double dir_refresh_hp(const Dims &D, const DirShared &s, int p) {
    const int lane = threadIdx.x & 31, H = D.H;
    const double cp = s.c[p];
    double acc = 0.0;
    for (int h = lane; h < H; h += 32) {
        const double te = s.b[h] * (dir_Q<SC>(D, s, p, h) * cp) + s.base[p * H + h];
        const double v = te * s.I[p * H + h];
        s.hp[p * H + h] = v;
        acc += v;
    }
    return warp_sum(acc);
}

template <int SC>
__device__ __forceinline__ double dir_imm(const Dims &D, const DirShared &s, int p) {
    const int S = SC > 0 ? SC : D.S;
    double im = 0.0;
#pragma unroll
    for (int sn = 0; sn < S; sn++) im += s.Tc[sn] * s.Sx[p * S + sn];
    return im;
}

// the three totals from the per-deme arrays: totalRate and the two sums behind totalMigrationRate = G*A - B
__device__ __forceinline__ void dir_totals(const Dims &D, const DirShared &s, double &Rt, double &A, double &B) {
    const int lane = threadIdx.x & 31;
    double a = 0.0, b = 0.0, r2 = 0.0;
    for (int q = lane; q < D.K; q += 32) {
        const double ms = s.maxEBM[q] * s.totSus[q];
        a += ms;
        b += ms * s.totInf[q];
        r2 += s.pr[q];
    }
    A = warp_sum(a);
    B = warp_sum(b);
    Rt = warp_sum(r2);
}

// everything derived from the compartments (UpdateAllRates, :279-351, state-dependent part): per-deme totals, hp, inf,
// imm, pr, the totals and globalInfectious
template <int SC>
__device__ __forceinline__ void dir_refresh_all(const Dims &D, const DirShared &s, double &Rt, double &A, double &B,
                                                double &ginf) {
    const int lane = threadIdx.x & 31, K = D.K, H = D.H, S = D.S;
    __syncwarp();
    double g = 0.0;
    for (int p = 0; p < K; p++) {
        double ti = 0.0, ts = 0.0;
        for (int h = lane; h < H; h += 32) ti += s.I[p * H + h];
        for (int sn = lane; sn < S; sn += 32) ts += s.Sx[p * S + sn];
        ti = warp_sum(ti);
        ts = warp_sum(ts);
        const double inf = dir_refresh_hp<SC>(D, s, p);
        const double imm = dir_imm<SC>(D, s, p);
        if (lane == 0) {
            s.totInf[p] = ti;
            s.totSus[p] = ts;
            s.inf[p] = inf;
            s.imm[p] = imm;
            s.pr[p] = inf + imm;
        }
        g += ti;
    }
    __syncwarp();
    dir_totals(D, s, Rt, A, B);
    ginf = g;
}

// 16 warps per CTA (one CTA per SM): the event loop is one dependent chain per replicate
template <int SC>
__global__ void __launch_bounds__(512, 1) direct_kernel(const __grid_constant__ DevState st, const __grid_constant__ SimArgs a,
                                                         const __grid_constant__ DirLayout L, int *work) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const Dims &D = st.D;
    const int K = D.K, H = D.H, S = SC > 0 ? SC : D.S, U = D.U;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    DirShared s;
    dir_carve(s, L, smem_raw, wib);
    if (L.par_shared) {
        dir_load_params(D, L, smem_raw + L.o_par, st.params + (size_t)L.pp0 * D.blob, threadIdx.x, blockDim.x);
        __syncthreads();
    }

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
        // ---- load
        __syncwarp();
        if (!L.par_shared) dir_load_params(D, L, smem_raw + L.o_warp0 + wib * L.warp_bytes, pp, lane, 32);
        int ovf = 0;
        for (int i = lane; i < K * H; i += 32) {
            const long long v = st.I[(size_t)r * K * H + i];
            if (v < 0 || v > 2147483647LL) ovf = 1;
            s.I[i] = (double)v;
        }
        for (int i = lane; i < K * S; i += 32) {
            const long long v = st.Sx[(size_t)r * K * S + i];
            if (v < 0 || v > 2147483647LL) ovf = 1;
            s.Sx[i] = (double)v;
        }
        for (int i = lane; i < K; i += 32) {
            s.cd[i] = st.cd[(size_t)r * K + i];
            s.c[i] = st.ceff[(size_t)r * K + i];
            s.maxEBM[i] = st.maxEBM[(size_t)r * K + i];
            s.lock[i] = st.lock[(size_t)r * K + i];
        }
        __syncwarp();
        if (__any_sync(0xffffffffu, ovf)) {
            if (lane == 0) st.err[r] |= ERR_COUNT_OVERFLOW;
            continue;
        }
        double Rt, mA, mB, ginf;
        dir_refresh_all<SC>(D, s, Rt, mA, mB, ginf);

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
        // log burst: event n of the burst sits in lane n's registers until 32 are there
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

        for (long long attempt = 0; attempt < a.attempts; attempt++) {
            epoch++;
            unsigned long long iter = 0;
            double Rm = K > 1 ? fmax(ginf * mA - mB, 0.0) : 0.0;
            if (Rt + Rm != 0.0 && ginf != 0.0) {
                // Random numbers for 32 iterations at a time, one iteration per LANE: lane l holds the exponential variate
                // and the choice uniform of iteration base + l (iteration i always uses Philox block i, so the stream does
                // not depend on this batching).  One Philox call, one log per 32 events and lane instead of one per event.
                double Emine = 0.0, u2mine = 0.0;
                while (evptr < ev_limit && (a.sample_size == -1 || cS <= a.sample_size) && (!a.has_time || t < (double)a.time)) {
                    // ---- SampleTime + GenerateEvent (:476-512): two uniforms per iteration
                    const int slot = (int)(iter & 31ull);
                    if (slot == 0) {
                        const unsigned long long it = iter + (unsigned)lane;
                        const uint4 w = philox4x32_10(make_uint4((uint32_t)it, (uint32_t)(it >> 32), epoch, 0x44495245u), key);
                        double u1 = u53(w.x, w.y);
                        if (u1 <= 0.0) u1 = 1.0 / 9007199254740992.0;
                        Emine = -log(u1);
                        u2mine = u53(w.z, w.w);
                    }
                    const double E = __shfl_sync(0xffffffffu, Emine, slot);
                    const double u2 = __shfl_sync(0xffffffffu, u2mine, slot);
                    iter++;
                    if ((iter & 1023ull) == 0) {  // bound the drift of the incremental totals
                        dir_totals(D, s, Rt, mA, mB);
                        Rm = K > 1 ? fmax(ginf * mA - mB, 0.0) : 0.0;
                    }
                    const double R = Rt + Rm;
                    t += E / R;
                    const double x = u2 * R;
                    int touched = -1;   // deme whose rates changed (or, for a rejected migration, the target deme)
                    double dS = 0.0, dI = 0.0;  // change of the touched deme's susceptible / infectious totals
                    bool logged = false;
                    unsigned long long desc = 0;
                    if (Rt > x) {
                        const Pick pk = warp_pick([&](int i) { return s.pr[i]; }, K, x);
                        const int p = pk.i;
                        if (p < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                        double y = pk.rest(x);  // in [0, popRate[p]): what the reference rebuilds as rn * popRate[pi]
                        const double immp = s.imm[p];
                        if (immp > y) {
                            // ---- ImmunityTransition (:550-564)
                            const Pick ps = small_pick([&](int i) { return s.Tc[i] * s.Sx[p * S + i]; }, S, y);
                            if (ps.i < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                            const int ssi = ps.i;
                            const double rn = ps.resid(y);
                            const Pick pt = small_pick([&](int i) { return s.T[ssi * S + i]; }, S, rn * s.Tc[ssi]);
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
                            const double *hprow = s.hp + p * H;
                            const Pick ph = warp_pick([&](int i) { return hprow[i]; }, H, y);
                            const int h = ph.i;
                            if (h < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                            const double z = ph.rest(y);  // in [0, hapPopRate[p,h]) = tEventHapPopRate * I
                            const double Ih = s.I[p * H + h];
                            const double bc = s.b[h] * s.c[p];
                            const double Q = dir_Q<SC>(D, s, p, h);
                            // eventHapPopRate[p,h,0:4] (:310-314) times the cell's count
                            const double e0 = s.b[h] * (Q * s.c[p]) * Ih, e1 = s.d[h] * Ih, e2 = s.sr[h] * s.sm[p] * Ih,
                                         e3 = s.tm[h] * Ih;
                            // the four event rates: z in [0, e0+e1+e2+e3); an event with zero weight owns an empty interval,
                            // so the strict comparisons never pick it; a z that rounding pushed past the total falls to
                            // the last positive weight (fastChoose's catch-all)
                            const double c1 = e0 + e1, c2 = c1 + e2;
                            int e = z < e0 ? 0 : z < c1 ? 1 : z < c2 ? 2 : 3;
                            if (e == 3 && !(e3 > 0.0)) e = e2 > 0.0 ? 2 : e1 > 0.0 ? 1 : 0;
                            Pick pe;
                            pe.i = e;
                            pe.before = e == 0 ? 0.0 : e == 1 ? e0 : e == 2 ? c1 : c2;
                            pe.w = e == 0 ? e0 : e == 1 ? e1 : e == 2 ? e2 : e3;
                            if (!(pe.w > 0.0)) { errbits |= ERR_ZERO_WEIGHT; break; }
                            if (e == 0) {
                                // ---- Birth (:568-605): the group of the newly infected, weights Sx[p,s] sigma[s,h]
                                const double sc = bc * Ih;
                                const Pick pg = small_pick([&](int i) { return s.Sx[p * S + i] * s.sig[i * H + h] * sc; }, S, pe.rest(z));
                                if (pg.i < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                                const int si = pg.i;
                                if (lane == 0) {
                                    s.Sx[p * S + si] -= 1.0;
                                    s.totSus[p] -= 1.0;
                                    s.I[p * H + h] += 1.0;
                                    s.totInf[p] += 1.0;
                                }
                                dS = -1.0;
                                dI = 1.0;
                                cB++;
                                desc = pack_event(EV_BIRTH, h, p, si, 0);
                            } else if (e == 1 || e == 2) {
                                // ---- Death / Sampling (:616-635)
                                const int g = s.g[h];
                                if (lane == 0) {
                                    s.Sx[p * S + g] += 1.0;
                                    s.totSus[p] += 1.0;
                                    s.I[p * H + h] -= 1.0;
                                    s.totInf[p] -= 1.0;
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
                                if (lane == 0) {
                                    s.I[p * H + nh] += 1.0;
                                    s.I[p * H + h] -= 1.0;
                                }
                                cM++;
                                desc = pack_event(EV_MUTATION, h, p, nh, 0);
                            }
                        }
                        logged = true;
                        touched = p;
                    } else {
                        // ---- GenerateMigration (:672-694): rejection-sampled cross-deme infection
                        auto mpw = [&](int i) { return s.maxEBM[i] * s.totSus[i] * (ginf - s.totInf[i]); };
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
                        const double xs = rn * (ginf - s.totInf[tp]);
                        const Pick psrc = warp_pick([&](int i) { return s.totInf[i]; }, K, xs, tp);
                        const int sp = psrc.i;
                        if (sp < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                        rn = psrc.resid(xs);
                        const double xh = rn * s.totInf[sp];
                        const double *Irow = s.I + sp * H;
                        const Pick ph = warp_pick([&](int i) { return Irow[i]; }, H, xh);
                        const int h = ph.i;
                        if (h < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                        rn = ph.resid(xh);
                        const double xg = rn * s.totSus[tp];
                        const Pick pg = small_pick([&](int i) { return s.Sx[tp * S + i]; }, S, xg);
                        const int si = pg.i;
                        if (si < 0) { errbits |= ERR_ZERO_WEIGHT; break; }
                        rn = pg.resid(xg);
                        const double p_accept = eff[sp * K + tp] * s.b[h] * s.sig[si * H + h] / s.maxEBM[tp];
                        touched = tp;  // the reference runs CheckLockdown on the target deme either way (:694)
                        if (rn < p_accept) {
                            if (lane == 0) {
                                s.Sx[tp * S + si] -= 1.0;
                                s.totSus[tp] -= 1.0;
                                s.I[tp * H + h] += 1.0;
                                s.totInf[tp] += 1.0;
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
                        // ---- UpdateRates (:516-546): the touched deme, then the totals by increments
                        __syncwarp();
                        const int p = touched;
                        const double inf = dir_refresh_hp<SC>(D, s, p);
                        const double imm = dir_imm<SC>(D, s, p);
                        const double pr_old = s.pr[p];
                        __syncwarp();
                        if (lane == 0) {
                            s.inf[p] = inf;
                            s.imm[p] = imm;
                            s.pr[p] = inf + imm;
                        }
                        Rt += (inf + imm) - pr_old;
                        if (dI != 0.0) {
                            // totSus and totInf of deme p already hold the new values
                            const double Sn = s.totSus[p], In = s.totInf[p];
                            const double m = s.maxEBM[p];
                            mA += m * dS;
                            mB += m * (Sn * In - (Sn - dS) * (In - dI));
                            ginf += dI;
                            Rm = K > 1 ? fmax(ginf * mA - mB, 0.0) : 0.0;
                        }
                        __syncwarp();
                        if (Rt <= 0.0 || ginf == 0.0) {
                            if (ginf != 0.0) {  // rounding of the increments must not end a live epidemic: recompute
                                dir_totals(D, s, Rt, mA, mB);
                                Rm = K > 1 ? fmax(ginf * mA - mB, 0.0) : 0.0;
                            }
                            if (Rt <= 0.0 || ginf == 0.0) break;
                        }
                    }
                    // ---- CheckLockdown(pi) (:412, :698-710): the lanes agree on the (rare) need for the sequential pass
                    {
                        const double ti = s.totInf[touched];
                        const int lk = s.lock[touched];
                        if ((ti > s.startN[touched] && lk == 0) || (ti < s.endN[touched] && lk == 1)) {
                            int flips = 0;
                            if (lane == 0)
                                flips = check_lockdown(D, pp, touched, (long long)ti, s.cd, s.lock, t, &st.loc_n[r], loc_sp, loc_t,
                                                       st.loc_cap, &st.err[r]);
                            flips = __shfl_sync(0xffffffffu, flips, 0);
                            if (flips) {
                                swaps += flips;
                                __syncwarp();
                                update_contact_rates(WarpGroup(), D, pp, s.cd, eff, s.c, s.maxEBM);
                                dir_refresh_all<SC>(D, s, Rt, mA, mB, ginf);
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
                for (int i = lane; i < K * H; i += 32) s.I[i] = (double)st.initI[(size_t)r * K * H + i];
                for (int i = lane; i < K * S; i += 32) s.Sx[i] = (double)st.initSx[(size_t)r * K * S + i];
                dir_refresh_all<SC>(D, s, Rt, mA, mB, ginf);
                int flips = 0;
                if (lane == 0)
                    for (int p = 0; p < K; p++)
                        flips += check_lockdown(D, pp, p, (long long)s.totInf[p], s.cd, s.lock, t, &st.loc_n[r], loc_sp, loc_t,
                                                st.loc_cap, &st.err[r]);
                flips = __shfl_sync(0xffffffffu, flips, 0);
                if (flips) {
                    swaps += flips;
                    __syncwarp();
                    update_contact_rates(WarpGroup(), D, pp, s.cd, eff, s.c, s.maxEBM);
                    dir_refresh_all<SC>(D, s, Rt, mA, mB, ginf);
                }
                good_attempt = 0;
            } else {
                good_attempt = attempt + 1;
                break;
            }
        }
        flush_log();

        // ---- commit
        __syncwarp();
        for (int i = lane; i < K * H; i += 32) st.I[(size_t)r * K * H + i] = (long long)s.I[i];
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
            // parity tap (UpdateRates, :516-546): the totals as the increments left them -- a fresh recompute from the final
            // state (vgsim_rates) must give the same numbers
            st.rate_tot[2 * (size_t)r] = Rt;
            st.rate_tot[2 * (size_t)r + 1] = K > 1 ? fmax(ginf * mA - mB, 0.0) : 0.0;
        }
        __syncwarp();
    }
}

// Deterministic parity tap: the rate hierarchy of replicate r's current state (UpdateAllRates, :279-351)
__global__ void rates_tap_kernel(const __grid_constant__ DevState st, const __grid_constant__ DirLayout L, int r, double *ev,
                                 double *hp, double *popRate, double *migPop, double *totals) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const Dims &D = st.D;
    const int lane = threadIdx.x & 31, K = D.K, H = D.H;
    DirShared s;
    dir_carve(s, L, smem_raw, 0);
    const double *pp = st.params + (size_t)st.rep_pp[r] * D.blob;
    dir_load_params(D, L, smem_raw + (L.par_shared ? L.o_par : L.o_warp0), pp, lane, 32);
    for (int i = lane; i < K * H; i += 32) s.I[i] = (double)st.I[(size_t)r * K * H + i];
    for (int i = lane; i < K * D.S; i += 32) s.Sx[i] = (double)st.Sx[(size_t)r * K * D.S + i];
    for (int i = lane; i < K; i += 32) {
        s.cd[i] = st.cd[(size_t)r * K + i];
        s.c[i] = st.ceff[(size_t)r * K + i];
        s.maxEBM[i] = st.maxEBM[(size_t)r * K + i];
    }
    __syncwarp();
    double Rt, A, B, ginf;
    dir_refresh_all<0>(D, s, Rt, A, B, ginf);
    __syncwarp();
    for (int i = lane; i < K * H; i += 32) {
        const int p = i / H, h = i - p * H;
        ev[i * 4 + 0] = s.b[h] * (dir_Q<0>(D, s, p, h) * s.c[p]);
        ev[i * 4 + 1] = s.d[h];
        ev[i * 4 + 2] = s.sr[h] * s.sm[p];
        ev[i * 4 + 3] = s.tm[h];
        hp[i] = s.hp[i];
    }
    double y = 0.0;
    for (int p = lane; p < K; p += 32) {
        popRate[p] = s.pr[p];
        const double m = s.maxEBM[p] * s.totSus[p] * (ginf - s.totInf[p]);
        migPop[p] = m;
        y += m;
    }
    y = warp_sum(y);
    if (lane == 0) {
        totals[0] = Rt;
        totals[1] = y;
    }
}

// Does one replicate's rate hierarchy fit one SM's shared memory?  uniform_pp >= 0: with the parameter block shared
// by the CTA (launch_direct when every replicate uses that point); < 0: in the warp's slice (launch_rates_tap too).
bool direct_fits_shared(const Dims &D, int uniform_pp) {
    return dir_layout(D, uniform_pp >= 0, uniform_pp >= 0 ? uniform_pp : 0, 227 * 1024, 16).nwarps >= 1;
}

cudaError_t launch_direct(const DevState &st, const SimArgs &a, cudaStream_t stream, int num_sms, int uniform_pp, int *work) {
    DirLayout L = dir_layout(st.D, uniform_pp >= 0, uniform_pp >= 0 ? uniform_pp : 0, 227 * 1024, 16);
    if (L.nwarps < 1) return cudaErrorInvalidConfiguration;
    const void *kern = st.D.S == 1 ? (const void *)direct_kernel<1> : st.D.S == 2 ? (const void *)direct_kernel<2>
                     : st.D.S == 3 ? (const void *)direct_kernel<3> : st.D.S == 4 ? (const void *)direct_kernel<4>
                                                                                  : (const void *)direct_kernel<0>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total_bytes);
    if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(work, 0, sizeof(int), stream);
    if (e != cudaSuccess) return e;
    int grid = (st.R + L.nwarps - 1) / L.nwarps;
    if (grid > num_sms) grid = num_sms;
    void *args[] = {(void *)&st, (void *)&a, (void *)&L, (void *)&work};
    return cudaLaunchKernel(kern, dim3(grid), dim3(L.nwarps * 32), args, L.total_bytes, stream);
}

cudaError_t launch_rates_tap(const DevState &st, int r, double *ev, double *hp, double *popRate, double *migPop,
                             double *totals, cudaStream_t stream) {
    DirLayout L = dir_layout(st.D, false, 0, 227 * 1024, 1);
    if (L.nwarps < 1) return cudaErrorInvalidConfiguration;
    cudaError_t e = cudaFuncSetAttribute(rates_tap_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total_bytes);
    if (e != cudaSuccess) return e;
    rates_tap_kernel<<<1, 32, L.total_bytes, stream>>>(st, L, r, ev, hp, popRate, migPop, totals);
    return cudaGetLastError();
}

}  // namespace vg
