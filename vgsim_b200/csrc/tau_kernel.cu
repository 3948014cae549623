// Replicate-batched tau-leaping (reference SimulatePopulation_tau, src/_BirthDeath.pyx:2293-2593).
//
// One CTA per replicate (grid-stride over replicates).  Compartment counts, drifts, per-leap deltas
// and the parameter point live in shared memory for the whole run.  The dense event log row of a leap
// (4*P bytes, one int32 count per positional channel, SURVEY App. A.4) is the only steady-state HBM
// traffic, so the kernel is organised around it:
//
//   0. the row is zero-filled with 16-byte coalesced stores as soon as the leap starts (the stores
//      drain while the CTA computes);
//   1. F[t,h] = sum_s eff[t,s] m[s,s] b[h] I[s,h] only for haplotypes present anywhere (colcnt[h] > 0);
//   2. net drifts and tau (ChooseTau, :2432-2450, incl. the float-epsilon quirk);
//   3. Poisson draws only where something can fire.  A compact list of infectious cells (p,h) with I > 0
//      is kept in shared memory; a cell owns LC = E + (K-1)*S channels: RECOVERY, SAMPLING, 3U MUTATION,
//      S TRANSMISSION, and its out-MIGRATION to every other deme x group.  Poisson(0) = 0 consumes no
//      randomness in the reference either (numpy random_poisson), so channels of empty cells are never
//      touched.  Per cell the kernel makes "primary" draws in blocks of 4 sharing one Philox4x32-10 call
//      keyed (seed; cell, leap, retry|epoch, block): RECOVERY, SAMPLING, the TOTAL of the mutation group,
//      the TOTAL of the out-migration group, and each TRANSMISSION channel.  A group total is used when
//      its lambda <= 1: independent Poissons conditioned on their sum are multinomial, so drawing the sum
//      and splitting a non-zero sum over the group's channels has exactly the reference's joint
//      distribution; larger groups are "expanded" and drawn channel by channel.  A draw whose count the
//      top 32 bits of its uniform already prove to be 0 (U < 1 - lambda) ends there; the others are pushed
//      to a shared-memory queue and finished in a second pass with all lanes busy (inversion for
//      lambda < 10 from the bottom of the queue, Hoermann PTRS from the top, so warps do not mix them).
//      Non-zero counts are scattered into the zero-filled row;
//   4. feasibility (:2522-2528, with the source-deme book-keeping quirk Q8); on failure tau is halved
//      and the whole leap redrawn (:2316-2321);
//   5. deltas applied, the infectious-cell list rebuilt, MULTITYPE row appended, CheckLockdown for
//      every deme (:2326-2329).
//
// variant 1 (vgsim_set_tau_variant) expands every group, i.e. draws each channel separately exactly like
// the reference; it is kept as a parity tap.  The same channel code backs the deterministic propensity
// tap (propensity_kernel).
#include "common.cuh"
#include "rates.cuh"
#include "samplers.cuh"

namespace vg {

extern __shared__ __align__(16) unsigned char smem_raw[];

// ---- teams ------------------------------------------------------------------------------------------
// A CTA is blockDim.y TEAMS of blockDim.x = 256 threads; every team simulates its own replicate with its own
// slice of the dynamic shared memory and its own named barrier, so threadIdx.x / blockDim.x are team-local and
// the per-replicate control flow stays independent.  All teams of the SM re-align at the top of every leap
// (align_teams): they then walk the same code at the same time, so an instruction line fetched from L2 by one
// team is found in the SM's instruction cache by the others.  The leap loop is far larger than the 32 KB L1.5
// instruction cache, and with independent CTAs the kernel was bound by instruction fetch (ncu: icc hit rate
// 59 %, gcc instruction requests 84 % of peak, every phase costing ~300 cycles per 128-byte code line).
#define TAU_TEAM 256
#define TAU_ZB 16384      // zero buffer (bytes) at the start of the CTA tail: source of the bulk row wipes
#define TAU_CTA_TAIL (TAU_ZB + 16)  // bytes after the team slices: zero buffer, then [0] = number of finished teams

__device__ __forceinline__ unsigned dyn_smem_bytes() {
    unsigned v;
    asm("mov.u32 %0, %%dynamic_smem_size;" : "=r"(v));
    return v;
}
__device__ __forceinline__ unsigned team_stride() { return (dyn_smem_bytes() - TAU_CTA_TAIL) / blockDim.y; }
__device__ __forceinline__ unsigned char *team_base() { return smem_raw + threadIdx.y * team_stride(); }
__device__ __forceinline__ unsigned char *zero_buf() { return smem_raw + (dyn_smem_bytes() - TAU_CTA_TAIL); }
__device__ __forceinline__ int *cta_tail() { return reinterpret_cast<int *>(smem_raw + (dyn_smem_bytes() - 16)); }
__device__ __forceinline__ void team_sync() { asm volatile("bar.sync %0, %1;" ::"r"(2 + (int)threadIdx.y), "r"(TAU_TEAM) : "memory"); }
__device__ __forceinline__ int team_or(int pred) {
    int r;
    asm volatile(
        "{\n\t.reg .pred p, q;\n\tsetp.ne.s32 q, %1, 0;\n\tbar.red.or.pred p, %2, %3, q;\n\tselp.s32 %0, 1, 0, p;\n\t}"
        : "=r"(r)
        : "r"(pred), "r"(2 + (int)threadIdx.y), "r"(TAU_TEAM)
        : "memory");
    return r;
}
// barrier 1: every thread of the CTA (running teams at the top of a leap, finished teams in their idle loop)
__device__ __forceinline__ void align_teams() {
    asm volatile("bar.sync 1, %0;" ::"r"((int)(blockDim.x * blockDim.y)) : "memory");
}
struct TeamGroup {
    __device__ __forceinline__ int tid() const { return threadIdx.x; }
    __device__ __forceinline__ int size() const { return blockDim.x; }
    __device__ __forceinline__ void sync() const { team_sync(); }
};

// A shared-memory array addressed by a 32-bit byte offset from the dynamic shared-memory base: keeps the
// ~30 array handles of TauShared in one register each and lets the compiler emit LDS/STS/ATOMS directly.
template <class T>
struct SArr {
    int off;
    __device__ __forceinline__ T *ptr() const { return reinterpret_cast<T *>(team_base() + off); }
    __device__ __forceinline__ T &operator[](int i) const { return ptr()[i]; }
    __device__ __forceinline__ operator T *() const { return ptr(); }
};

struct TauShared {
    static constexpr bool has_qin = false;
    // fp64 parameters
    SArr<double> b, d, sr, q, tmq, sigT, sb, T, sm, cd, c, mdiag, sizeD, maxEBM, startN, endN, effS;
    bool has_effS;
    // fp64 state (counts are exact in fp64; kept as doubles so the rate arithmetic needs no conversions)
    SArr<double> I, Sx;       // infectious [K][H], susceptible [K][S]
    SArr<double> dI, dS, Qm;  // drifts; Q[p,h] = sum_s Sx[p,s] sigma[s,h]
    SArr<double> Mg;          // Mg[p,s] = sum_{t != p} eff[t,p] Sx[t,s]: what deme p's emigrants meet abroad, by group (mig_total)
    SArr<double> Bp, Rp;      // per (deme, group): infection pressure sum_h sigma b I, and return flow into the group
    SArr<double> red;
    SArr<unsigned long long> nbrmask;  // [H] (H <= 64) haplotypes one substitution away from h
    SArr<unsigned long long> rowmask;  // [K] (H <= 64) haplotypes present in deme p
    // int32
    SArr<int> chkI, updI, dSx, g, lock;
    SArr<int> tot;        // per-deme infectious totals (built by the apply pass)
    SArr<int> colcnt;     // #demes holding haplotype h
    SArr<int> colmask;    // (K <= 32) bit p set when deme p holds haplotype h
    SArr<int> act;        // cells with I > 0 in ascending cell order (so every sum over it has a fixed order)
    SArr<int> dstart;     // [K+1] first entry of deme p in act
    SArr<int> segcnt;     // infectious cells per 32-cell segment (ordered compaction)
    SArr<int> qhi, qoc;   // slow-path queue: primary Philox word; owner id | draw code << 20
    SArr<int> xq;         // expansion queues: [0,256) cells whose mutation group, [256,512) whose migration group
                          // is drawn channel by channel
    SArr<int> flags;      // [0..5]=per-leap tallies by event type (EV_*) [6]=flip flag [7]=overflow [8]=nAct
                          // [10]=flips total [12+4*parity .. +3]=queue counters of the live draw round
    SArr<long long> tally64;  // [0..5] events by type since the kernel (or the last Restart) began
    int nseg;             // number of 32-cell segments
    int qcap;             // slow-path queue capacity
    bool store_drift;     // the propensity tap keeps dI/dS; the simulation kernel only needs tau
    bool use_masks;       // H <= 64 and K <= 32: presence bit masks drive the sparse drift sums
    int bytes;
};

__host__ __device__ inline bool tau_eff_in_smem(const Dims &D) { return D.K <= 32; }

__host__ __device__ inline TauShared tau_layout(const Dims &D, bool store_drift, int nt = 256) {
    TauShared s;
    s.store_drift = store_drift;
    s.qcap = 4 * nt;  // slow-path queue entries per round: at most 4 pushes per thread
    int o = 0;
    auto dbl = [&](SArr<double> &a, int n) { a.off = o; o += n * 8; };
    auto u64 = [&](SArr<unsigned long long> &a, int n) { a.off = o; o += n * 8; };
    auto i32 = [&](SArr<int> &a, int n) { a.off = o; o += n * 4; };
    auto i64 = [&](SArr<long long> &a, int n) { o = (o + 7) & ~7; a.off = o; o += n * 8; };
    const int KH = D.K * D.H, KS = D.K * D.S;
    s.use_masks = D.H <= 64 && D.K <= 32;
    s.nseg = (KH + 31) / 32;
    dbl(s.b, D.H); dbl(s.d, D.H); dbl(s.sr, D.H); dbl(s.tmq, D.H);
    dbl(s.q, D.H * D.U * 3);
    dbl(s.sigT, D.S * D.H); dbl(s.sb, D.S * D.H);
    dbl(s.T, D.S * D.S);
    dbl(s.sm, D.K); dbl(s.cd, D.K); dbl(s.c, D.K); dbl(s.mdiag, D.K); dbl(s.sizeD, D.K); dbl(s.maxEBM, D.K);
    dbl(s.startN, D.K); dbl(s.endN, D.K);
    s.has_effS = tau_eff_in_smem(D);
    s.effS.off = o;
    if (s.has_effS) o += D.K * D.K * 8;
    dbl(s.I, KH); dbl(s.Sx, KS);
    dbl(s.dI, store_drift ? KH : 0); dbl(s.dS, store_drift ? KS : 0); dbl(s.Qm, KH);
    dbl(s.Bp, KS); dbl(s.Rp, KS); dbl(s.Mg, KS);
    dbl(s.red, 64);
    u64(s.nbrmask, s.use_masks ? D.H : 0); u64(s.rowmask, s.use_masks ? D.K : 0);
    i32(s.chkI, KH); i32(s.updI, KH); i32(s.act, KH);
    i32(s.dSx, KS);
    i32(s.g, D.H); i32(s.colcnt, D.H); i32(s.colmask, D.H);
    i32(s.lock, D.K); i32(s.tot, D.K); i32(s.dstart, D.K + 1);
    i32(s.segcnt, s.nseg + 1);
    i32(s.qhi, s.qcap); i32(s.qoc, s.qcap); i32(s.xq, 2 * nt);
    i32(s.flags, 24);
    i64(s.tally64, 8);
    s.bytes = o;
    return s;
}

// One reaction channel: propensity (per unit time) plus where its count goes.
struct Channel {
    int type;        // EV_* ; EV_MULTITYPE = padding (c >= P)
    int i_dec;       // I cell that loses n   (-1 none)
    int i_inc;       // I cell that gains n   (-1 none)
    int i_chk;       // I cell the feasibility check books the gain on (quirk Q8: source deme for migration)
    int s_dec;       // Sx cell that loses n  (-1 none)
    int s_inc;       // Sx cell that gains n  (-1 none)
    double prop;
};

// Channel l of infectious cell (p,h): l < E are the deme-block events RECOVERY, SAMPLING, MUTATION[u][k],
// TRANSMISSION[s]; l >= E is out-migration of h from p to the (l-E)/S-th other deme, group (l-E)%S.
// Returns the positional index c of the channel in the dense row.
template <class SH>
__device__ __forceinline__ int cell_channel(int p, int h, int l, const Dims &D, const SH &s, const double *eff,
                                            Channel &ch) {
    const int K = D.K, H = D.H, S = D.S;
    const int cell = p * H + h;
    const double Ii = s.I[cell];
    ch.i_dec = ch.i_inc = ch.i_chk = ch.s_dec = ch.s_inc = -1;
    ch.prop = 0.0;
    if (l < D.E) {
        if (l == 0) {  // RECOVERY (:2386)
            ch.type = EV_DEATH;
            ch.i_dec = cell;
            ch.s_inc = p * S + s.g[h];
            ch.prop = s.d[h] * Ii;
        } else if (l == 1) {  // SAMPLING (:2392)
            ch.type = EV_SAMPLING;
            ch.i_dec = cell;
            ch.s_inc = p * S + s.g[h];
            ch.prop = s.sr[h] * Ii * s.sm[p];
        } else if (l < 2 + 3 * D.U) {  // MUTATION (:2400-2401)
            int uk = l - 2, u = uk / 3, k = uk - u * 3;
            ch.type = EV_MUTATION;
            ch.i_dec = cell;
            ch.i_inc = ch.i_chk = p * H + mutate_hap(h, u, k, D.U);
            ch.prop = s.q[h * D.U * 3 + uk] * Ii;
        } else {  // TRANSMISSION (:2410-2414)
            int sn = l - 2 - 3 * D.U;
            ch.type = EV_BIRTH;
            ch.i_inc = ch.i_chk = cell;
            ch.s_dec = p * S + sn;
            if (Ii != 0.0) ch.prop = s.b[h] * s.sigT[sn * H + h] * s.c[p] * s.Sx[p * S + sn] * Ii;
        }
        return D.NA + p * D.PD + D.SS1 + h * D.E + l;
    }
    // MIGRATION  [sp][tp != sp][s][h]  (:2366-2367)
    int mm = l - D.E;
    int tpp = mm / S, sn = mm - tpp * S;
    int tp = tpp + (tpp >= p ? 1 : 0);
    ch.type = EV_MIGRATION;
    ch.i_inc = tp * H + h;
    ch.i_chk = cell;
    ch.s_dec = tp * S + sn;
    if (Ii != 0.0) ch.prop = eff[tp * K + p] * s.Sx[tp * S + sn] * Ii * s.b[h] * s.sigT[sn * H + h] * s.mdiag[p];
    return ((p * (K - 1) + tpp) * S + sn) * H + h;
}

// SUSCCHANGE channel l of deme p: [ss][ts != ss]  (:2378)
template <class SH>
__device__ __forceinline__ int susc_channel(int p, int l, const Dims &D, const SH &s, Channel &ch) {
    const int S = D.S;
    int ss = l / (S - 1), tsp = l - ss * (S - 1);
    int ts = tsp + (tsp >= ss ? 1 : 0);
    ch.i_dec = ch.i_inc = ch.i_chk = -1;
    ch.type = EV_SUSCCHANGE;
    ch.s_dec = p * S + ss;
    ch.s_inc = p * S + ts;
    ch.prop = s.T[ss * S + ts] * s.Sx[p * S + ss];
    return D.NA + p * D.PD + l;
}

// Positional index c -> channel, and its Philox address (owner id, local index).
__device__ __forceinline__ void decode_channel(int c, const Dims &D, const TauShared &s, const double *eff, Channel &ch,
                                               int &owner, int &l) {
    const int K = D.K, H = D.H, S = D.S;
    if (c >= D.P) {
        ch.i_dec = ch.i_inc = ch.i_chk = ch.s_dec = ch.s_inc = -1;
        ch.prop = 0.0;
        ch.type = EV_MULTITYPE;
        owner = l = 0;
        return;
    }
    if (c < D.NA) {
        int row = c >> D.hshift, h = c & (H - 1);
        int pair = row / S, sn = row - pair * S;
        int sp = pair / (K - 1), tpp = pair - sp * (K - 1);
        owner = sp * H + h;
        l = D.E + tpp * S + sn;
        cell_channel(sp, h, l, D, s, eff, ch);
        return;
    }
    int c2 = c - D.NA;
    int p = c2 / D.PD, r = c2 - p * D.PD;
    if (r < D.SS1) {
        owner = K * H + p;
        l = r;
        susc_channel(p, r, D, s, ch);
        return;
    }
    int r2 = r - D.SS1;
    int h = r2 / D.E;
    l = r2 - h * D.E;
    owner = p * H + h;
    cell_channel(p, h, l, D, s, eff, ch);
}

// fixed-slot minimum over the CTA with ONE barrier: `slot` alternates between calls so that the previous call's
// values are never overwritten while a slower warp still reads them
__device__ __forceinline__ double block_min(double v, double *red, int slot) {
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    const int w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    double *r = red + 32 * (slot & 1);
    if ((threadIdx.x & 31) == 0) r[w] = v;
    align_teams();  // generation barrier 4 of 5 (see tau_kernel)
    v = r[0];
    for (int i = 1; i < nw; i++) v = fmin(v, r[i]);
    return v;
}

__device__ __forceinline__ int warp_sum_i(int v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- ordered compaction of the infectious cells ------------------------------------------------------
// Pass 1 (count_cells): one ballot per 32-cell segment -> segcnt[]; also clears the presence tables.
// Pass 2 (write_lists, after a barrier): every segment's base is the sum of the counts before it, so the
// list comes out in ascending cell order regardless of warp scheduling; deme p's cells are the range
// [dstart[p], dstart[p+1]).  colcnt / colmask / rowmask record where each haplotype is present.
__device__ __forceinline__ void count_cells(const Dims &D, const TauShared &s) {
    const int tid = threadIdx.x, nt = blockDim.x, KH = D.K * D.H;
    for (int base = 0; base < KH; base += nt) {
        const int i = base + tid;
        const bool on = i < KH && s.I[i] != 0.0;
        const unsigned m = __ballot_sync(0xffffffffu, on);
        if ((tid & 31) == 0 && base + tid < KH) s.segcnt[i >> 5] = __popc(m);
    }
    for (int i = tid; i < D.H; i += nt) {
        s.colcnt[i] = 0;
        s.colmask[i] = 0;
    }
    if (s.use_masks)
        for (int i = tid; i < D.K; i += nt) s.rowmask[i] = 0ull;
}

// number of infectious cells = sum of segcnt (every thread gets the value; warp-parallel, no barrier)
__device__ __forceinline__ int total_cells(const TauShared &s) {
    int acc = 0;
    for (int k = threadIdx.x & 31; k < s.nseg; k += 32) acc += s.segcnt[k];
    return warp_sum_i(acc);
}

__device__ __forceinline__ void write_lists(const Dims &D, const TauShared &s) {
    const int tid = threadIdx.x, nt = blockDim.x, KH = D.K * D.H, lane = tid & 31;
    for (int base = 0; base < KH; base += nt) {
        const int i = base + tid;
        const int seg = (base + (tid & ~31)) >> 5;  // this warp's segment in this sweep
        int before = 0;
        for (int k = lane; k < seg && k < s.nseg; k += 32) before += s.segcnt[k];
        before = warp_sum_i(before);
        const bool on = i < KH && s.I[i] != 0.0;
        const unsigned m = __ballot_sync(0xffffffffu, on);
        const int pos = before + __popc(m & ((1u << lane) - 1u));
        if (i < KH) {
            const int p = i >> D.hshift, h = i & (D.H - 1);
            if (h == 0) s.dstart[p] = pos;
            if (on) {
                s.act[pos] = i;
                atomicAdd(&s.colcnt[h], 1);
                if (s.use_masks) {
                    atomicOr(&s.colmask[h], 1 << p);
                    atomicOr(&s.rowmask[p], 1ull << h);
                }
            }
            if (i == KH - 1) {
                s.dstart[D.K] = pos + (on ? 1 : 0);
                s.flags[8] = pos + (on ? 1 : 0);
            }
        }
    }
}

// full rebuild from s.I (load, Restart): leaves tot[] too
__device__ void rebuild_lists(const Dims &D, const TauShared &s) {
    const int tid = threadIdx.x, nt = blockDim.x;
    team_sync();
    for (int i = tid; i < D.K; i += nt) s.tot[i] = 0;
    count_cells(D, s);
    team_sync();
    for (int i = tid; i < D.K * D.H; i += nt) {
        const double v = s.I[i];
        if (v != 0.0) atomicAdd(&s.tot[i >> D.hshift], (int)v);
    }
    write_lists(D, s);
    team_sync();
}

// Q[p,h] = sum_s Sx[p,s] sigma[s,h] for every cell (needs only Sx; runs before the list barrier)
__device__ __forceinline__ void q_pass(const Dims &D, const TauShared &s) {
    const int H = D.H, S = D.S;
    for (int i = threadIdx.x; i < D.K * H; i += blockDim.x) {
        const int p = i >> D.hshift, h = i & (H - 1);
        double Q = 0.0;
        for (int sn = 0; sn < S; sn++) Q += s.Sx[p * S + sn] * s.sigT[sn * H + h];
        s.Qm[i] = Q;
    }
}

// Mg[p,s] = sum_{t != p} eff[t,p] Sx[t,s] (needs only Sx; runs beside q_pass).  Same loop order in the warp kernel.
template <class DIMS, class SH>
__device__ __forceinline__ void mig_pressure(int i, const DIMS &D, const SH &s, const double *eff) {
    const int K = D.K, S = D.S;
    const int p = i / S, sn = i - p * S;
    double acc = 0.0;
#pragma unroll 1
    for (int tp = 0; tp < K; tp++)
        if (tp != p) acc += eff[tp * K + p] * s.Sx[tp * S + sn];
    s.Mg[i] = acc;
}

// Net drift of infectious cell i = (p,h): force of infection (own deme + migration from every deme holding h),
// removal, and mutation inflow from the haplotypes one substitution away that are present in the deme
// (Propensities :2351-2417 summed per compartment).  Every sum runs in ascending index order.
template <class DIMS, class SH>
__device__ __forceinline__ double drift_I_cell(int i, const DIMS &D, const SH &s, const double *eff) {
    const int K = D.K, H = D.H, U = D.U;
        const int p = i >> D.hshift, h = i & (H - 1);
        const double Iv = s.I[i];
        double v = 0.0;
        if (s.colcnt[h] != 0) {
            // force of infection on (p,h): own deme + migration from every deme holding h  (:2366-2367, :2410-2414)
            double F = 0.0;
            if (s.use_masks) {
                unsigned cm = (unsigned)s.colmask[h] & ~(1u << p);
                while (cm) {
                    const int sp = __ffs(cm) - 1;
                    cm &= cm - 1;
                    F += eff[p * K + sp] * s.mdiag[sp] * (s.b[h] * s.I[sp * H + h]);
                }
            } else {
                for (int sp = 0; sp < K; sp++) {
                    const double Is = s.I[sp * H + h];
                    if (sp != p && Is != 0.0) F += eff[p * K + sp] * s.mdiag[sp] * (s.b[h] * Is);
                }
            }
            const double Q = s.Qm[i];
            v = Q * F + s.c[p] * s.b[h] * Iv * Q - (s.d[h] + s.sr[h] * s.sm[p] + s.tmq[h]) * Iv;
        }
        // mutation inflow from the haplotypes one substitution away that are present in this deme (:2400-2401)
        if constexpr (SH::has_qin) {
            if (s.use_masks) {  // same terms in the same order, rates read from the inflow table qin[h][neighbour slot]
                const unsigned long long nb = s.nbrmask[h];
                unsigned long long nm = s.rowmask[p] & nb;
                const int n3 = 3 * U;
                while (nm) {
                    const int src = __ffsll((long long)nm) - 1;
                    nm &= nm - 1;
                    const int slot = __popcll(nb & ((1ull << src) - 1ull));
                    v += s.qin[h * n3 + slot] * s.I[p * H + src];
                }
                return v;
            }
        }
        if (s.use_masks) {
            unsigned long long nm = s.rowmask[p] & s.nbrmask[h];
            while (nm) {
                const int src = __ffsll((long long)nm) - 1;
                nm &= nm - 1;
                const int x = src ^ h;
                const int sh = (31 - __clz(x)) & ~1;
                const int u = U - 1 - (sh >> 1);
                const int as = (src >> sh) & 3, hu = (h >> sh) & 3;
                const int k = hu - (hu > as ? 1 : 0);
                v += s.q[(src * U + u) * 3 + k] * s.I[p * H + src];
            }
        } else {
            for (int u = 0; u < U; u++) {
                const int sh = 2 * (U - u - 1);
                const int hu = (h >> sh) & 3;
                for (int a = 0; a < 4; a++) {
                    if (a == hu) continue;
                    const int src = h + ((a - hu) << sh);
                    const double Is = s.I[p * H + src];
                    if (Is != 0.0) v += s.q[(src * U + u) * 3 + (hu - (hu > a ? 1 : 0))] * Is;
                }
            }
        }
        return v;
}

// Net drift of susceptible compartment i = (p, sn)
template <class DIMS, class SH>
__device__ __forceinline__ double drift_S_cell(int i, const DIMS &D, const SH &s, const double *eff) {
    const int K = D.K, S = D.S;
        const int p = i / S, sn = i - p * S;
        double phi = s.c[p] * s.Bp[i];
        for (int sp = 0; sp < K; sp++)
            if (sp != p) phi += eff[p * K + sp] * s.mdiag[sp] * s.Bp[sp * S + sn];
        const double Sv = s.Sx[i];
        double v = -Sv * phi + s.Rp[i];
        for (int s2 = 0; s2 < S; s2++)
            if (s2 != sn) v += s.T[s2 * S + sn] * s.Sx[p * S + s2] - s.T[sn * S + s2] * Sv;
        return v;
}

// Drifts and tau of the current shared-memory state (Propensities :2351-2417 summed per compartment, ChooseTau
// :2432-2450).  Needs the lists and Qm; contains two barriers; returns tau (uniform).  Every sum runs over the
// ordered cell list / set bits in ascending order, so the result does not depend on warp scheduling.
__device__ double drifts_and_tau(const Dims &D, const TauShared &s, const double *eff, int slot) {
    const int K = D.K, H = D.H, S = D.S, U = D.U;
    const int tid = threadIdx.x, nt = blockDim.x;
    // ---- A. per (deme, group): pressure B = sum_h sigma[s,h] b[h] I[p,h], return flow R = sum_{g[h]=s} (d + sr sm) I.
    //         8 lanes share one (deme, group) sum (strided over the deme's cells) and combine in a fixed butterfly.
    for (int t0 = 0; t0 < K * S; t0 += nt >> 3) {
        const int task = t0 + (tid >> 3), j = tid & 7;
        double Bv = 0.0, Rv = 0.0;
        int p = 0, sn = 0;
        if (task < K * S) {
            p = task / S;
            sn = task - p * S;
            const int a1 = s.dstart[p + 1];
            for (int a = s.dstart[p] + j; a < a1; a += 8) {
                const int cell = s.act[a], h = cell & (H - 1);
                const double Iv = s.I[cell];
                Bv += s.sb[sn * H + h] * Iv;
                if (s.g[h] == sn) Rv += (s.d[h] + s.sr[h] * s.sm[p]) * Iv;
            }
        }
        for (int o = 4; o > 0; o >>= 1) {
            Bv += __shfl_xor_sync(0xffffffffu, Bv, o);
            Rv += __shfl_xor_sync(0xffffffffu, Rv, o);
        }
        if (task < K * S && j == 0) {
            s.Bp[task] = Bv;
            s.Rp[task] = Rv;
        }
    }
    align_teams();  // generation barrier 3 of 5
    double tmin = 1.0;
    const float eps = 0.03f;
    // ---- B1. infectious drifts, one thread per cell
    for (int i = tid; i < K * H; i += nt) {
        const double Iv = s.I[i];
        const double v = drift_I_cell(i, D, s, eff);
        if (s.store_drift) s.dI[i] = v;
        const double av = fabs(v);
        if (av >= 1e-8) {
            double x = (double)(eps * (float)Iv) / 2.0;  // float product, like the reference's generated C
            x = 1.0 > x ? 1.0 : x;
            if (x < tmin * av) tmin = fmin(tmin, x / av);  // divide only when the candidate can lower the minimum
        }
    }
    // ---- B2. susceptible drifts, one thread per (deme, group), taken from the END of the CTA (those threads
    //          own one cell fewer in B1)
    for (int i = nt - 1 - tid; i < K * S; i += nt) {
        const double Sv = s.Sx[i];
        const double v = drift_S_cell(i, D, s, eff);
        if (s.store_drift) s.dS[i] = v;
        const double av = fabs(v);
        if (av >= 1e-8) {
            double x = (double)(eps * (float)Sv) / 2.0;
            x = 1.0 > x ? 1.0 : x;
            if (x < tmin * av) tmin = fmin(tmin, x / av);
        }
    }
    return block_min(tmin, s.red, slot);
}

// Load the parameter point and replicate state into shared memory and build the lists.
__device__ void load_replicate(const DevState &st, int r, const Dims &D, const TauShared &s, const double *pp,
                               const double *eff_g) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const int K = D.K, H = D.H, S = D.S, U = D.U;
    for (int i = tid; i < H; i += nt) {
        s.b[i] = pp[D.o_b + i];
        s.d[i] = pp[D.o_d + i];
        s.sr[i] = pp[D.o_sr + i];
        s.tmq[i] = pp[D.o_tmq + i];
        s.g[i] = (int)pp[D.o_g + i];
        if (s.use_masks) {
            unsigned long long m = 0ull;
            for (int u = 0; u < U; u++)
                for (int a = 1; a < 4; a++) m |= 1ull << (i ^ (a << (2 * u)));
            s.nbrmask[i] = m;
        }
    }
    for (int i = tid; i < H * U * 3; i += nt) s.q[i] = pp[D.o_q + i];
    for (int i = tid; i < S * H; i += nt) {
        s.sigT[i] = pp[D.o_sigT + i];
        s.sb[i] = pp[D.o_sigT + i] * pp[D.o_b + (i % H)];
    }
    for (int i = tid; i < S * S; i += nt) s.T[i] = pp[D.o_T + i];
    for (int i = tid; i < K; i += nt) {
        s.sm[i] = pp[D.o_sm + i];
        s.mdiag[i] = pp[D.o_m + i * K + i];
        s.sizeD[i] = pp[D.o_size + i];
        s.startN[i] = pp[D.o_startN + i];
        s.endN[i] = pp[D.o_endN + i];
        s.cd[i] = st.cd[(size_t)r * K + i];
        s.c[i] = st.ceff[(size_t)r * K + i];
        s.maxEBM[i] = st.maxEBM[(size_t)r * K + i];
        s.lock[i] = st.lock[(size_t)r * K + i];
    }
    if (s.has_effS)
        for (int i = tid; i < K * K; i += nt) s.effS[i] = eff_g[i];
    int ovf = 0;
    for (int i = tid; i < K * H; i += nt) {
        long long v = st.I[(size_t)r * K * H + i];
        if (v > 2147483647LL || v < 0) ovf = 1;
        s.I[i] = (double)v;
    }
    for (int i = tid; i < K * S; i += nt) {
        long long v = st.Sx[(size_t)r * K * S + i];
        if (v > 2147483647LL || v < 0) ovf = 1;
        s.Sx[i] = (double)v;
    }
    if (tid < 24) s.flags[tid] = 0;
    if (tid < 6) s.tally64[tid] = 0;
    team_sync();
    if (ovf) atomicOr(&s.flags[7], 1);
    rebuild_lists(D, s);
}

// CheckLockdown for every deme (:2328-2329 / :449-450 / :736-737).  All threads vote whether any deme
// crosses a threshold; only then thread 0 runs the sequential reference pass and the CTA refreshes the
// contact-density dependent rates.  Ends with a barrier only when something flipped.
__device__ __forceinline__ void lockdown_pass(const DevState &st, int r, const Dims &D, const TauShared &s,
                                              const double *pp, double *eff_g, double now, const int *tot) {
    int pred = 0;
    for (int p = threadIdx.x; p < D.K; p += blockDim.x) {
        double ti = (double)tot[p];
        if ((ti > s.startN[p] && s.lock[p] == 0) || (ti < s.endN[p] && s.lock[p] == 1)) pred = 1;
    }
    if (!team_or(pred)) return;
    if (threadIdx.x == 0) {
        int flips = 0;
        for (int p = 0; p < D.K; p++)
            flips += check_lockdown(D, pp, p, (long long)tot[p], s.cd, s.lock, now, &st.loc_n[r],
                                    st.loc_sp + (size_t)r * st.loc_cap, st.loc_t + (size_t)r * st.loc_cap, st.loc_cap,
                                    &st.err[r]);
        s.flags[6] = flips;
        s.flags[10] += flips;
    }
    team_sync();
    if (s.flags[6]) {
        update_contact_rates(TeamGroup(), D, pp, s.cd, eff_g, s.c, s.maxEBM);
        if (s.has_effS) {
            for (int i = threadIdx.x; i < D.K * D.K; i += blockDim.x) s.effS[i] = eff_g[i];
            team_sync();
        }
    }
}

// Phase timing tap (variant bit 1): thread 0 of every CTA accumulates the cycles between consecutive barrier exits
// of the leap loop, i.e. the critical path of each phase, into this buffer (read by vgsim_debug_tau_phases).
__device__ unsigned long long g_tau_phase_cycles[16];
__device__ unsigned long long g_tau_cta_end[1024];  // timing tap: [2b] when CTA b's first warp ran out of work, [2b+1] its last (global timer, ns)
#define TAU_MARK(k)                                   \
    if (prof && tid == 0) {                           \
        const long long now_ = clock64();             \
        pc[k] += (unsigned long long)(now_ - tmark);  \
        tmark = now_;                                 \
    }

struct LeapTally {
    int B, Dd, Sm, M, I, G;
};

// book n events of channel ch into the shared-memory deltas and the per-thread tallies
template <class SH>
__device__ __forceinline__ void book(const Channel &ch, int n, const SH &s, LeapTally &t) {
    if (ch.i_dec >= 0) {
        atomicSub(&s.chkI[ch.i_dec], n);
        atomicSub(&s.updI[ch.i_dec], n);
    }
    if (ch.i_inc >= 0) {
        atomicAdd(&s.updI[ch.i_inc], n);
        atomicAdd(&s.chkI[ch.i_chk], n);
    }
    if (ch.s_dec >= 0) atomicSub(&s.dSx[ch.s_dec], n);
    if (ch.s_inc >= 0) atomicAdd(&s.dSx[ch.s_inc], n);
    if (ch.type == EV_MIGRATION) t.G += n;
    else if (ch.type == EV_BIRTH) t.B += n;
    else if (ch.type == EV_DEATH) t.Dd += n;
    else if (ch.type == EV_SAMPLING) t.Sm += n;
    else if (ch.type == EV_MUTATION) t.M += n;
    else t.I += n;
}

// Zero-fill of a dense log row by the TMA engine: thread 0 of the team issues shared->global bulk copies out
// of the CTA's zero buffer (no LSU store instructions, no registers, the SM keeps computing); the writes are
// complete once wipe_wait() returns, which the team calls before the first count is scattered into the row.
__device__ __forceinline__ void wipe_row_async(int *row, int bytes) {
    const unsigned src = (unsigned)__cvta_generic_to_shared(zero_buf());
    unsigned long long dst = (unsigned long long)(uintptr_t)row;
    asm volatile("fence.proxy.async;" ::: "memory");  // earlier generic-proxy stores to this row (a failed draw) stay before the wipe
    for (int off = 0; off < bytes; off += TAU_ZB) {
        const int n = bytes - off < TAU_ZB ? bytes - off : TAU_ZB;
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst + off), "r"(src), "r"(n) : "memory");
    }
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void wipe_wait() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// clear everything a (re)draw of the leap accumulates into: the dense row, the deltas, the type tallies
__device__ __forceinline__ void wipe_leap(const Dims &D, const TauShared &s, int *row) {
    const int tid = threadIdx.x, nt = blockDim.x;
    if (tid == 0) wipe_row_async(row, D.Pp * 4);
    for (int i = tid; i < D.K * D.H; i += nt) {
        s.chkI[i] = 0;
        s.updI[i] = 0;
    }
    for (int i = tid; i < D.K * D.S; i += nt) s.dSx[i] = 0;
    if (tid < 6) s.flags[tid] = 0;
}

// the apply pass re-accumulates the per-deme totals: clear them at the top of the leap (CheckLockdown of the
// previous leap has consumed them by then)
__device__ __forceinline__ void zero_totals(const Dims &D, const TauShared &s) {
    for (int i = threadIdx.x; i < D.K; i += blockDim.x) s.tot[i] = 0;
}

// Geometry of the draws one owner makes in a leap, and of its Philox domains (word 3 of the counter).
// An owner is an infectious cell (p,h) (id p*H+h) or deme p's SUSCCHANGE block (id K*H+p).
//   primary block 0 of a cell : {RECOVERY, SAMPLING, total MUTATION, total out-MIGRATION}
//   primary blocks 1..        : TRANSMISSION to group s, 4 per block
//   primary blocks of a deme  : its S(S-1) SUSCCHANGE channels, 4 per block
//   then the per-channel blocks of an EXPANDED mutation group, of an EXPANDED migration group, and the
//   domains that feed the multinomial split of an aggregated total.
struct DrawGeom {
    int NB1;   // primary blocks per cell
    int G2;    // primary blocks per deme (SUSCCHANGE)
    int NBP;   // max(NB1, G2): first expanded-mutation domain
    int nbm;   // blocks of an expanded mutation group  (3U channels)
    int nbg;   // blocks of an expanded migration group ((K-1)S channels)
    int GS;    // domains per owner = stride between Philox "kinds"
    int LC;    // channels owned by a cell
};

template <class DIMS>
__device__ __forceinline__ DrawGeom draw_geom(const DIMS &D) {
    DrawGeom g;
    g.LC = D.E + (D.K - 1) * D.S;
    g.NB1 = 1 + ((D.S + 3) >> 2);
    g.G2 = (D.SS1 + 3) >> 2;
    g.NBP = g.NB1 > g.G2 ? g.NB1 : g.G2;
    g.nbm = (3 * D.U + 3) >> 2;
    g.nbg = ((D.K - 1) * D.S + 3) >> 2;
    g.GS = g.NBP + g.nbm + g.nbg + 2;
    return g;
}

// a mutation / out-migration group is drawn as ONE Poisson total when lam_total <= theta (exact for any theta < 10).
// The total wins when it is almost surely 0 (one early-out instead of 9 / 27 channel draws); a non-zero total costs a
// serial multinomial split in one lane while the warp waits.  Measured at T3: theta 8 / 3 / 1 / 0.3 / 0.15 / 0.1 / 0.03
// -> 8.60 / 7.19 / 6.38 / 6.17 / 6.16 / 6.19 / 6.43 ms per 131,072 leaps.
// Separate thresholds for the two kinds of groups (3U mutation channels / (K-1)S out-migration channels); both < 10.
#define TAU_THETA_MUT 0.25
#define TAU_THETA_MIG 0.5  // with the two-stage split of a non-zero total (S + K - 1 terms per event) the (K-1)S out-migration
                           // channels are worth aggregating up to lambda = 0.5: t = 90 12.3 -> 11.8 ms, t = 60 / 120 unchanged
static_assert(TAU_THETA_MUT < 10.0 && TAU_THETA_MIG < 10.0, "aggregated totals are drawn by inversion (lambda < 10)");

// total out-migration propensity of cell (p,h): the sum over targets t and groups s of the channel propensities
// I b[h] m[p,p] eff[t,p] Sx[t,s] sigma[s,h], with the sum over targets taken once per leap and (deme, group):
// sum_s sigma[s,h] Mg[p,s] -- S multiply-adds per cell instead of (K-1) S (the targets' Q[t,h] = sum_s Sx[t,s] sigma[s,h]
// were 7 % of a dense leap's instructions in the warp kernel, whose Q table no longer fits when most haplotypes are present)
template <class DIMS, class SH>
__device__ __forceinline__ double mig_total(int p, int h, double Ii, const DIMS &D, const SH &s, const double *eff) {
    (void)eff;
    double acc = 0.0;
#pragma unroll 1
    for (int sn = 0; sn < D.S; sn++) acc += s.sigT[sn * D.H + h] * s.Mg[p * D.S + sn];
    return Ii * s.b[h] * s.mdiag[p] * acc;
}

// One event of an aggregated out-migration total of cell (p,h): its local channel, or -1 when every weight is zero.
// Shared by both kernels (same arithmetic, same pick for the same uniform).
template <class DIMS, class SH>
__device__ __forceinline__ int split_migration(int p, int h, double u, const DIMS &D, const SH &s, const double *eff) {
    const int K = D.K, H = D.H, S = D.S;
    double tot = 0.0;
#pragma unroll 1
    for (int sn = 0; sn < S; sn++) tot += s.sigT[sn * H + h] * s.Mg[p * S + sn];
    const double x = u * tot;
    double acc = 0.0, before = 0.0;
    int ssel = -1;
#pragma unroll 1
    for (int sn = 0; sn < S; sn++) {
        const double wt = s.sigT[sn * H + h] * s.Mg[p * S + sn];
        if (wt > 0.0) {
            ssel = sn;
            before = acc;
            acc += wt;
            if (x < acc) break;
        }
    }
    if (ssel < 0) return -1;
    const double sg = s.sigT[ssel * H + h], x2 = x - before;  // x2 in [0, sigma[ssel,h] * Mg[p,ssel])
    double acc2 = 0.0;
    int tsel = -1;
#pragma unroll 1
    for (int tp = 0; tp < K; tp++) {
        if (tp == p) continue;
        const double pr = eff[tp * K + p] * s.Sx[tp * S + ssel] * sg;
        if (pr > 0.0) {
            tsel = tp;
            acc2 += pr;
            if (x2 < acc2) break;
        }
    }
    if (tsel < 0) return -1;
    return D.E + (tsel - (tsel > p ? 1 : 0)) * S + ssel;
}

// One primary draw: nothing to do for lam == 0 (numpy's random_poisson(0) consumes no randomness either); a
// count that the top 32 bits of the uniform already prove to be 0 is settled here; everything else goes to
// the slow-path queue (inversion entries from the bottom, PTRS entries from the top) or, for group totals
// that are too large to aggregate, to the expansion queues.
template <class SH>
__device__ __forceinline__ void primary_draw(double lam, uint32_t hi, int owner, int code, const SH &s, int *qn) {
    int e;
    if (lam < 10.0) {
        if ((double)hi + 1.0 <= (1.0 - lam) * 4294967296.0) return;  // U < 1-lam <= exp(-lam)  =>  0
        e = atomicAdd(&qn[0], 1);
    } else {
        e = s.qcap - 1 - atomicAdd(&qn[1], 1);
    }
    s.qhi[e] = (int)hi;
    s.qoc[e] = owner | (code << 20);
}

// multinomial split of an aggregated total: n events of cell (p,h), each assigned to one channel of the
// group with probability prop_channel / prop_total (exact: independent Poissons conditioned on their sum)
template <class SH>
__device__ __forceinline__ int split_total_impl(int n, int p, int h, int code, int *row, const Dims &D, const SH &s,
                                                const double *eff, const DrawGeom &g, PhiloxCtx ctx) {
    LeapTally tr;  // the events are all of one type: the caller tallies the returned count
    tr.B = tr.Dd = tr.Sm = tr.M = tr.I = tr.G = 0;
    int booked = 0;
    const int K = D.K, H = D.H, S = D.S, U = D.U;
    const int cell = p * H + h;
    const double Ii = s.I[cell];
    ctx.dom0 = (uint32_t)(g.NBP + g.nbm + g.nbg + (code == 2 ? 0 : 1));
    uint4 w = make_uint4(0, 0, 0, 0);
    for (int e = 0; e < n; e++) {
        if ((e & 1) == 0) w = ctx.draw((uint32_t)(e >> 1));
        const double u = (e & 1) ? u53(w.z, w.w) : u53(w.x, w.y);
        int l = -1;
        if (code == 2) {  // mutation: 3U channels with propensities q[h][uk] * I
            const double x = u * (s.tmq[h] * Ii);
            double acc = 0.0;
            for (int uk = 0; uk < 3 * U; uk++) {
                double pr = s.q[h * U * 3 + uk] * Ii;
                if (pr > 0.0) {
                    l = 2 + uk;
                    acc += pr;
                    if (x < acc) break;
                }
            }
        } else {  // out-migration: the channel (target t, group s) has weight eff[t,p] Sx[t,s] sigma[s,h] (the cell's common
                  // factor cancels).  First the group by sigma[s,h] Mg[p,s] (Mg = the sum over targets, once per leap), then
                  // the target inside the group with what is left of the uniform: S + K - 1 terms, no Q[t,h] needed.
            l = split_migration(p, h, u, D, s, eff);
        }
        if (l >= 0) {
            Channel ch;
            int c = cell_channel(p, h, l, D, s, eff, ch);
            atomicAdd(&row[c], 1);
            book(ch, 1, s, tr);
            booked++;
        }
    }
    return booked;
}

// Team kernel: one out-of-line copy (the 1024-thread CTA is capped at 64 registers).  Warp kernel: inlined -- out of
// line, every `s.X[...]` inside re-read the view's (offset, stride) pair through a GENERIC pointer to the
// __grid_constant__ parameter block (LD.E, ~145 per leap, each a long-scoreboard wait with two live lanes while the
// other 13 warps of the CTA sat at the generation barrier; ncu profiles/r1_i_*).
template <class SH>
static __device__ __noinline__ int split_total(int n, int p, int h, int code, int *row, const Dims &D, const SH &s,
                                                const double *eff, const DrawGeom &g, PhiloxCtx ctx) {
    return split_total_impl(n, p, h, code, row, D, s, eff, g, ctx);
}

// one slow-path queue entry: recompute its lambda (same expression as the primary pass), finish the Poisson
// draw, then write / split the count
template <class SH>
__device__ __forceinline__ void process_entry(int e, double tau, int *row, const Dims &D, const SH &s,
                                              const double *eff, const DrawGeom &g, PhiloxCtx &ctx, LeapTally &tr) {
    const uint32_t hi = (uint32_t)s.qhi[e];
    const int oc = s.qoc[e];
    const int owner = oc & 0xfffff, code = oc >> 20;
    const int KH = D.K * D.H;
    Channel ch;
    ctx.c0 = (uint32_t)owner;
    if (owner >= KH) {  // SUSCCHANGE channel `code` of deme owner - KH
        const int c = susc_channel(owner - KH, code, D, s, ch);
        const double lam = ch.prop * tau;
        ctx.dom0 = (uint32_t)(code >> 2);
        const int n = (int)(lam < 10.0 ? poisson_inversion(lam, hi, ctx, code & 3) : poisson_ptrs(lam, ctx, code & 3));
        if (n != 0) {
            row[c] = n;
            book(ch, n, s, tr);
        }
        return;
    }
    const int p = owner >> D.hshift, h = owner & (D.H - 1);
    if (code == 2 || code == 3) {  // aggregated total of the mutation / out-migration group (lambda <= theta < 10)
        const double Ii = s.I[owner];
        const double lam = code == 2 ? s.tmq[h] * Ii * tau : mig_total(p, h, Ii, D, s, eff) * tau;
        ctx.dom0 = 0u;
        const int n = (int)poisson_inversion(lam, hi, ctx, code);
        if (n != 0) {
            int nb;
            if constexpr (SH::has_qin) nb = split_total_impl(n, p, h, code, row, D, s, eff, g, ctx);
            else nb = split_total(n, p, h, code, row, D, s, eff, g, ctx);
            if (code == 2) tr.M += nb;
            else tr.G += nb;
        }
        return;
    }
    const int l = code == 0 ? 0 : code == 1 ? 1 : 2 + 3 * D.U + (code - 4);
    const int c = cell_channel(p, h, l, D, s, eff, ch);
    const double lam = ch.prop * tau;
    const int blk = code < 4 ? 0 : 1 + ((code - 4) >> 2), q = code < 4 ? code : (code - 4) & 3;
    ctx.dom0 = (uint32_t)blk;
    const int n = (int)(lam < 10.0 ? poisson_inversion(lam, hi, ctx, q) : poisson_ptrs(lam, ctx, q));
    if (n != 0) {
        row[c] = n;
        book(ch, n, s, tr);
    }
}

template <int TEAMS>
__global__ void __launch_bounds__(TAU_TEAM * TEAMS, 1) tau_kernel(const __grid_constant__ DevState st, const __grid_constant__ SimArgs a,
                                                     const __grid_constant__ TauShared s, const int variant) {
    const Dims &D = st.D;
    const int K = D.K, H = D.H, S = D.S;
    const int tid = threadIdx.x, nt = blockDim.x;
    const DrawGeom g = draw_geom(D);
    const bool prof = (variant & 2) != 0;
    unsigned long long pc[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    long long tmark = 0;

    for (int i = threadIdx.y * blockDim.x + threadIdx.x; i < TAU_ZB / 16; i += blockDim.x * blockDim.y)
        reinterpret_cast<int4 *>(zero_buf())[i] = make_int4(0, 0, 0, 0);
    if (threadIdx.x == 0 && threadIdx.y == 0) cta_tail()[0] = 0;
    __syncthreads();  // barrier 0, once: zero buffer and tail are initialised before any team uses them
    if (tid == 0) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic writes -> async-proxy reads
    for (int r = blockIdx.x * blockDim.y + threadIdx.y; r < st.R; r += gridDim.x * blockDim.y) {
        const double *pp = st.params + (size_t)st.rep_pp[r] * D.blob;
        double *eff_g = st.eff + (size_t)r * K * K;
        long long *ctr = st.counters + (size_t)r * NCOUNT;
        const uint64_t seed = st.seeds[r];
        team_sync();
        load_replicate(st, r, D, s, pp, eff_g);
        const double *eff = s.has_effS ? (const double *)s.effS.ptr() : eff_g;
        if (s.flags[7]) {
            if (tid == 0) st.err[r] |= ERR_COUNT_OVERFLOW;
            continue;
        }
        unsigned rnd = 0;    // draw-round parity: which pair of queue counters is live
        bool restarted = false;
        long long sC = ctr[C_S];
        long long evptr = ctr[C_EVPTR], leaps = ctr[C_LEAPS];
        double t = st.time[r];
        unsigned epoch = st.epoch[r];
        long long good_attempt = ctr[C_GOOD];
        const long long ev_limit = evptr + a.iterations;  // events.ptr < events.size (:2312), intended capacity
        long long dbase = st.dense_base[r];  // leaps whose rows went to the archive: leap L is dense row L - dbase
        int *tau_counts = st.tau_counts + (size_t)r * st.dense_cap * D.Pp;
        bool lists_ready = true;  // false: segcnt is current but act/dstart/masks still have to be written

        for (long long attempt = 0; attempt < a.attempts; attempt++) {
            if (!(a.cont && attempt == 0)) epoch++;
            if (s.flags[8] != 0) {
                while (evptr < ev_limit && evptr < st.ev_cap && leaps < st.leap_cap && leaps - dbase < st.dense_cap &&
                       (a.sample_size == -1 || sC < a.sample_size) && (!a.has_time || t < (double)a.time)) {
                    int *row = tau_counts + (size_t)(leaps - dbase) * D.Pp;
                    // A leap is one GENERATION of the CTA: every team passes exactly five CTA-wide barriers (here, after
                    // Q, after the pressure sums, inside the tau minimum, after the apply pass), so all teams of the SM
                    // enter every long phase together and share its instruction fetch.  The barriers inside the
                    // variable-trip loops (draw rounds, tau halving) stay team-local.
                    align_teams();  // generation barrier 1 of 5
                    if (prof && tid == 0) tmark = clock64();
                    // ---- 0. zero-fill the dense row, clear the per-leap deltas, finish the cell lists of the
                    //         state the previous leap left, Q[p,h]
                    wipe_leap(D, s, row);
                    zero_totals(D, s);
                    if (!lists_ready) write_lists(D, s);
                    lists_ready = true;
                    q_pass(D, s);
                    for (int i = threadIdx.x; i < D.K * D.S; i += blockDim.x) mig_pressure(i, D, s, eff);
                    align_teams();  // generation barrier 2 of 5
                    TAU_MARK(0)
                    // ---- 1-2. drifts and tau (the barriers also order the zero-fill before the scatter below)
                    double tau = drifts_and_tau(D, s, eff, (int)leaps);
                    TAU_MARK(1)
                    const int nAct = s.flags[8];
                    const int *act = s.act;
                    // ---- 3. draw; halve tau and redraw on an infeasible leap (:2316-2321)
                    for (unsigned retry = 0;; retry++) {
                        LeapTally tr;
                        tr.B = tr.Dd = tr.Sm = tr.M = tr.I = tr.G = 0;
                        PhiloxCtx ctx;
                        ctx.key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
                        ctx.c1 = (uint32_t)leaps;
                        ctx.c2 = (retry & 0xffu) | (epoch << 8);
                        ctx.dstride = (uint32_t)g.GS;
                        const int n1 = nAct * g.NB1, nItems = n1 + K * g.G2;
                        for (int base = 0; base < nItems; base += nt, rnd++) {
                            int *qn = &s.flags[12 + 4 * (rnd & 1)];  // [0] inversion [1] PTRS [2] expand-mut [3] expand-mig
                            const int item = base + tid;
                            // ---- 3a. primary draws of this round's owners
                            if (item < n1) {
                                const int ai = item / g.NB1, blk = item - ai * g.NB1;
                                const int cell = act[ai];
                                const int p = cell >> D.hshift, h = cell & (H - 1);
                                const double Ii = s.I[cell];
                                double lam[4];
                                if (blk == 0) {
                                    lam[0] = s.d[h] * Ii * tau;
                                    lam[1] = s.sr[h] * Ii * s.sm[p] * tau;
                                    lam[2] = s.tmq[h] * Ii * tau;
                                    lam[3] = K > 1 ? mig_total(p, h, Ii, D, s, eff) * tau : 0.0;
                                    if (lam[2] > 0.0 && ((variant & 1) || lam[2] > TAU_THETA_MUT)) {
                                        s.xq[atomicAdd(&qn[2], 1)] = cell;
                                        lam[2] = 0.0;
                                    }
                                    if (lam[3] > 0.0 && ((variant & 1) || lam[3] > TAU_THETA_MIG)) {
                                        s.xq[nt + atomicAdd(&qn[3], 1)] = cell;
                                        lam[3] = 0.0;
                                    }
                                } else {
#pragma unroll
                                    for (int q = 0; q < 4; q++) {
                                        const int sn = (blk - 1) * 4 + q;
                                        lam[q] = sn < S ? s.b[h] * s.sigT[sn * H + h] * s.c[p] * s.Sx[p * S + sn] * Ii * tau
                                                        : 0.0;
                                    }
                                }
                                if (lam[0] > 0.0 || lam[1] > 0.0 || lam[2] > 0.0 || lam[3] > 0.0) {
                                    ctx.c0 = (uint32_t)cell;
                                    ctx.dom0 = (uint32_t)blk;
                                    const uint4 w = ctx.draw(0u);
                                    const int code0 = blk == 0 ? 0 : 4 + (blk - 1) * 4;
                                    if (lam[0] > 0.0) primary_draw(lam[0], w.x, cell, code0, s, qn);
                                    if (lam[1] > 0.0) primary_draw(lam[1], w.y, cell, code0 + 1, s, qn);
                                    if (lam[2] > 0.0) primary_draw(lam[2], w.z, cell, code0 + 2, s, qn);
                                    if (lam[3] > 0.0) primary_draw(lam[3], w.w, cell, code0 + 3, s, qn);
                                }
                            } else if (item < nItems) {
                                const int it = item - n1;
                                const int p = it / g.G2, j = it - p * g.G2;
                                double lam[4];
                                Channel ch;
#pragma unroll
                                for (int q = 0; q < 4; q++) {
                                    const int l = j * 4 + q;
                                    lam[q] = 0.0;
                                    if (l < D.SS1) {
                                        susc_channel(p, l, D, s, ch);
                                        lam[q] = ch.prop * tau;
                                    }
                                }
                                if (lam[0] > 0.0 || lam[1] > 0.0 || lam[2] > 0.0 || lam[3] > 0.0) {
                                    ctx.c0 = (uint32_t)(K * H + p);
                                    ctx.dom0 = (uint32_t)j;
                                    const uint4 w = ctx.draw(0u);
                                    if (lam[0] > 0.0) primary_draw(lam[0], w.x, K * H + p, j * 4, s, qn);
                                    if (lam[1] > 0.0) primary_draw(lam[1], w.y, K * H + p, j * 4 + 1, s, qn);
                                    if (lam[2] > 0.0) primary_draw(lam[2], w.z, K * H + p, j * 4 + 2, s, qn);
                                    if (lam[3] > 0.0) primary_draw(lam[3], w.w, K * H + p, j * 4 + 3, s, qn);
                                }
                            }
                            if (tid == 0) wipe_wait();  // the row is zero in HBM/L2 before any count is scattered into it
                            team_sync();
                            TAU_MARK(2)
                            // ---- 3b. drain.  The round's critical path is its slowest warp, so the three kinds of
                            //          slow work go to different warps and every unit gets its own thread:
                            //          inversion entries from thread 0 up, PTRS entries from the last thread
                            //          down, the channels of expanded groups from the first warp after the
                            //          inversion entries (one CHANNEL per thread; its Philox block is shared
                            //          by 4 channels, each thread recomputes it and keeps its own word)
                            const int ninv = qn[0], nptr = qn[1], nxm = qn[2], nxg = qn[3];
                            if (tid < 4) s.flags[12 + 4 * ((rnd + 1) & 1) + tid] = 0;
                            for (int e = tid; e < ninv; e += nt) process_entry(e, tau, row, D, s, eff, g, ctx, tr);
                            for (int k = nt - 1 - tid; k < nptr; k += nt) process_entry(s.qcap - 1 - k, tau, row, D, s, eff, g, ctx, tr);
                            const int nchM = 3 * D.U, nchG = (K - 1) * S;
                            const int itM = nxm * nchM, itX = itM + nxg * nchG;
                            if (itX > 0) {
                                const int first = (ninv + 31) & ~31 & (nt - 1);
                                for (int it = (tid - first) & (nt - 1); it < itX; it += nt) {
                                    int owner, lc, lbase, domb;
                                    if (it < itM) {
                                        const int xi = it / nchM;
                                        lc = it - xi * nchM;
                                        owner = s.xq[xi];
                                        lbase = 2;
                                        domb = g.NBP;
                                    } else {
                                        const int it2 = it - itM, xi = it2 / nchG;
                                        lc = it2 - xi * nchG;
                                        owner = s.xq[nt + xi];
                                        lbase = D.E;
                                        domb = g.NBP + g.nbm;
                                    }
                                    const int p = owner >> D.hshift, h = owner & (H - 1);
                                    Channel ch;
                                    const int c = cell_channel(p, h, lbase + lc, D, s, eff, ch);
                                    const double lam = ch.prop * tau;
                                    if (lam > 0.0) {
                                        ctx.c0 = (uint32_t)owner;
                                        ctx.dom0 = (uint32_t)(domb + (lc >> 2));
                                        const uint4 w = ctx.draw(0u);
                                        const int n = (int)poisson_draw(lam, pick_word(w, lc & 3), ctx, lc & 3);
                                        if (n != 0) {
                                            row[c] = n;
                                            book(ch, n, s, tr);
                                        }
                                    }
                                }
                            }
                            if (tr.B) atomicAdd(&s.flags[EV_BIRTH], tr.B);
                            if (tr.Dd) atomicAdd(&s.flags[EV_DEATH], tr.Dd);
                            if (tr.Sm) atomicAdd(&s.flags[EV_SAMPLING], tr.Sm);
                            if (tr.M) atomicAdd(&s.flags[EV_MUTATION], tr.M);
                            if (tr.I) atomicAdd(&s.flags[EV_SUSCCHANGE], tr.I);
                            if (tr.G) atomicAdd(&s.flags[EV_MIGRATION], tr.G);
                            tr.B = tr.Dd = tr.Sm = tr.M = tr.I = tr.G = 0;
                            team_sync();
                            TAU_MARK(3)
                        }
                        // feasibility (:2522-2528).  The reference books migration arrivals on the SOURCE cell
                        // (quirk Q8), so its test can pass while the cell that is really depleted goes negative;
                        // from then on every redraw fails and the reference halves tau forever.  Here a leap must
                        // pass the reference's test AND leave the applied state inside [0, size].
                        int bad = 0;
                        for (int i = tid; i < K * H; i += nt) {
                            const double sz = s.sizeD[i >> D.hshift];
                            const double v = s.I[i] + (double)s.chkI[i];
                            const double u = s.I[i] + (double)s.updI[i];
                            if (v < 0.0 || v > sz || u < 0.0 || u > sz) bad = 1;
                        }
                        for (int i = tid; i < K * S; i += nt) {
                            const double v = s.Sx[i] + (double)s.dSx[i];
                            if (v < 0.0 || v > s.sizeD[i / S]) bad = 1;
                        }
                        bad = team_or(bad);
                        TAU_MARK(4)
                        if (!bad) break;
                        tau *= 0.5;
                        wipe_leap(D, s, row);  // rare path
                        team_sync();
                        if (retry >= 80) {  // tau * 2^-80: nothing can fire any more, yet the state fails the test
                            if (tid == 0) st.err[r] |= ERR_TAU_STUCK;
                            tau = 0.0;
                            break;
                        }
                    }
                    // ---- 5. apply (UpdateCompartmentCounts_tau, :2536-2593); per-deme totals; first pass of the
                    //         ordered cell compaction (the second pass runs at the top of the next leap)
                    for (int i = tid; i < K * H; i += nt) {
                        const double v = s.I[i] + (double)s.updI[i];
                        s.I[i] = v;
                        if (v != 0.0) atomicAdd(&s.tot[i >> D.hshift], (int)v);
                    }
                    for (int i = tid; i < K * S; i += nt) s.Sx[i] += (double)s.dSx[i];
                    count_cells(D, s);
                    lists_ready = false;
                    t += tau;
                    sC += s.flags[EV_SAMPLING];  // sCounter gates the loop (:2312): exact per leap
                    if (tid < 6) s.tally64[tid] += s.flags[tid];
                    if (tid == 0) {
                        double *tau_tt = st.tau_tt + ((size_t)r * st.leap_cap + leaps) * 2;
                        tau_tt[0] = t;
                        tau_tt[1] = tau;
                        st.ev_time[(size_t)r * st.ev_cap + evptr] = t;
                        st.ev_desc[(size_t)r * st.ev_cap + evptr] = pack_multi((uint32_t)leaps);
                    }
                    leaps++;
                    evptr++;
                    align_teams();  // generation barrier 5 of 5
                    TAU_MARK(5)
                    // ---- extinction test and CheckLockdown for every deme (:2326-2329)
                    const int alive = total_cells(s);
                    if (tid == 0) s.flags[8] = alive;  // (every thread computed the same value; nobody reads it before
                                                       //  the next barrier)
                    if (alive == 0) break;
                    lockdown_pass(st, r, D, s, pp, eff_g, t, s.tot);
                    TAU_MARK(6)
                    if (prof && tid == 0) pc[7] += 1;
                }
            }
            // ---- extinction-retry (:2331-2335): <= 100 log rows with iterations > 100 => Restart (:714-738)
            if (evptr + st.ev_base[r] <= 100 && a.iterations > 100) {
                evptr = 0;
                leaps = 0;
                sC = 0;
                t = 0.0;
                restarted = true;
                team_sync();
                if (tid < 6) s.tally64[tid] = 0;
                for (int i = tid; i < K * H; i += nt) s.I[i] = (double)st.initI[(size_t)r * K * H + i];
                for (int i = tid; i < K * S; i += nt) s.Sx[i] = (double)st.initSx[(size_t)r * K * S + i];
                rebuild_lists(D, s);
                lists_ready = true;
                lockdown_pass(st, r, D, s, pp, eff_g, t, s.tot);
                team_sync();
                good_attempt = 0;
                dbase = 0;  // the archive of the wiped leaps goes with them
                if (tid == 0) {
                    ctr[C_MIGN] = 0;
                    st.dense_base[r] = 0;
                    st.sp_n[r] = 0;
                }
            } else {
                good_attempt = attempt + 1;
                break;
            }
        }

        // ---- commit the replicate back to HBM
        if (tid == 0) wipe_wait();
        team_sync();
        for (int i = tid; i < K * H; i += nt) st.I[(size_t)r * K * H + i] = (long long)s.I[i];
        for (int i = tid; i < K * S; i += nt) st.Sx[(size_t)r * K * S + i] = (long long)s.Sx[i];
        for (int i = tid; i < K; i += nt) {
            st.cd[(size_t)r * K + i] = s.cd[i];
            st.ceff[(size_t)r * K + i] = s.c[i];
            st.maxEBM[(size_t)r * K + i] = s.maxEBM[i];
            st.lock[(size_t)r * K + i] = s.lock[i];
        }
        if (tid == 0) {
            // counters carried over from earlier calls unless a Restart wiped them (:714-738)
            static_assert(C_B == EV_BIRTH && C_D == EV_DEATH && C_S == EV_SAMPLING && C_M == EV_MUTATION &&
                          C_I == EV_SUSCCHANGE && C_MIGP == EV_MIGRATION, "counter order follows the event codes");
            for (int j = 0; j < 6; j++) ctr[j] = (restarted ? 0 : ctr[j]) + s.tally64[j];
            ctr[C_S] = sC;
            ctr[C_SWAP] += s.flags[10];
            ctr[C_GOOD] = good_attempt;
            ctr[C_EVPTR] = evptr;
            ctr[C_LEAPS] = leaps;
            long long ginf = 0;
            for (int i = 0; i < K * H; i++) ginf += (long long)s.I[i];
            ctr[C_GINF] = ginf;
            st.time[r] = t;
            st.epoch[r] = epoch;
        }
        team_sync();
    }
    if (prof && tid == 0)
        for (int k = 0; k < 8; k++) atomicAdd(&g_tau_phase_cycles[k], pc[k]);
    // ---- this team is out of replicates: keep answering the generation barriers until every team is.  A team
    // announces itself between barrier 5 of its last generation and barrier 1 of the next; the counter is read
    // between barriers 1 and 2, where no announcement can be in flight, so all teams take the same decision.
    team_sync();
    if (tid == 0) atomicAdd(&cta_tail()[0], 1);
    for (;;) {
        align_teams();
        if (*(volatile int *)cta_tail() >= (int)blockDim.y) break;
        align_teams();
        align_teams();
        align_teams();
        align_teams();
    }
}

// Deterministic parity tap: propensities of the current state in positional order, drifts and tau.
__global__ void __launch_bounds__(256) propensity_kernel(const __grid_constant__ DevState st,
                                                         const __grid_constant__ TauShared s, int r, double *out,
                                                         double *dI, double *dS, double *tau_out) {
    const Dims &D = st.D;
    const double *pp = st.params + (size_t)st.rep_pp[r] * D.blob;
    const double *eff_g = st.eff + (size_t)r * D.K * D.K;
    load_replicate(st, r, D, s, pp, eff_g);
    const double *eff = s.has_effS ? (const double *)s.effS.ptr() : eff_g;
    q_pass(D, s);
    for (int i = threadIdx.x; i < D.K * D.S; i += blockDim.x) mig_pressure(i, D, s, eff);
    team_sync();
    double tau = drifts_and_tau(D, s, eff, 0);
    for (int c = threadIdx.x; c < D.P; c += blockDim.x) {
        Channel ch;
        int owner, l;
        decode_channel(c, D, s, eff, ch, owner, l);
        out[c] = ch.prop;
    }
    for (int i = threadIdx.x; i < D.K * D.H; i += blockDim.x) dI[i] = s.dI[i];
    for (int i = threadIdx.x; i < D.K * D.S; i += blockDim.x) dS[i] = s.dS[i];
    if (threadIdx.x == 0) *tau_out = tau;
}

}  // namespace vg
#include "tau_warp.cuh"
namespace vg {

// host launchers ---------------------------------------------------------------------------------
template <int TEAMS>
static cudaError_t launch_tau_cfg(const DevState &st, const SimArgs &a, cudaStream_t stream, int num_sms, int variant) {
    const TauShared lay = tau_layout(st.D, false, TAU_TEAM);
    const size_t stride = ((size_t)lay.bytes + 15) & ~(size_t)15;
    const size_t smem = stride * TEAMS + TAU_CTA_TAIL;
    cudaError_t e = cudaFuncSetAttribute(tau_kernel<TEAMS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int per_sm = 1;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tau_kernel<TEAMS>, TAU_TEAM * TEAMS, smem);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    int grid = num_sms * per_sm;
    const int need = (st.R + TEAMS - 1) / TEAMS;
    if (grid > need) grid = need;
    tau_kernel<TEAMS><<<grid, dim3(TAU_TEAM, TEAMS), smem, stream>>>(st, a, lay, variant);
    return cudaGetLastError();
}

// Can the warp-per-replicate kernel hold the shape in layout L?  Cell ids are held as uint16, a cell's local channels
// in the 12-bit field of a queue entry.
static bool tau_warp_fits(const Dims &D, const WarpLayout &L) {
    return L.nwarps >= 1 && D.K * D.H < 65536 && D.E + (D.K - 1) * D.S < 4000;
}
static size_t tau_team_stride(const Dims &D) { return ((size_t)tau_layout(D, false, TAU_TEAM).bytes + 15) & ~(size_t)15; }

// Can any tau kernel hold one replicate of this shape (launch_tau's own test, without the variant bits that force one
// of the two mappings)?
bool tau_fits(const Dims &D, int uniform_pp) {
    if ((long long)D.K * D.H + D.K >= (1 << 20)) return false;
    if (tau_team_stride(D) + TAU_CTA_TAIL <= (size_t)227 * 1024) return true;
    return tau_warp_fits(D, warp_layout(D, uniform_pp >= 0, uniform_pp >= 0 ? uniform_pp : 0, 227 * 1024));
}

// Warp kernel instances with the model shape compiled in (DimsC), all on the mask path with eff in shared memory:
// T3 (3, 10, 3), the benchmark's model, and (2, 10, 3), the Table 3 model of the configs[4] sweep.  nullptr when the
// shape is another one.
template <int U, int K, int S>
static const void *tau_warp_fixed(const Dims &D, bool prof) {
    if (!DimsC<U, K, S>::matches(D)) return nullptr;
    return prof ? (const void *)tau_warp_kernel<DimsC<U, K, S>, true, true, true>
                : (const void *)tau_warp_kernel<DimsC<U, K, S>, false, true, true>;
}

// Default: the warp-per-replicate kernel (tau_warp.cuh), one CTA per SM with as many warps as the shared memory
// holds (<= 14), with the model shape compiled in where an instance exists for it (variant bit 6: the runtime-shape
// instance on every shape).  The team kernel (256-thread teams, CTA-wide generations) stays available as a parity tap:
// variant bit 2 (vgsim_set_tau_variant); bit 3 forces the warp kernel.  *fixed_shape gets U << 16 | K << 8 | S of the
// compiled-in shape that ran, 0 for a runtime-shape kernel.
cudaError_t launch_tau(const DevState &st, const SimArgs &a, cudaStream_t stream, int num_sms, int variant, int uniform_pp,
                       int *order_buf, int *fixed_shape) {
    *fixed_shape = 0;
    if ((long long)st.D.K * st.D.H + st.D.K >= (1 << 20)) return cudaErrorInvalidValue;  // owner id is packed in 20 bits
    const size_t stride = tau_team_stride(st.D);
    int teams = (int)((227 * 1024 - TAU_CTA_TAIL) / stride);
    if (teams > 4) teams = 4;
    if (teams < 1) teams = 1;
    bool team = (variant & 4) != 0;
    const bool force_warp = (variant & 8) != 0;
    // Few replicates (all of them resident at once as 256-thread teams): the GPU is latency- not throughput-bound, and a
    // team walks a leap sooner than a single warp does -- 8.1x at the world shape (K = 100: the K x K x H force-of-
    // infection sums), 32 replicates x 1,200 leaps: 607 ms vs 4,948 ms (profiles/r1_k_*), same log bit for bit.
    const bool team_fits = stride + TAU_CTA_TAIL <= (size_t)227 * 1024;  // else only the warp kernel's leaner slice may fit
    if (!team && !force_warp && team_fits && st.R <= num_sms * teams) team = true;
    if (!team) {
        WarpLayout L = warp_layout(st.D, uniform_pp >= 0, uniform_pp >= 0 ? uniform_pp : 0, 227 * 1024);
        L.gsync = (variant & 16) ? 0 : 3;  // lockstep generations: the warps of a CTA meet at leap start and before the draws
        if (tau_warp_fits(st.D, L)) {
            const WS ws = make_ws(L, st.D);
            const bool prof = (variant & 2) != 0, masks = L.use_masks != 0;
            const void *kern = nullptr;
            if (L.has_eff && masks && !(variant & 64)) {
                if ((kern = tau_warp_fixed<3, 10, 3>(st.D, prof))) *fixed_shape = 3 << 16 | 10 << 8 | 3;
                else if ((kern = tau_warp_fixed<2, 10, 3>(st.D, prof))) *fixed_shape = 2 << 16 | 10 << 8 | 3;
            }
            if (!kern)
                kern = L.has_eff ? (masks ? (prof ? (const void *)tau_warp_kernel<Dims, true, true, true> : (const void *)tau_warp_kernel<Dims, false, true, true>)
                                          : (prof ? (const void *)tau_warp_kernel<Dims, true, true, false> : (const void *)tau_warp_kernel<Dims, false, true, false>))
                                 : (prof ? (const void *)tau_warp_kernel<Dims, true, false, false> : (const void *)tau_warp_kernel<Dims, false, false, false>);
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total_bytes);
            if (e != cudaSuccess) return e;
            int grid = (st.R + L.nwarps - 1) / L.nwarps;
            if (grid > num_sms) grid = num_sms;
            // size-sorted schedule (only useful with lockstep generations and more than one visit per CTA)
            const bool sorted = L.gsync != 0 && order_buf != nullptr && st.R > grid * L.nwarps && !(variant & 32);
            if (sorted) {
                tau_weight_kernel<<<(st.R * 32 + 255) / 256, 256, 0, stream>>>(st, order_buf);
                tau_order_kernel<<<1, 1024, 0, stream>>>(st.R, st.D.K * st.D.H, order_buf, order_buf + st.R);
            }
            const int *order = sorted ? order_buf + st.R : nullptr;
            void *args[] = {(void *)&st, (void *)&a, (void *)&L, (void *)&ws, (void *)&variant, (void *)&order};
            return cudaLaunchKernel(kern, dim3(grid), dim3(L.nwarps * 32), args, L.total_bytes, stream);
        }
        // a single replicate's state does not fit one warp slice: fall through to the team kernel
    }
    if (teams >= 4) return launch_tau_cfg<4>(st, a, stream, num_sms, variant);
    if (teams == 3) return launch_tau_cfg<3>(st, a, stream, num_sms, variant);
    if (teams == 2) return launch_tau_cfg<2>(st, a, stream, num_sms, variant);
    return launch_tau_cfg<1>(st, a, stream, num_sms, variant);
}

cudaError_t tau_cta_end(unsigned long long *out1024, int reset) {
    cudaError_t e = cudaMemcpyFromSymbol(out1024, g_tau_cta_end, 1024 * sizeof(unsigned long long));
    if (e == cudaSuccess && reset) {
        static unsigned long long z[1024];
        for (int i = 0; i < 1024; i++) z[i] = (i & 1) ? 0ull : ~0ull;
        e = cudaMemcpyToSymbol(g_tau_cta_end, z, sizeof(z));
    }
    return e;
}

cudaError_t tau_phase_cycles(unsigned long long *out16, int reset) {
    cudaError_t e = cudaMemcpyFromSymbol(out16, g_tau_phase_cycles, 16 * sizeof(unsigned long long));
    if (e == cudaSuccess && reset) {
        unsigned long long z[16] = {0};
        z[11] = ~0ull;  // slot 11 is a minimum
        e = cudaMemcpyToSymbol(g_tau_phase_cycles, z, sizeof(z));
    }
    return e;
}

cudaError_t launch_propensities(const DevState &st, int r, double *out, double *dI, double *dS, double *tau,
                                cudaStream_t stream) {
    const TauShared lay = tau_layout(st.D, true);
    size_t smem = (((size_t)lay.bytes + 15) & ~(size_t)15) + TAU_CTA_TAIL;
    cudaError_t e = cudaFuncSetAttribute(propensity_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    propensity_kernel<<<1, dim3(TAU_TEAM, 1), smem, stream>>>(st, lay, r, out, dI, dS, tau);
    return cudaGetLastError();
}

}  // namespace vg
