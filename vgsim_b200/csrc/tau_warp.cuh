// Warp-per-replicate tau-leaping kernel (included by tau_kernel.cu; shares its channel / draw helpers).
//
// Why a second mapping: ncu of the team kernel (profiles/r1_e_*) shows 66 % of all warp samples parked on
// barriers -- every phase of a leap lasts as long as its slowest warp (a handful of Poisson slow paths, a
// 1-lane multinomial split) while the other 31 warps of the SM idle, and the 64-register cap of a
// 1024-thread CTA spills.  At T3 a leap touches ~70 infectious cells and ~200 real Poisson draws: that is
// warp-sized work.  Here ONE WARP owns a replicate: no named barriers, no CTA-wide generations, every phase
// is a lane-strided loop closed by __syncwarp(), and 14 independent replicates per SM keep the issue
// slots busy while any one of them waits on a dependent chain.
//
// Per-replicate state lives in the warp's slice of dynamic shared memory: I as int32 (converted on use),
// per-leap deltas, the ordered list of infectious cells, presence masks, the slow-path queue.  Q[p,h] is
// recomputed where needed instead of stored.  The parameter point is staged ONCE per CTA when every
// replicate of the launch uses the same point (the common case), else once per warp.
//
// The arithmetic is the team kernel's: same drift / propensity expressions (shared template functions),
// same summation orders, same Philox addressing (owner, leap, retry|epoch, block), same samplers -- a leap
// is a pure function of (state, seed), so the two kernels produce the same log.  The team kernel stays as a
// parity tap (variant bit 2).
//
// The kernel and its helpers are templated on the dims type: `Dims` reads the model shape at run time, `DimsC<U, K, S>`
// has it compiled in (T3 (3, 10, 3) and the configs[4] model (2, 10, 3); launch_tau picks the instance, variant bit 6
// forces the runtime one).  Same source, same arithmetic, same log; the fixed-shape instance does without the runtime
// divisions of the item decode and the per-cell sums, the shape-derived values held in registers across the leap loop,
// and the branches the shape never takes.
#pragma once

namespace vg {

// Slow-path queue entries per warp.  >= 64: half a round (two words per lane) must fit an empty queue.  Round 2, final
// kernel (ms at t = 60 / 90 / 120): 96 entries 4.39 / 12.64 / 26.34, 112 entries 4.36 / 12.32 / 25.95 -- the out-migration
// totals no longer read the per-leap Q table, so the queue gets the room
constexpr int TW_QCAP = 112;
// Warps (= replicates in flight) per CTA: 148 x 14 = 2072 replicates in flight.  ptxas gives a 448-thread CTA 128 registers
// per thread (4 warps of an SM sub-partition share 16 K registers; 144 does not launch), so 15-16 warps would cost no
// registers -- at T3 the shared-memory slice (14.4 KB + Q table) is the limit
constexpr int TW_MAX_WARPS = 14;

struct WarpLayout {
    int nwarps;        // warps (= replicates in flight) per CTA
    int par_shared;    // 1: one parameter block per CTA (all replicates use point pp0); 0: one per warp
    int pp0;
    int o_par, o_nbr, o_warp0, warp_bytes;
    // inside the parameter block (bytes)
    int p_b, p_d, p_sr, p_tmq, p_q, p_sigT, p_sb, p_T, p_sm, p_mdiag, p_sizeD, p_startN, p_endN, p_g, p_qmax, par_bytes;
    // inside a warp slice (bytes)
    int w_par, w_cd, w_c, w_maxEBM, w_eff, w_Sx, w_Bp, w_Rp, w_I, w_chk, w_upd, w_act, w_dSx, w_lock, w_tot, w_dstart,
        w_colcnt, w_colmask, w_rowmask, w_hlist, w_qlam, w_qhi, w_qoc, w_xq, w_sqp, w_cnt, w_tally, w_hidx, w_qtab;
    int qtab_cap;      // doubles in the per-leap Q table (0: always recompute)
    int qcap, xcap;
    int has_eff, use_masks;
    int o_done, gsync, gevery;  // gevery: the warps meet only every gevery-th leap of each warp
    int ggroup;                  // warps per lockstep group (0: the whole CTA); every group has its own named barrier
    int total_bytes;
    // n / d = __umulhi(n, m) for the small divisors of the item decode (n < 2^20, d <= 4096: exact)
    unsigned mS, mS1, mNBT, mG2, mnbm, mnbg, mK;
};
// The model dimensions as compile-time constants (make_dims' formulas) for the kernel instances of the common shapes.
// Every dimension the leap loop reads is shadowed by a constant of the same name, so the helpers, templated on the dims
// type, read D.K, D.H, ... alike for both: with a DimsC the divisions by K, S and 3U become multiplies, the loop bounds
// and group sizes constants, the branches the shape never takes drop out, and nothing of it holds a register.  The
// members that only the cold paths read (P, the blob offsets) stay those of the Dims it is built from.
template <int U_, int K_, int S_>
struct DimsC : Dims {
    static constexpr int U = U_, K = K_, S = S_, H = 1 << (2 * U_), hshift = 2 * U_;
    static constexpr int E = 2 + 3 * U + S, SS1 = S * (S - 1), PD = SS1 + H * E, NA = K * (K - 1) * S * H;
    static constexpr int Pp = (NA + K * PD + 7) & ~7;
    __device__ DimsC(const Dims &d) : Dims(d) {}
    static bool matches(const Dims &d) {
        return d.U == U && d.K == K && d.S == S && d.H == H && d.hshift == hshift && d.E == E && d.SS1 == SS1 &&
               d.PD == PD && d.NA == NA && d.Pp == Pp;
    }
};
// how the kernel holds its dimensions: the runtime shape by reference into its parameter block, a DimsC by value
template <class DIMS>
struct DimsRef {
    using type = const DIMS;
};
template <>
struct DimsRef<Dims> {
    using type = const Dims &;
};

inline unsigned div_magic(int d) { return d > 1 ? (unsigned)((0x100000000ull + (unsigned)d - 1) / (unsigned)d) : 0u; }
__device__ __forceinline__ int fdiv(int n, unsigned magic, int d) { return d > 1 ? (int)__umulhi((unsigned)n, magic) : n; }

inline WarpLayout warp_layout(const Dims &D, bool par_shared, int pp0, int max_bytes) {
    WarpLayout L;
    L.gsync = 0;
    L.gevery = 1;
    L.ggroup = 0;
    const int K = D.K, H = D.H, S = D.S, U = D.U, KH = K * H, KS = K * S;
    L.par_shared = par_shared ? 1 : 0;
    L.pp0 = pp0;
    L.use_masks = (H <= 64 && K <= 32) ? 1 : 0;
    L.has_eff = tau_eff_in_smem(D) ? 1 : 0;
    L.qcap = TW_QCAP;
    L.xcap = 64;
    {
        const int NBT = (S + 3) >> 2, G2 = (S * (S - 1) + 3) >> 2, nbm = (3 * U + 3) >> 2, nbg = ((K - 1) * S + 3) >> 2;
        L.mS = div_magic(S); L.mS1 = div_magic(S - 1); L.mNBT = div_magic(NBT); L.mG2 = div_magic(G2);
        L.mnbm = div_magic(nbm); L.mnbg = div_magic(nbg); L.mK = div_magic(K);
    }
    int o = 0;
    auto take = [&](int &f, int bytes, int align) {
        o = (o + align - 1) & ~(align - 1);
        f = o;
        o += bytes;
    };
    // parameter block
    take(L.p_b, H * 8, 8); take(L.p_d, H * 8, 8); take(L.p_sr, H * 8, 8); take(L.p_tmq, H * 8, 8);
    take(L.p_q, L.use_masks ? H * U * 3 * 8 : 0, 8);  /* qin: inflow rates by (target haplotype, neighbour slot) */ take(L.p_sigT, S * H * 8, 8); take(L.p_sb, S * H * 8, 8); take(L.p_T, S * S * 8, 8);
    take(L.p_sm, K * 8, 8); take(L.p_mdiag, K * 8, 8); take(L.p_sizeD, K * 8, 8); take(L.p_startN, K * 8, 8);
    take(L.p_endN, K * 8, 8); take(L.p_g, H * 4, 8); take(L.p_qmax, 8, 8);
    L.par_bytes = (o + 15) & ~15;
    // warp slice
    o = 0;
    L.w_par = 0;
    if (!par_shared) o = L.par_bytes;
    take(L.w_cd, K * 8, 8); take(L.w_c, K * 8, 8); take(L.w_maxEBM, K * 8, 8);
    take(L.w_qlam, L.qcap * 8, 8);
    take(L.w_eff, L.has_eff ? K * K * 8 : 0, 8);
    take(L.w_Sx, KS * 8, 8); take(L.w_Bp, KS * 8, 8); take(L.w_Rp, KS * 8, 8);
    take(L.w_rowmask, L.use_masks ? K * 8 : 0, 8);
    take(L.w_tally, 8 * 8, 8);
    take(L.w_I, KH * 4, 16);
    take(L.w_chk, KH * 4, 16);   // chk and upd are wiped together: keep them adjacent
    take(L.w_upd, KH * 4, 16);
    take(L.w_act, KH * 2, 16);  // uint16 cell ids (KH < 65536); 16-aligned: the int4 wipe of chk/upd may round up into the padding before it
    take(L.w_dSx, KS * 4, 4); take(L.w_lock, K * 4, 4); take(L.w_tot, K * 4, 4); take(L.w_dstart, (K + 1) * 4, 4);
    take(L.w_colmask, L.use_masks ? H * 4 : 0, 4);
    if (L.use_masks) L.w_colcnt = L.w_colmask;  // "present anywhere" is colmask != 0 on the mask path
    else take(L.w_colcnt, H * 4, 4);
    take(L.w_hlist, H * 4, 4);
    take(L.w_qhi, L.qcap * 4, 4); take(L.w_qoc, L.qcap * 4, 4); take(L.w_xq, 2 * L.xcap * 2, 4);  // uint16 cell ids
    take(L.w_sqp, 64 * 4, 4);  // parked totals: owner | kind | n in one word, TW_SQCAP of them
    take(L.w_cnt, 8 * 4, 4);
    take(L.w_hidx, H * 2, 2);
    const int fixed_bytes = (o + 15) & ~15;
    L.w_qtab = fixed_bytes;
    L.qtab_cap = 0;
    L.warp_bytes = fixed_bytes;
    // CTA
    o = 0;
    L.o_done = o;
    o += 64;  // one counter per lockstep group (<= 15 groups)
    L.o_par = o;
    if (par_shared) o += L.par_bytes;
    L.o_nbr = o;
    if (L.use_masks) o += H * 8;
    o = (o + 15) & ~15;
    L.o_warp0 = o;
    int nw = (max_bytes - o) / L.warp_bytes;
    if (nw > TW_MAX_WARPS) nw = TW_MAX_WARPS;
    L.nwarps = nw;
    if (nw >= 1) {  // what is left of the shared memory holds the per-leap table of Q[p, present h]
        int spare = ((max_bytes - o) / nw - L.warp_bytes) & ~15;
        if (spare > KH * 8) spare = (KH * 8 + 15) & ~15;
        L.qtab_cap = spare / 8;
        L.warp_bytes += spare;
    }
    L.total_bytes = o + (nw > 0 ? nw : 0) * L.warp_bytes;
    return L;
}

// ---- shared-memory views handed to the channel / draw helpers (same member names as TauShared) ---------
// A view is (byte offset, per-warp stride): address = smem + off + scale * warp index.  CTA-shared arrays have
// scale 0.  The whole WS is a __grid_constant__ kernel parameter, so the ~50 pairs sit in the constant bank
// (one IMAD per address) and helpers can take it by reference without a local-memory copy.
__device__ __forceinline__ unsigned w_index() { return threadIdx.x >> 5; }
template <class T>
struct WArr {
    int off, scale;
    __device__ __forceinline__ T *ptr() const { return reinterpret_cast<T *>(smem_raw + (unsigned)(off + scale * (int)w_index())); }
    __device__ __forceinline__ T &operator[](int i) const { return ptr()[i]; }
    __device__ __forceinline__ operator T *() const { return ptr(); }
};
struct WIval {  // infectious counts: int32 in shared memory, fp64 to the arithmetic
    WArr<int> raw;
    __device__ __forceinline__ double operator[](int i) const { return (double)raw.ptr()[i]; }
};
struct WQval {  // Q[p,h] = sum_s Sx[p,s] sigma[s,h] (same order as the team kernel's q_pass): read from the per-leap
                // table of (deme, present haplotype) pairs when it fits (cnt[4] = its row stride), else recomputed
    WArr<double> Sx, sg, tab;
    WArr<unsigned short> hidx;
    WArr<int> cnt;
    int H, S, hshift;
    __device__ __forceinline__ double operator[](int i) const {
        const int p = i >> hshift, h = i & (H - 1);
        const int stride = cnt.ptr()[4];
        if (stride > 0) return tab.ptr()[p * stride + hidx.ptr()[h]];
        const double *sx = Sx.ptr(), *sig = sg.ptr();
        double Q = 0.0;
#pragma unroll 1
        for (int sn = 0; sn < S; sn++) Q += sx[p * S + sn] * sig[sn * H + h];
        return Q;
    }
};
struct WGq {  // mutation channel rates q[h][u][k]: read from the parameter blob in global memory (cold: a mutation
              // event or an expanded group); the hot drift sums use the shared-memory inflow table qin instead
    WArr<long long> slot;  // tally64: entry 7 holds the replicate's blob pointer
    int o_q;
    __device__ __forceinline__ double operator[](int i) const {
        return __ldg(reinterpret_cast<const double *>(slot.ptr()[7]) + o_q + i);
    }
};
struct WS {
    static constexpr bool has_qin = true;
    WArr<double> b, d, sr, qin, tmq, sigT, sb, T, sm, mdiag, sizeD, startN, endN;
    WArr<double> qmax;  // [0]: largest mutation channel rate of the parameter point (bounds the inflow into empty cells)
    WGq q;
    WArr<int> g;
    WArr<double> cd, c, maxEBM, effS, Sx, Bp, Rp, Mg;
    WIval I;
    WQval Qm;
    WArr<int> Iraw, chkI, updI, dSx, lock, tot, dstart, colcnt, colmask, hlist, qhi, qoc, sqp, cnt;
    WArr<unsigned short> act, hidx, xq;
    WArr<double> qtab, qlam;
    int qtab_cap;
    WArr<long long> tally64;
    WArr<unsigned long long> rowmask, nbrmask;
    int qcap;
    bool has_effS;
};
// the mask path (H <= 64, K <= 32) is a compile-time property of the kernel instance: helpers see s.use_masks as a constant
template <bool MASKS>
struct WSX : WS {
    static constexpr bool use_masks = MASKS;
};

inline WS make_ws(const WarpLayout &L, const Dims &D) {
    WS s;
    const int wb = L.o_warp0, ws = L.warp_bytes;
    const int pb = L.par_shared ? L.o_par : wb + L.w_par, ps = L.par_shared ? 0 : ws;
    auto P = [&](int o) { WArr<double> a; a.off = pb + o; a.scale = ps; return a; };
    auto Wd = [&](int o) { WArr<double> a; a.off = wb + o; a.scale = ws; return a; };
    auto Wi = [&](int o) { WArr<int> a; a.off = wb + o; a.scale = ws; return a; };
    s.b = P(L.p_b); s.d = P(L.p_d); s.sr = P(L.p_sr); s.tmq = P(L.p_tmq); s.qin = P(L.p_q); s.sigT = P(L.p_sigT);
    s.sb = P(L.p_sb); s.T = P(L.p_T); s.sm = P(L.p_sm); s.mdiag = P(L.p_mdiag); s.sizeD = P(L.p_sizeD);
    s.startN = P(L.p_startN); s.endN = P(L.p_endN); s.qmax = P(L.p_qmax);
    s.g.off = pb + L.p_g; s.g.scale = ps;
    s.cd = Wd(L.w_cd); s.c = Wd(L.w_c); s.maxEBM = Wd(L.w_maxEBM); s.effS = Wd(L.w_eff);
    s.Sx = Wd(L.w_Sx); s.Bp = Wd(L.w_Bp); s.Rp = Wd(L.w_Rp);
    s.Mg = s.Rp;  // the return-flow sums are dead once the susceptible drifts are done: Mg takes their place until the next leap
    s.Iraw = Wi(L.w_I); s.I.raw = s.Iraw;
    s.chkI = Wi(L.w_chk); s.updI = Wi(L.w_upd); s.act.off = wb + L.w_act; s.act.scale = ws; s.dSx = Wi(L.w_dSx); s.lock = Wi(L.w_lock);
    s.tot = Wi(L.w_tot); s.dstart = Wi(L.w_dstart); s.colcnt = Wi(L.w_colcnt); s.colmask = Wi(L.w_colmask);
    s.hlist = Wi(L.w_hlist); s.qhi = Wi(L.w_qhi); s.qoc = Wi(L.w_qoc); s.xq.off = wb + L.w_xq; s.xq.scale = ws; s.sqp = Wi(L.w_sqp); s.cnt = Wi(L.w_cnt);
    s.tally64.off = wb + L.w_tally; s.tally64.scale = ws;
    s.q.slot = s.tally64; s.q.o_q = D.o_q;
    s.hidx.off = wb + L.w_hidx; s.hidx.scale = ws;
    s.qtab = Wd(L.w_qtab);
    s.qlam = Wd(L.w_qlam);
    s.qtab_cap = L.qtab_cap;
    s.Qm.Sx = s.Sx; s.Qm.sg = s.sigT; s.Qm.H = D.H; s.Qm.S = D.S; s.Qm.hshift = D.hshift;
    s.Qm.tab = s.qtab; s.Qm.hidx = s.hidx; s.Qm.cnt = s.cnt;
    s.rowmask.off = wb + L.w_rowmask; s.rowmask.scale = ws;
    s.nbrmask.off = L.o_nbr; s.nbrmask.scale = 0;
    s.qcap = L.qcap;
    s.has_effS = L.has_eff != 0;
    return s;
}

// Zero-fill of a dense log row with 256-bit stores (STG.E.256 of RZ: no data registers; rows are 32-byte aligned
// because Dims::Pp is a multiple of 8): one 1 KB line group per warp instruction, 103 instructions for a T3 row.
// The TMA bulk-copy wipe of the team kernel stalled its issuing lane for 14 % of all warp samples here (ncu,
// profiles/r1_f_*): with one warp per replicate nobody else hides that, plain stores do.  The later scatter into
// the row is ordered behind these stores by the __syncwarp()s in between.
struct alignas(32) Row32 {
    int v[8];
};
__device__ __forceinline__ void st_zero32(Row32 *p) {
    asm volatile("st.global.v8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};" ::"l"(p), "r"(0) : "memory");
}
__device__ __forceinline__ void w_wipe_row(int *row, int n32) {
    Row32 *z = reinterpret_cast<Row32 *>(row);
#pragma unroll 4
    for (int i = threadIdx.x & 31; i < n32; i += 32) st_zero32(z + i);
}

// The wipe of the NEXT leap's row is spread over the dense loops of the current leap (a few stores per round):
// issued in one burst at the top of a leap, the 14 lockstepped warps of every SM push 1.5 MB into the store path at
// the same moment and sit on it (18 % of all warp samples, ncu profiles/r1_g_*).
struct RowWiper {
    Row32 *z;  // row being wiped
    int idx;   // this lane's next 32-byte index; >= n32 when there is nothing (left) to do
    __device__ __forceinline__ void begin(int *row) {
        z = reinterpret_cast<Row32 *>(row);
        idx = threadIdx.x & 31;
    }
    __device__ __forceinline__ void idle() { idx = 0x3fffffff; }
    // k2 groups of two stores per lane (2 KB per warp and group)
    __device__ __forceinline__ void some(int k2, int n32) {
#pragma unroll 1
        for (int j = 0; j < k2; j++) {
            if (idx + 32 < n32) {
                st_zero32(z + idx);
                st_zero32(z + idx + 32);
            } else if (idx < n32) {
                st_zero32(z + idx);
            }
            idx += 64;
        }
    }
    __device__ __forceinline__ void finish(int n32) {
#pragma unroll 4
        for (; idx < n32; idx += 32) st_zero32(z + idx);
    }
};

struct LaneGroup {  // rates.cuh group interface for one warp
    __device__ __forceinline__ int tid() const { return threadIdx.x & 31; }
    __device__ __forceinline__ int size() const { return 32; }
    __device__ __forceinline__ void sync() const { __syncwarp(); }
};

// CheckLockdown for every deme (:2328-2329 / :449-450 / :736-737): the lanes vote whether any deme crosses a
// threshold; only then lane 0 runs the sequential reference pass and the warp refreshes the contact-density
// dependent rates.  Returns the number of flips.
template <class WSQ>
static __device__ __noinline__ int w_lockdown_slow(const DevState &st, int r, const Dims &D, const WSQ &s, const double *pp,
                                                   double *eff_g, double now) {
    const int lane = threadIdx.x & 31, K = D.K;
    int flips = 0;
    if (lane == 0)
        for (int p = 0; p < K; p++)
            flips += check_lockdown(D, pp, p, (long long)s.tot[p], s.cd, s.lock, now, &st.loc_n[r],
                                    st.loc_sp + (size_t)r * st.loc_cap, st.loc_t + (size_t)r * st.loc_cap, st.loc_cap,
                                    &st.err[r]);
    flips = __shfl_sync(0xffffffffu, flips, 0);
    __syncwarp();
    if (flips) {
        update_contact_rates(LaneGroup(), D, pp, s.cd, eff_g, s.c, s.maxEBM);
        if (s.has_effS) {
            for (int i = lane; i < K * K; i += 32) s.effS[i] = eff_g[i];
            __syncwarp();
        }
    }
    return flips;
}
template <class DIMS, class WSQ>
__device__ __forceinline__ int w_lockdown(const DevState &st, int r, const DIMS &D, const WSQ &s, const double *pp,
                                          double *eff_g, double now) {
    int pred = 0;
#pragma unroll 1
    for (int p = threadIdx.x & 31; p < D.K; p += 32) {
        const double ti = (double)s.tot[p];
        if ((ti > s.startN[p] && s.lock[p] == 0) || (ti < s.endN[p] && s.lock[p] == 1)) pred = 1;
    }
    if (!__any_sync(0xffffffffu, pred)) return 0;
    return w_lockdown_slow(st, r, st.D, s, pp, eff_g, now);  // out of line: the runtime Dims, not a local copy
}

// stage one parameter point (blob layout of common.cuh) into a shared-memory parameter block
template <class DIMS, class WSQ>
__device__ __forceinline__ void w_load_params(const DIMS &D, const WSQ &s, const double *pp, int t, int n) {
    const int K = D.K, H = D.H, S = D.S, U = D.U;
#pragma unroll 1
    for (int i = t; i < H; i += n) {
        s.b[i] = pp[D.o_b + i];
        s.d[i] = pp[D.o_d + i];
        s.sr[i] = pp[D.o_sr + i];
        s.tmq[i] = pp[D.o_tmq + i];
        s.g[i] = (int)pp[D.o_g + i];
    }
    // qin[h][j]: rate of the mutation channel that turns the j-th (ascending) one-substitution neighbour of h into h
    // (mask path only; nbrmask is complete by now)
    if (s.use_masks) {
#pragma unroll 1
        for (int i = t; i < H * U * 3; i += n) {
            const int h = i / (3 * U), j = i - h * 3 * U;
            unsigned long long m = s.nbrmask[h];
            for (int c = 0; c < j; c++) m &= m - 1;
            const int src = __ffsll((long long)m) - 1;
            const int x = src ^ h;
            const int sh = (31 - __clz(x)) & ~1;
            const int u = U - 1 - (sh >> 1);
            const int as = (src >> sh) & 3, hu = (h >> sh) & 3;
            const int k = hu - (hu > as ? 1 : 0);
            s.qin[i] = pp[D.o_q + (src * U + u) * 3 + k];
        }
    }
#pragma unroll 1
    for (int i = t; i < S * H; i += n) {
        s.sigT[i] = pp[D.o_sigT + i];
        s.sb[i] = pp[D.o_sigT + i] * pp[D.o_b + (i % H)];
    }
#pragma unroll 1
    for (int i = t; i < S * S; i += n) s.T[i] = pp[D.o_T + i];
    {  // qmax (the caller zeroed it before its last barrier): non-negative doubles order like their bit patterns
        double m = 0.0;
#pragma unroll 1
        for (int i = t; i < H * U * 3; i += n) m = fmax(m, pp[D.o_q + i]);
        if (m > 0.0) atomicMax(reinterpret_cast<unsigned long long *>(s.qmax.ptr()), (unsigned long long)__double_as_longlong(m));
    }
#pragma unroll 1
    for (int i = t; i < K; i += n) {
        s.sm[i] = pp[D.o_sm + i];
        s.mdiag[i] = pp[D.o_m + i * K + i];
        s.sizeD[i] = pp[D.o_size + i];
        s.startN[i] = pp[D.o_startN + i];
        s.endN[i] = pp[D.o_endN + i];
    }
}

// Ordered compaction of the infectious cells of the CURRENT counts (+ upd when APPLY): act[] ascending, dstart[],
// presence masks / counts, per-deme totals, the ascending list of haplotypes present anywhere.  Returns the
// number of infectious cells; nhap gets the number of present haplotypes.  One warp, ends with __syncwarp().
template <class DIMS, class WSQ, bool APPLY>
__device__ __forceinline__ int w_lists(const DIMS &D, const WSQ &s, int &nhap, RowWiper &wp, int wk, int n32) {
    const int lane = threadIdx.x & 31, K = D.K, H = D.H, KH = K * H;
#pragma unroll 1
    for (int i = lane; i < H; i += 32) s.colcnt[i] = 0;  // (= colmask on the mask path)
#pragma unroll 1
    for (int i = lane; i < K; i += 32) {
        s.tot[i] = 0;
        if (s.use_masks) s.rowmask[i] = 0ull;
    }
    __syncwarp();
    int cnt = 0;
    int *I = s.Iraw;
    if ((H & 31) == 0) {
        // a round of 32 cells lies inside one deme and lane l always meets the haplotypes l, l+32, ...: the presence
        // word of the round is the ballot itself and no two lanes ever touch the same table entry -> no atomics
#pragma unroll 1
        for (int base = 0; base < KH; base += 32) {
            const int i = base + lane;
            int v = I[i];
            if (APPLY) {
                v += s.updI[i];
                I[i] = v;
                wp.some(wk, n32);
            }
            const bool on = v != 0;
            const unsigned m = __ballot_sync(0xffffffffu, on);
            const int p = base >> D.hshift, hb = base & (H - 1);
            if (on) {
                s.act[cnt + __popc(m & ((1u << lane) - 1u))] = (unsigned short)i;
                if (s.use_masks) s.colmask[hb + lane] |= 1 << p;
                else s.colcnt[hb + lane] += 1;
            }
            const int sum = __reduce_add_sync(0xffffffffu, v);
            if (lane == 0) {
                if (hb == 0) s.dstart[p] = cnt;
                s.tot[p] += sum;
                if (s.use_masks) reinterpret_cast<unsigned *>(s.rowmask.ptr() + p)[hb >> 5] = m;
            }
            cnt += __popc(m);
        }
    } else {
#pragma unroll 1
        for (int base = 0; base < KH; base += 32) {
            const int i = base + lane;
            int v = 0;
            if (i < KH) {
                v = I[i];
                if (APPLY) {
                    v += s.updI[i];
                    I[i] = v;
                }
            }
            if (APPLY) wp.some(wk, n32);
            const bool on = v != 0;
            const unsigned m = __ballot_sync(0xffffffffu, on);
            const int pos = cnt + __popc(m & ((1u << lane) - 1u));
            if (i < KH) {
                const int p = i >> D.hshift, h = i & (H - 1);
                if (h == 0) s.dstart[p] = pos;
                if (on) {
                    s.act[pos] = (unsigned short)i;
                    atomicAdd(&s.tot[p], v);
                    if (s.use_masks) {
                        atomicOr(&s.colmask[h], 1 << p);
                        atomicOr(reinterpret_cast<unsigned *>(s.rowmask.ptr() + p) + (h >> 5), 1u << (h & 31));
                    } else {
                        atomicAdd(&s.colcnt[h], 1);
                    }
                }
            }
            cnt += __popc(m);
        }
    }
    if (lane == 0) s.dstart[K] = cnt;
    __syncwarp();
    int nh = 0;
#pragma unroll 1
    for (int base = 0; base < H; base += 32) {
        const int h = base + lane;
        const bool on = h < H && s.colcnt[h] != 0;
        const unsigned m = __ballot_sync(0xffffffffu, on);
        if (on) {
            const int pos = nh + __popc(m & ((1u << lane) - 1u));
            s.hlist[pos] = h;
            s.hidx[h] = (unsigned short)pos;
        }
        nh += __popc(m);
    }
    nhap = nh;
    __syncwarp();
    // per-leap table Q[p, j] for the present haplotypes hlist[j] (the susceptible counts are final for this leap)
    const bool tab = K * nh <= s.qtab_cap;
    if (tab) {
        const int S = D.S;
#pragma unroll 1
        for (int i = lane; i < K * nh; i += 32) {
            const int p = i / nh, h = s.hlist[i - p * nh];
            double Q = 0.0;
#pragma unroll 1
            for (int sn = 0; sn < S; sn++) Q += s.Sx[p * S + sn] * s.sigT[sn * H + h];
            s.qtab[i] = Q;
        }
    }
    if (lane == 0) s.cnt[4] = tab ? nh : 0;
    __syncwarp();
    return cnt;
}

__device__ __forceinline__ double warp_min_d(double v) {
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Drifts and tau (ChooseTau :2432-2450) of the warp's state; same sums as the team kernel's drifts_and_tau.
template <class DIMS, class WSQ>
__device__ __forceinline__ double w_drifts_and_tau(const DIMS &D, const WSQ &s, const double *eff, int nhap, int nAct,
                                                   RowWiper &wp, int wk, int n32) {
    const int K = D.K, H = D.H, S = D.S, KS = K * S;
    const int lane = threadIdx.x & 31;
    // ---- A. pressure / return-flow sums per (deme, group): 8 lanes per sum, fixed butterfly
#pragma unroll 1
    for (int t0 = 0; t0 < KS; t0 += 4) {
        const int task = t0 + (lane >> 3), j = lane & 7;
        double Bv = 0.0, Rv = 0.0;
        int p = 0, sn = 0;
        if (task < KS) {
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
        if (task < KS && j == 0) {
            s.Bp[task] = Bv;
            s.Rp[task] = Rv;
        }
    }
    __syncwarp();
    double tmin = 1.0;
    const float eps = 0.03f;
    auto candidate = [&](double v, double cnt) {
        const double av = fabs(v);
        if (av >= 1e-8) {
            double x = (double)(eps * (float)cnt) / 2.0;  // float product, like the reference's generated C
            x = 1.0 > x ? 1.0 : x;
            if (x < tmin * av) tmin = fmin(tmin, x / av);
        }
    };
    // ---- B1a. cells whose haplotype is present somewhere: force of infection + removal + mutation inflow.
    //           Walks (present haplotype, deme) pairs: every lane has the long sum to do, and neighbouring lanes
    //           share the haplotype, i.e. the trip count of the presence loop.
    const int n1 = K * nhap;
#pragma unroll 1
    for (int i = lane; i < n1; i += 32) {
        const int hi = i / K, p = i - hi * K, h = s.hlist[hi];
        const int cell = p * H + h;
        candidate(drift_I_cell(cell, D, s, eff), s.I[cell]);
    }
    // ---- B1b. cells whose haplotype is present nowhere: count 0, drift = mutation inflow from the <= 3U one-substitution
    //           neighbours present in the deme.  Such a cell proposes tau = 1 / inflow, which undercuts tmin <= 1 only when
    //           inflow > 1, i.e. only when at least one neighbour contributes more than 1 / (3U); a neighbour (p, src)
    //           contributes at most qmax * I[p,src].  So only the neighbours of "big" cells (qmax * I * 3U >= 1) have to be
    //           looked at -- a handful of (cell, neighbour) pairs instead of a pass over all K x H cells; skipping the rest
    //           is exact (their proposal is >= 1 and tau = min(1, ...)).  Pairs reached twice just repeat a candidate.
    // Sparse states (few infectious cells) enumerate; dense ones (measured: from ~1/8 of the cells on) are cheaper with
    // the plain pass over all K x H cells, which is skipped when qmax * (deme prevalence) < 1 in every deme.
    if (nAct * 8 <= K * H) {
        const int U = D.U, n3 = 3 * U;
        const int per = n3 > 0 ? 32 / n3 : 0;  // big cells handled per round
        const double q3 = s.qmax[0] * (double)n3;
        if (per > 0) {
#pragma unroll 1
            for (int base = 0; base < nAct; base += 32) {
                const int a = base + lane;
                const int cell = a < nAct ? (int)s.act[a] : 0;
                const bool big = a < nAct && q3 * s.I[cell] >= 0.999;
                unsigned bm = __ballot_sync(0xffffffffu, big);
#pragma unroll 1
                while (bm) {
                    // this round's big cells: the first `per` set bits
                    const int slot = lane / n3, j = lane - slot * n3;
                    unsigned m = bm;
                    for (int k = 0; k < slot && m; k++) m &= m - 1;
                    const int src_lane = m ? __ffs(m) - 1 : 0;
                    const int bc = __shfl_sync(0xffffffffu, cell, src_lane);
                    if (m && slot < per) {
                        const int p = bc >> D.hshift, h = bc & (H - 1);
                        const int u = j / 3, al = 1 + (j - u * 3);
                        const int hn = h ^ (al << (2 * u));
                        if (s.colcnt[hn] == 0) candidate(drift_I_cell(p * H + hn, D, s, eff), 0.0);
                    }
                    for (int k = 0; k < per && bm; k++) bm &= bm - 1;
                }
            }
        } else if (U > 0) {  // more than 10 sites: one big cell per round, its neighbours strided over the lanes
#pragma unroll 1
            for (int a = 0; a < nAct; a++) {
                const int bc = s.act[a];
                if (!(q3 * s.I[bc] >= 0.999)) continue;
                const int p = bc >> D.hshift, h = bc & (H - 1);
                for (int j = lane; j < n3; j += 32) {
                    const int u = j / 3, al = 1 + (j - u * 3);
                    const int hn = h ^ (al << (2 * u));
                    if (s.colcnt[hn] == 0) candidate(drift_I_cell(p * H + hn, D, s, eff), 0.0);
                }
            }
        }
    } else {
        int need = 0;
#pragma unroll 1
        for (int p = lane; p < K; p += 32) need |= s.qmax[0] * (double)s.tot[p] >= 0.999;
        if (__any_sync(0xffffffffu, need)) {
#pragma unroll 1
            for (int i = lane; i < K * H; i += 32) {
                wp.some(wk, n32);
                if (s.colcnt[i & (H - 1)] != 0) continue;
                candidate(drift_I_cell(i, D, s, eff), 0.0);
            }
        }
    }
    // ---- B2. susceptible drifts
#pragma unroll 1
    for (int i = lane; i < KS; i += 32) candidate(drift_S_cell(i, D, s, eff), s.Sx[i]);
    // ---- C. Mg[p,s] for the out-migration totals of the draws (overwrites Rp, which nobody reads any more)
    __syncwarp();
#pragma unroll 1
    for (int i = lane; i < KS; i += 32) mig_pressure(i, D, s, eff);
    return warp_min_d(tmin);
}

__device__ __forceinline__ int warp_sum32(int v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- draws of the warp kernel ------------------------------------------------------------------------------
// Same draws as the team kernel (same lambda expressions, same Philox addresses, same samplers: a leap stays a pure
// function of state and seed and both kernels leave the same log), organised so that the lanes of a warp stay converged:
//   * every unit of work is a BLOCK of four channels that share one Philox call: block 0 of a cell (RECOVERY, SAMPLING,
//     total of the mutation group, total of the out-migration group), its TRANSMISSION blocks, a deme's SUSCCHANGE
//     blocks, and -- for a group whose total is too large to aggregate -- the blocks of its individual channels;
//   * a draw that the top 32 bits of its uniform do not settle goes to the queue WITH its lambda: (lambda, word,
//     owner | local channel << 20), inversion entries from the bottom, PTRS entries from the top.  Pushes are
//     warp-aggregated (ballot + popcount; the counters are warp-uniform registers, no shared-memory atomics);
//   * the drain runs ONE inlined copy of each sampler over the queue with all lanes busy, then books the counts from
//     the (owner, local channel) pair alone (integer decode, no propensity is recomputed); an aggregated total that
//     came out non-zero is split lane-parallel, one event per lane and iteration.
// ncu of the previous structure (one queue entry per lane through a switch over draw kinds, three call sites per
// sampler, expanded groups drawn channel by channel inside the drain): 34 % of a leap's instructions at t = 60 and
// 67 % at t = 120 ran with 4-7 of 32 lanes active (profiles/r1_n_*, profiles/r2_a_*).
#define TW_L_TOT_MUT 0xFFE
#define TW_L_TOT_MIG 0xFFF
#define TW_XCAP 64

struct DrawState {  // warp-uniform registers of one attempt at a leap
    int ninv, nptr, nxm, nxg, nsq;
};

// Philox domain and word index of the draw (owner, l)
template <class DIMS>
__device__ __forceinline__ void tw_addr(int owner, int l, const DIMS &D, const DrawGeom &g, int &dom, int &q) {
    const int KH = D.K * D.H;
    if (owner >= KH) {  // SUSCCHANGE channel l of a deme
        dom = l >> 2;
        q = l & 3;
    } else if (l >= TW_L_TOT_MUT) {
        dom = 0;
        q = l == TW_L_TOT_MUT ? 2 : 3;
    } else if (l < 2) {
        dom = 0;
        q = l;
    } else if (l < 2 + 3 * D.U) {
        dom = g.NBP + ((l - 2) >> 2);
        q = (l - 2) & 3;
    } else if (l < D.E) {
        const int sn = l - 2 - 3 * D.U;
        dom = 1 + (sn >> 2);
        q = sn & 3;
    } else {
        const int lc = l - D.E;
        dom = g.NBP + g.nbm + (lc >> 2);
        q = lc & 3;
    }
}

// where the n events of channel (owner, l) go (cell_channel / susc_channel without the propensity) + the row index
template <class DIMS, class WSQ>
__device__ __forceinline__ int tw_channel_ids(int owner, int l, const DIMS &D, const WSQ &s, const WarpLayout &L, Channel &ch) {
    const int K = D.K, H = D.H, S = D.S, KH = K * H;
    ch.i_dec = ch.i_inc = ch.i_chk = ch.s_dec = ch.s_inc = -1;
    ch.prop = 0.0;
    if (owner >= KH) {
        const int p = owner - KH;
        const int ss = fdiv(l, L.mS1, S - 1), tsp = l - ss * (S - 1);
        const int ts = tsp + (tsp >= ss ? 1 : 0);
        ch.type = EV_SUSCCHANGE;
        ch.s_dec = p * S + ss;
        ch.s_inc = p * S + ts;
        return D.NA + p * D.PD + l;
    }
    const int p = owner >> D.hshift, h = owner & (H - 1);
    if (l < D.E) {
        if (l < 2) {
            ch.type = l == 0 ? EV_DEATH : EV_SAMPLING;
            ch.i_dec = owner;
            ch.s_inc = p * S + s.g[h];
        } else if (l < 2 + 3 * D.U) {
            const int uk = l - 2, u = uk / 3, k = uk - u * 3;
            ch.type = EV_MUTATION;
            ch.i_dec = owner;
            ch.i_inc = ch.i_chk = p * H + mutate_hap(h, u, k, D.U);
        } else {
            ch.type = EV_BIRTH;
            ch.i_inc = ch.i_chk = owner;
            ch.s_dec = p * S + (l - 2 - 3 * D.U);
        }
        return D.NA + p * D.PD + D.SS1 + h * D.E + l;
    }
    const int mm = l - D.E;
    const int tpp = fdiv(mm, L.mS, S), sn = mm - tpp * S;
    const int tp = tpp + (tpp >= p ? 1 : 0);
    ch.type = EV_MIGRATION;
    ch.i_inc = tp * H + h;
    ch.i_chk = owner;
    ch.s_dec = tp * S + sn;
    return ((p * (K - 1) + tpp) * S + sn) * H + h;
}

// One event of the multinomial split of an aggregated total (split_total_impl of the team kernel, one event):
// event e of the total of cell `owner` (kind 2: mutation group, 3: out-migration group) picks its channel with the
// e-th 53-bit uniform of the group's split domain.  Returns the local channel or -1.
template <class DIMS, class WSQ>
__device__ __forceinline__ int tw_split_event(int owner, int kind, int e, const DIMS &D, const WSQ &s, const double *eff,
                                              const DrawGeom &g, PhiloxCtx &ctx) {
    const int K = D.K, H = D.H, S = D.S, U = D.U;
    const int p = owner >> D.hshift, h = owner & (H - 1);
    const double Ii = s.I[owner];
    ctx.c0 = (uint32_t)owner;
    ctx.dom0 = (uint32_t)(g.NBP + g.nbm + g.nbg + (kind == 2 ? 0 : 1));
    const uint4 w = ctx.draw((uint32_t)(e >> 1));
    const double u = (e & 1) ? u53(w.z, w.w) : u53(w.x, w.y);
    int l = -1;
    if (kind == 2) {
        const double x = u * (s.tmq[h] * Ii);
        double acc = 0.0;
#pragma unroll 1
        for (int uk = 0; uk < 3 * U; uk++) {
            const double pr = s.q[h * U * 3 + uk] * Ii;
            if (pr > 0.0) {
                l = 2 + uk;
                acc += pr;
                if (x < acc) break;
            }
        }
    } else {
        l = split_migration(p, h, u, D, s, eff);
    }
    return l;
}

// One round (<= 32, taken from the end of the list) of parked aggregated totals: every lane splits one total, one event
// per iteration.
template <class DIMS, class WSQ>
__device__ __forceinline__ void w_split_parked(int *row, const DIMS &D, const WSQ &s, const double *eff, const DrawGeom &g,
                                               const WarpLayout &L, PhiloxCtx &ctx, LeapTally &tr, DrawState &q) {
    const int lane = threadIdx.x & 31;
    const int take = q.nsq < 32 ? q.nsq : 32;
    const int e = q.nsq - take + lane;
    const bool valid = lane < take;
    const unsigned pw = valid ? (unsigned)s.sqp[e] : 0u;
    const int owner = (int)(pw & 0xfffffu), kind = (pw >> 20) & 1u ? 3 : 2, ns = (int)(pw >> 21);
#pragma unroll 1
    for (int ev = 0; __any_sync(0xffffffffu, ev < ns); ev++) {
        if (ev < ns) {
            const int ls = tw_split_event(owner, kind, ev, D, s, eff, g, ctx);
            if (ls >= 0) {
                Channel ch;
                const int c = tw_channel_ids(owner, ls, D, s, L, ch);
                atomicAdd(&row[c], 1);
                book(ch, 1, s, tr);
            }
        }
    }
    q.nsq -= take;
    __syncwarp();
}

// Finish every queued draw and book the counts; all lanes walk the same code.
//   * inversion entries in rounds of 32.  A channel's count is booked at once; an aggregated total that came out
//     non-zero is parked as a (owner | kind, n) pair, and the pairs are split 32 at a time -- as soon as 32 are there,
//     and the rest when the leap's last drain runs (`final`) -- so that the split walks run with the lanes full
//     (they ran with 1.5 of 32 lanes when every drain split its own few totals, ncu profiles/r2_c_*);
//   * PTRS entries in rounds of 32, one inlined copy of the sampler.
#define TW_SQCAP 64
template <class DIMS, class WSQ>
__device__ __forceinline__ void w_drain(int *row, const DIMS &D, const WSQ &s, const double *eff, const DrawGeom &g,
                                        const WarpLayout &L, PhiloxCtx &ctx, LeapTally &tr, DrawState &q, bool final) {
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    __syncwarp();
    // ---- inversion entries: channels with lambda < 10 and aggregated totals
#pragma unroll 1
    for (int k0 = 0;; k0 += 32) {
        const bool more = k0 < q.ninv;
        if (more) {
            const int k = k0 + lane;
            const bool valid = k < q.ninv;
            const double lam = valid ? s.qlam[k] : 0.0;
            const uint32_t hi = valid ? (uint32_t)s.qhi[k] : 0u;
            const unsigned oc = valid ? (unsigned)s.qoc[k] : 0u;
            const int owner = (int)(oc & 0xfffffu), l = (int)(oc >> 20);
            int dom, qq;
            tw_addr(owner, l, D, g, dom, qq);
            int n = 0;
            if (valid) {
                ctx.c0 = (uint32_t)owner;
                ctx.dom0 = (uint32_t)dom;
                n = (int)poisson_inversion_impl(lam, hi, ctx, qq);
            }
            const bool tot = l >= TW_L_TOT_MUT;
            if (n != 0 && !tot) {
                Channel ch;
                const int c = tw_channel_ids(owner, l, D, s, L, ch);
                row[c] = n;
                book(ch, n, s, tr);
            }
            const bool park = tot && n != 0;
            const unsigned pm = __ballot_sync(0xffffffffu, park);
            if (park) {  // one word: owner | kind << 20 | n << 21 (n < 256: the inversion sampler's cap)
                const int e = q.nsq + __popc(pm & lt);
                s.sqp[e] = (int)((unsigned)owner | (l == TW_L_TOT_MIG ? 1u << 20 : 0u) | ((unsigned)n << 21));
            }
            q.nsq += __popc(pm);
            __syncwarp();
        }
        // split one round of parked totals (taken from the end of the list)
        if (q.nsq >= 32 || (!more && final && q.nsq > 0)) w_split_parked(row, D, s, eff, g, L, ctx, tr, q);
        if (!more && !(final && q.nsq > 0)) break;
    }
    // ---- PTRS entries (lambda >= 10) sit at the top of the queue.  (A two-pass variant -- trial 0 with the quick
    //      acceptance test for everybody, then the complete sampler for the compacted rest -- measured SLOWER: 15.8 vs
    //      13.8 ms at t = 90, gpurun r2_e: the second pass repeats trial 0 and the queue traffic outweighs the lanes won.)
#pragma unroll 1
    for (int k0 = 0; k0 < q.nptr; k0 += 32) {
        const int k = k0 + lane;
        const bool valid = k < q.nptr;
        const int e = s.qcap - 1 - k;
        const double lam = valid ? s.qlam[e] : 100.0;
        const unsigned oc = valid ? (unsigned)s.qoc[e] : 0u;
        const int owner = (int)(oc & 0xfffffu), l = (int)(oc >> 20);
        int dom, qq;
        tw_addr(owner, l, D, g, dom, qq);
        if (valid) {
            ctx.c0 = (uint32_t)owner;
            ctx.dom0 = (uint32_t)dom;
            const int n = (int)poisson_ptrs_impl(lam, ctx, qq);
            if (n != 0) {
                Channel ch;
                const int c = tw_channel_ids(owner, l, D, s, L, ch);
                row[c] = n;
                book(ch, n, s, tr);
            }
        }
    }
    q.ninv = q.nptr = 0;
    __syncwarp();
}

struct RoundOut {  // what a lane's block leaves for the queue
    double lam[4];
    uint4 w4;
    unsigned mi[4], mp[4];  // per word: lanes that push an inversion / a PTRS entry
    int need[2];            // queue entries of words 0-1 / words 2-3 (each <= 64: a half always fits an empty queue)
    int owner, lb;          // local channel of word w = lb + w; lb < 0: block 0 of a cell (0, 1, the two totals)
};

// One round of 32 block items: lambdas, the Philox block, early-outs; returns the number of queue entries the round
// needs (w_push stores them).  mode 0: the primary item space [cells: block 0 | cells x transmission blocks | demes x
// SUSCCHANGE blocks]; mode 1: the blocks of the groups listed in the expansion queues [mutation | out-migration].
template <class DIMS, class WSQ>
__device__ __forceinline__ int w_round(int item, int mode, int nAct, double tau, int variant, const DIMS &D, const WSQ &s,
                                       const double *eff, const DrawGeom &g, const WarpLayout &L, PhiloxCtx &ctx,
                                       DrawState &q, RoundOut &ro) {
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    const int K = D.K, H = D.H, S = D.S, U = D.U, KH = K * H;
    const int NBT = g.NB1 - 1;
    double lam[4] = {0.0, 0.0, 0.0, 0.0};
    int owner = 0, dom = 0, lb = 0;  // local channel of word w = lb + w (block 0 of a cell: 0, 1, the two totals)
    int kind = -1;
    if (mode == 0) {
        const int nB = nAct * NBT;
        if (item < nAct) {
            kind = 0;
            owner = s.act[item];
            const int p = owner >> D.hshift, h = owner & (H - 1);
            const double Ii = s.I[owner];
            lam[0] = s.d[h] * Ii * tau;
            lam[1] = s.sr[h] * Ii * s.sm[p] * tau;
            lam[2] = s.tmq[h] * Ii * tau;
            lam[3] = K > 1 ? mig_total(p, h, Ii, D, s, eff) * tau : 0.0;
        } else if (item < nAct + nB) {
            kind = 1;
            const int it2 = item - nAct;
            const int ai = fdiv(it2, L.mNBT, NBT), j = it2 - ai * NBT;
            owner = s.act[ai];
            const int p = owner >> D.hshift, h = owner & (H - 1);
            const double Ii = s.I[owner];
            dom = 1 + j;
            lb = 2 + 3 * U + j * 4;
#pragma unroll
            for (int w = 0; w < 4; w++) {
                const int sn = j * 4 + w;
                if (sn < S) lam[w] = s.b[h] * s.sigT[sn * H + h] * s.c[p] * s.Sx[p * S + sn] * Ii * tau;
            }
        } else if (item < nAct + nB + K * g.G2) {
            kind = 2;
            const int it = item - nAct - nB;
            const int p = fdiv(it, L.mG2, g.G2), j = it - p * g.G2;
            owner = KH + p;
            dom = j;
            lb = j * 4;
#pragma unroll
            for (int w = 0; w < 4; w++) {
                const int l = j * 4 + w;
                if (l < D.SS1) {
                    const int ss = fdiv(l, L.mS1, S - 1), tsp = l - ss * (S - 1);
                    const int ts = tsp + (tsp >= ss ? 1 : 0);
                    lam[w] = s.T[ss * S + ts] * s.Sx[p * S + ss] * tau;
                }
            }
        }
    } else {
        const int itM = q.nxm * g.nbm;
        if (item < itM) {
            kind = 3;
            const int xi = fdiv(item, L.mnbm, g.nbm), j = item - xi * g.nbm;
            owner = s.xq[xi];
            const int h = owner & (H - 1);
            const double Ii = s.I[owner];
            dom = g.NBP + j;
            lb = 2 + j * 4;
#pragma unroll
            for (int w = 0; w < 4; w++) {
                const int uk = j * 4 + w;
                if (uk < 3 * U) lam[w] = s.q[h * U * 3 + uk] * Ii * tau;
            }
        } else if (item < itM + q.nxg * g.nbg) {
            kind = 4;
            const int it2 = item - itM;
            const int xi = fdiv(it2, L.mnbg, g.nbg), j = it2 - xi * g.nbg;
            owner = s.xq[TW_XCAP + xi];
            const int p = owner >> D.hshift, h = owner & (H - 1);
            const double Ii = s.I[owner];
            dom = g.NBP + g.nbm + j;
            lb = D.E + j * 4;
#pragma unroll
            for (int w = 0; w < 4; w++) {
                const int lc = j * 4 + w;
                if (lc < (K - 1) * S && Ii != 0.0) {
                    const int tpp = fdiv(lc, L.mS, S), sn = lc - tpp * S;
                    const int tp = tpp + (tpp >= p ? 1 : 0);
                    lam[w] = eff[tp * K + p] * s.Sx[tp * S + sn] * Ii * s.b[h] * s.sigT[sn * H + h] * s.mdiag[p] * tau;
                }
            }
        }
    }
    // groups too large to aggregate: list the cell, its channels are drawn block by block in mode 1
    {
        const bool xm = kind == 0 && lam[2] > 0.0 && ((variant & 1) || lam[2] > TAU_THETA_MUT);
        const bool xg = kind == 0 && lam[3] > 0.0 && ((variant & 1) || lam[3] > TAU_THETA_MIG);
        const unsigned bm = __ballot_sync(0xffffffffu, xm), bg = __ballot_sync(0xffffffffu, xg);
        if (xm) {
            s.xq[q.nxm + __popc(bm & lt)] = (unsigned short)owner;
            lam[2] = 0.0;
        }
        if (xg) {
            s.xq[TW_XCAP + q.nxg + __popc(bg & lt)] = (unsigned short)owner;
            lam[3] = 0.0;
        }
        q.nxm += __popc(bm);
        q.nxg += __popc(bg);
    }
    ro.w4 = make_uint4(0, 0, 0, 0);
    if (lam[0] > 0.0 || lam[1] > 0.0 || lam[2] > 0.0 || lam[3] > 0.0) {
        ctx.c0 = (uint32_t)owner;
        ctx.dom0 = (uint32_t)dom;
        ro.w4 = ctx.draw(0u);
    }
    ro.owner = owner;
    ro.lb = kind == 0 ? -1 : lb;
    ro.need[0] = ro.need[1] = 0;
#pragma unroll
    for (int w = 0; w < 4; w++) {
        const uint32_t hi = w == 0 ? ro.w4.x : w == 1 ? ro.w4.y : w == 2 ? ro.w4.z : ro.w4.w;
        const double lm = lam[w];
        ro.lam[w] = lm;
        // U = (hi + f)/2^32 with f in [0,1).  (hi+1)/2^32 <= 1 - lam  =>  U < 1-lam <= exp(-lam)  =>  0
        const bool inv = lm > 0.0 && lm < 10.0 && !((double)hi + 1.0 <= (1.0 - lm) * 4294967296.0);
        const bool ptr = lm >= 10.0;
        ro.mi[w] = __ballot_sync(0xffffffffu, inv);
        ro.mp[w] = __ballot_sync(0xffffffffu, ptr);
        ro.need[w >> 1] += __popc(ro.mi[w]) + __popc(ro.mp[w]);
    }
    return ro.need[0] + ro.need[1];
}

// store the unsettled draws of words [W0, W1) of the round (the caller has made room): inversion entries from the
// bottom, PTRS from the top
template <int W0, int W1, class WSQ>
__device__ __forceinline__ void w_push(const RoundOut &ro, const WSQ &s, DrawState &q) {
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u, me = 1u << lane;
#pragma unroll
    for (int w = W0; w < W1; w++) {
        const bool inv = (ro.mi[w] & me) != 0, ptr = (ro.mp[w] & me) != 0;
        if (inv || ptr) {
            const uint32_t hi = w == 0 ? ro.w4.x : w == 1 ? ro.w4.y : w == 2 ? ro.w4.z : ro.w4.w;
            const int e = inv ? q.ninv + __popc(ro.mi[w] & lt) : s.qcap - 1 - (q.nptr + __popc(ro.mp[w] & lt));
            const int l = (ro.lb < 0) ? (w < 2 ? w : w == 2 ? TW_L_TOT_MUT : TW_L_TOT_MIG) : ro.lb + w;
            s.qlam[e] = ro.lam[w];
            s.qhi[e] = (int)hi;
            s.qoc[e] = (int)((unsigned)ro.owner | ((unsigned)l << 20));
        }
        q.ninv += __popc(ro.mi[w]);
        q.nptr += __popc(ro.mp[w]);
    }
}

// ---- size-sorted schedule -----------------------------------------------------------------------------
// With lockstep generations a leap costs every warp of the CTA as much as it costs the slowest one, and a
// leap's cost grows with the number of infectious cells of the replicate.  So replicates of similar size share
// a CTA: weight = #infectious cells, sorted descending, consecutive groups of `nwarps` go to one CTA visit, and
// the CTAs walk the groups boustrophedon (b, 2G-1-b, 2G+b, ...) so that every CTA gets the same mix of heavy and
// light groups.  (KH below is the largest possible weight.)  Scheduling only: every replicate's result is a function of its own state and seed.
__global__ void tau_weight_kernel(const DevState st, int *weight) {
    const int lane = threadIdx.x & 31, KH = st.D.K * st.D.H;
    const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= st.R) return;
    int n = 0;
    for (int i = lane; i < KH; i += 32) n += st.I[(size_t)r * KH + i] != 0;
    n = __reduce_add_sync(0xffffffffu, n);
    if (lane == 0) weight[r] = n;
}
// one CTA: counting sort by weight (descending) into order[]
__global__ void __launch_bounds__(1024) tau_order_kernel(int R, int KH, const int *weight, int *order) {
    __shared__ int bins[2049];
    const int NB = 2048;
    for (int i = threadIdx.x; i <= NB; i += blockDim.x) bins[i] = 0;
    __syncthreads();
    for (int r = threadIdx.x; r < R; r += blockDim.x) {
        const int b = NB - 1 - (int)(((long long)weight[r] * (NB - 1)) / (KH > 0 ? KH : 1));  // heavy first
        atomicAdd(&bins[b + 1], 1);
    }
    __syncthreads();
    if (threadIdx.x == 0)
        for (int i = 0; i < NB; i++) bins[i + 1] += bins[i];
    __syncthreads();
    for (int r = threadIdx.x; r < R; r += blockDim.x) {
        const int b = NB - 1 - (int)(((long long)weight[r] * (NB - 1)) / (KH > 0 ? KH : 1));
        order[atomicAdd(&bins[b], 1)] = r;
    }
}

template <class DIMS, bool PROF, bool EFFS, bool MASKS>
__global__ void __launch_bounds__(TW_MAX_WARPS * 32, 1)
    tau_warp_kernel(const __grid_constant__ DevState st, const __grid_constant__ SimArgs a,
                    const __grid_constant__ WarpLayout L, const __grid_constant__ WSX<MASKS> s, const int variant,
                    const int *__restrict__ order) {
    typename DimsRef<DIMS>::type D = st.D;
    const int K = D.K, H = D.H, S = D.S, KH = K * H, KS = K * S;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const DrawGeom g = draw_geom(D);
    const int n32 = D.Pp >> 3;  // 256-bit stores per log row
    // groups of 2 stores per lane per dense-loop round so that three dense loops (drift, feasibility, apply) cover a row
    const int wk = (((n32 + 31) / 32 + 3 * ((KH + 31) / 32) - 1) / (3 * ((KH + 31) / 32)) + 1) / 2;  // in groups of 2
    const bool prof = PROF;
    unsigned long long pc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long tmark = 0;
#define TW_MARK(k)                                    \
    if (prof && lane == 0) {                          \
        const long long now_ = clock64();             \
        pc[k] += (unsigned long long)(now_ - tmark);  \
        tmark = now_;                                 \
    }

    // Optional lockstep ("generations"): with a bit of `gsync` set every warp of the CTA meets at a CTA-wide barrier
    // at that point of every leap (1: leap start, 2: before the draws, 4: before the apply pass), so the warps of
    // an SM walk the same phase at the same time and share its instruction fetch.  A warp that ran out of
    // replicates keeps answering the barriers until all are done (see the end of the kernel).
    const int gsync = L.gsync;
    int gen = 0;  // leaps this warp has walked; it joins the barriers of every gevery-th one
    const int gsz = (L.ggroup > 0 && L.ggroup < nw && (nw + L.ggroup - 1) / L.ggroup <= 15) ? L.ggroup : nw;
    const int grp = wid / gsz;
    const int gmembers = (nw - grp * gsz < gsz) ? nw - grp * gsz : gsz;  // warps in this warp's group
#define TW_GEN_SYNC() asm volatile("bar.sync %0, %1;" ::"r"(1 + grp), "r"(gmembers * 32) : "memory")
    int *done_warps = reinterpret_cast<int *>(smem_raw + L.o_done) + grp;
    if (threadIdx.x < 16) reinterpret_cast<int *>(smem_raw + L.o_done)[threadIdx.x] = 0;
    // ---- CTA prologue: neighbour masks, the shared parameter point
    if (s.use_masks)
#pragma unroll 1
        for (int i = threadIdx.x; i < H; i += blockDim.x) {
            unsigned long long m = 0ull;
            for (int u = 0; u < D.U; u++)
                for (int al = 1; al < 4; al++) m |= 1ull << (i ^ (al << (2 * u)));
            s.nbrmask[i] = m;
        }
    if (L.par_shared && threadIdx.x == 0) s.qmax[0] = 0.0;
    __syncthreads();  // nbrmask is read by the parameter staging
    if (L.par_shared) w_load_params(D, s, st.params + (size_t)L.pp0 * D.blob, threadIdx.x, blockDim.x);
    __syncthreads();

    for (int visit = 0;; visit++) {
        int r;
        if (order) {  // boustrophedon walk over the size-sorted groups
            const int G = gridDim.x;
            const int grp = (visit & 1) ? (visit + 1) * G - 1 - (int)blockIdx.x : visit * G + (int)blockIdx.x;
            if ((long long)(visit & ~1) * G * nw >= st.R) break;  // both groups of this pair of visits are past the end
            const int pos = grp * nw + wid;
            if (pos >= st.R) continue;
            r = order[pos];
        } else {
            r = (visit * (int)gridDim.x + (int)blockIdx.x) * nw + wid;
            if (r >= st.R) break;
        }
        const double *pp = st.params + (size_t)st.rep_pp[r] * D.blob;
        double *eff_g = st.eff + (size_t)r * K * K;
        long long *ctr = st.counters + (size_t)r * NCOUNT;
        const uint64_t seed = st.seeds[r];
        if (lane == 0) s.tally64[6] = (long long)seed;  // reread once per leap instead of living in two registers
        if (!L.par_shared && lane == 0) s.qmax[0] = 0.0;
        __syncwarp();
        // ---- load the replicate
        if (!L.par_shared) w_load_params(D, s, pp, lane, 32);
#pragma unroll 1
        for (int i = lane; i < K; i += 32) {
            s.cd[i] = st.cd[(size_t)r * K + i];
            s.c[i] = st.ceff[(size_t)r * K + i];
            s.maxEBM[i] = st.maxEBM[(size_t)r * K + i];
            s.lock[i] = st.lock[(size_t)r * K + i];
        }
        if (EFFS)
#pragma unroll 1
            for (int i = lane; i < K * K; i += 32) s.effS[i] = eff_g[i];
        int ovf = 0;
#pragma unroll 1
        for (int i = lane; i < KH; i += 32) {
            const long long v = st.I[(size_t)r * KH + i];
            if (v > 2147483647LL || v < 0) ovf = 1;
            s.Iraw[i] = (int)v;
        }
#pragma unroll 1
        for (int i = lane; i < K; i += 32)
            if (s.sizeD[i] > 2147483647.0) ovf = 1;  // counts are held as int32 and bounded by the deme size
#pragma unroll 1
        for (int i = lane; i < KS; i += 32) {
            const long long v = st.Sx[(size_t)r * KS + i];
            if (v > 2147483647LL || v < 0) ovf = 1;
            s.Sx[i] = (double)v;
        }
        if (lane < 8) s.cnt[lane] = 0;
        __syncwarp();
        if (__any_sync(0xffffffffu, ovf)) {
            if (lane == 0) st.err[r] |= ERR_COUNT_OVERFLOW;
            continue;
        }
        // EFFS (K <= 32): the effective-migration matrix sits in the warp slice -- a compile-time choice so that the
        // pointer keeps its shared-memory address space (LDS, 32-bit addresses) through the inlined helpers
        const double *eff = EFFS ? (const double *)s.effS.ptr() : (const double *)eff_g;
        int nhap = 0;
        RowWiper wp;
        wp.idle();
        int pre_row = -1;  // leap whose row the wiper is working on / has finished
        int nAct = w_lists<DIMS, WSX<MASKS>, false>(D, s, nhap, wp, 0, n32);

        bool restarted = false;
        if (lane < 6) s.tally64[lane] = 0;
        if (lane == 7) s.tally64[7] = (long long)(uintptr_t)pp;
        int flips_total = 0;
        long long sC = ctr[C_S];
        long long evptr = ctr[C_EVPTR], leaps = ctr[C_LEAPS];
        double t = st.time[r];
        unsigned epoch = st.epoch[r];
        long long good_attempt = ctr[C_GOOD];
        const long long ev_limit = evptr + a.iterations;
        long long dbase = st.dense_base[r];  // leaps whose rows went to the archive: leap L is dense row L - dbase
        int *tau_counts = st.tau_counts + (size_t)r * st.dense_cap * D.Pp;

        for (long long attempt = 0; attempt < a.attempts; attempt++) {
            if (!(a.cont && attempt == 0)) epoch++;
            if (nAct != 0) {
                while (evptr < ev_limit && evptr < st.ev_cap && leaps < st.leap_cap && leaps - dbase < st.dense_cap &&
                       (a.sample_size == -1 || sC < a.sample_size) && (!a.has_time || t < (double)a.time)) {
                    int *row = tau_counts + (size_t)(leaps - dbase) * D.Pp;
                    const bool meet = gsync && (L.gevery <= 1 || gen % L.gevery == 0);
                    gen++;
                    if (meet) {
                        TW_GEN_SYNC();
                        if (gsync == 1) TW_GEN_SYNC();  // the end-of-kernel protocol needs two barriers per generation
                    }
                    if (prof && lane == 0) tmark = clock64();
                    // ---- 0. this leap's row: finish the wipe started during the previous leap (or do all of it: first
                    //         leap of the call, Restart), then start on the next row; 1-2. drifts and tau
                    if (pre_row != (int)leaps) wp.begin(row);
                    wp.finish(n32);
                    if (leaps + 1 < st.leap_cap && leaps + 1 - dbase < st.dense_cap && evptr + 1 < ev_limit && evptr + 1 < st.ev_cap) {
                        wp.begin(row + D.Pp);
                        pre_row = (int)leaps + 1;
                    } else {
                        wp.idle();
                        pre_row = -1;
                    }
                    double tau = w_drifts_and_tau(D, s, eff, nhap, nAct, wp, wk, n32);
                    TW_MARK(1)
                    if (meet && (gsync & 2)) TW_GEN_SYNC();
                    if (prof && lane == 0) tmark = clock64();
                    // ---- 3. draw; halve tau and redraw on an infeasible leap (:2316-2321)
                    int tB = 0, tD = 0, tS = 0, tM = 0, tI = 0, tG = 0;
                    for (unsigned retry = 0;; retry++) {
                        // clear the per-leap deltas (chk and upd are adjacent)
                        {
                            int4 *z = reinterpret_cast<int4 *>(s.chkI.ptr());
                            const int n16 = (int)((s.updI.off - s.chkI.off) + KH * 4 + 15) >> 4;
#pragma unroll 1
                            for (int i = lane; i < n16; i += 32) {
                                z[i] = make_int4(0, 0, 0, 0);
                                wp.some(1, n32);
                            }
#pragma unroll 1
                            for (int i = lane; i < KS; i += 32) s.dSx[i] = 0;
                        }
                        __syncwarp();
                        LeapTally tr;
                        tr.B = tr.Dd = tr.Sm = tr.M = tr.I = tr.G = 0;
                        PhiloxCtx ctx;
                        {
                            const unsigned long long sd = (unsigned long long)s.tally64[6];
                            ctx.key = make_uint2((uint32_t)sd, (uint32_t)(sd >> 32));
                        }
                        ctx.c1 = (uint32_t)leaps;
                        ctx.c2 = (retry & 0xffu) | (epoch << 8);
                        ctx.dstride = (uint32_t)g.GS;
                        // One loop, one call site per helper (the leap loop has to stay small: the SM's instruction cache is
                        // shared by 14 warps): primary rounds; whenever an expansion queue could overflow -- and once more
                        // after the last primary round -- the rounds over the listed groups' channel blocks; a drain
                        // whenever the next round could overflow the slow-path queue and after the last round.
                        const int nItems = nAct * g.NB1 + K * g.G2;
                        DrawState dq;
                        dq.ninv = dq.nptr = dq.nxm = dq.nxg = dq.nsq = 0;
                        int pbase = 0, xbase = 0, xlimit = 0;
                        bool flush = false;  // the iteration after the last round only drains
#pragma unroll 1
                        for (;;) {
                            const bool inx = xbase < xlimit;
                            RoundOut ro;
                            int pushes = 0;
                            if (!flush)
                                pushes = w_round((inx ? xbase : pbase) + lane, inx ? 1 : 0, nAct, tau, variant, D, s, eff, g, L, ctx, dq, ro);
                            if (flush || dq.ninv + dq.nptr + pushes > s.qcap) w_drain(row, D, s, eff, g, L, ctx, tr, dq, flush);
                            if (flush) break;
                            if (pushes <= s.qcap) {
                                w_push<0, 4>(ro, s, dq);
                            } else {
                                // (cold) a round can leave up to 128 entries, the queue holds 96: two halves of <= 64 with a
                                // drain in between.  Needs > 3 unsettled draws per lane on average -- dense states only.
                                w_push<0, 2>(ro, s, dq);
                                w_drain(row, D, s, eff, g, L, ctx, tr, dq, false);
                                w_push<2, 4>(ro, s, dq);
                            }
                            if (flush) break;
                            if (inx) {
                                xbase += 32;
                                if (xbase >= xlimit) {
                                    dq.nxm = dq.nxg = 0;
                                    xbase = xlimit = 0;
                                    __syncwarp();  // every lane has read the lists before the next round refills them
                                }
                            } else {
                                pbase += 32;
                            }
                            const bool primary_done = pbase >= nItems;
                            if (xlimit == 0 && (dq.nxm + 32 > TW_XCAP || dq.nxg + 32 > TW_XCAP || (primary_done && (dq.nxm | dq.nxg)))) {
                                xlimit = dq.nxm * g.nbm + dq.nxg * g.nbg;
                                __syncwarp();      // the lists are complete before the rounds that read them
                            }
                            flush = primary_done && xlimit == 0;
                        }
                        TW_MARK(2)
                        // ---- 4. feasibility (:2522-2528, quirk Q8) -- see the team kernel for the extra state test
                        int bad = 0;
#pragma unroll 1
                        for (int i = lane; i < KH; i += 32) {
                            wp.some(1, n32);
                            const double sz = s.sizeD[i >> D.hshift];
                            const double Iv = s.I[i];
                            const double v = Iv + (double)s.chkI[i];
                            const double u = Iv + (double)s.updI[i];
                            if (v < 0.0 || v > sz || u < 0.0 || u > sz) bad = 1;
                        }
#pragma unroll 1
                        for (int i = lane; i < KS; i += 32) {
                            const double v = s.Sx[i] + (double)s.dSx[i];
                            if (v < 0.0 || v > s.sizeD[i / S]) bad = 1;
                        }
                        bad = __any_sync(0xffffffffu, bad);
                        tB = __reduce_add_sync(0xffffffffu, tr.B); tD = __reduce_add_sync(0xffffffffu, tr.Dd);
                        tS = __reduce_add_sync(0xffffffffu, tr.Sm); tM = __reduce_add_sync(0xffffffffu, tr.M);
                        tI = __reduce_add_sync(0xffffffffu, tr.I); tG = __reduce_add_sync(0xffffffffu, tr.G);
                        TW_MARK(3)
                        if (!bad) break;
                        tau *= 0.5;
                        w_wipe_row(row, D.Pp >> 3);  // rare path
                        if (retry >= 80) {  // tau * 2^-80: nothing can fire any more, yet the state fails the test
                            if (lane == 0) st.err[r] |= ERR_TAU_STUCK;
                            tau = 0.0;
                            tB = tD = tS = tM = tI = tG = 0;
                            {
                                int4 *z = reinterpret_cast<int4 *>(s.chkI.ptr());
                                const int n16 = (int)((s.updI.off - s.chkI.off) + KH * 4 + 15) >> 4;
#pragma unroll 1
                                for (int i = lane; i < n16; i += 32) z[i] = make_int4(0, 0, 0, 0);
#pragma unroll 1
                                for (int i = lane; i < KS; i += 32) s.dSx[i] = 0;
                            }
                            __syncwarp();
                            break;
                        }
                    }
                    if (meet && (gsync & 4)) TW_GEN_SYNC();
                    if (prof && lane == 0) tmark = clock64();
                    t += tau;
                    sC += tS;
                    if (lane == 0) {
                        long long *ty = s.tally64;
                        ty[EV_BIRTH] += tB; ty[EV_DEATH] += tD; ty[EV_SAMPLING] += tS;
                        ty[EV_MUTATION] += tM; ty[EV_SUSCCHANGE] += tI; ty[EV_MIGRATION] += tG;
                    }
                    // ---- 5. apply (UpdateCompartmentCounts_tau, :2536-2593) fused with the list rebuild
#pragma unroll 1
                    for (int i = lane; i < KS; i += 32) s.Sx[i] += (double)s.dSx[i];
                    nAct = w_lists<DIMS, WSX<MASKS>, true>(D, s, nhap, wp, 1, n32);
                    if (lane == 0) {
                        double *tau_tt = st.tau_tt + ((size_t)r * st.leap_cap + leaps) * 2;
                        tau_tt[0] = t;
                        tau_tt[1] = tau;
                        st.ev_time[(size_t)r * st.ev_cap + evptr] = t;
                        st.ev_desc[(size_t)r * st.ev_cap + evptr] = pack_multi((uint32_t)leaps);
                    }
                    leaps++;
                    evptr++;
                    TW_MARK(4)
                    if (prof && lane == 0) pc[7] += 1;
                    // ---- extinction test and CheckLockdown for every deme (:2326-2329)
                    if (nAct == 0) break;
                    flips_total += w_lockdown(st, r, D, s, pp, eff_g, t);
                }
            }
            // ---- extinction-retry (:2331-2335): <= 100 log rows with iterations > 100 => Restart (:714-738)
            if (evptr + st.ev_base[r] <= 100 && a.iterations > 100) {
                evptr = 0;
                leaps = 0;
                sC = 0;
                t = 0.0;
                restarted = true;
                if (lane < 6) s.tally64[lane] = 0;
                __syncwarp();
#pragma unroll 1
                for (int i = lane; i < KH; i += 32) s.Iraw[i] = (int)st.initI[(size_t)r * KH + i];
#pragma unroll 1
                for (int i = lane; i < KS; i += 32) s.Sx[i] = (double)st.initSx[(size_t)r * KS + i];
                __syncwarp();
                nAct = w_lists<DIMS, WSX<MASKS>, false>(D, s, nhap, wp, 0, n32);
                flips_total += w_lockdown(st, r, D, s, pp, eff_g, t);
                good_attempt = 0;
                dbase = 0;  // the archive of the wiped leaps goes with them
                if (lane == 0) {
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
        __syncwarp();
        long long ginf = 0;
#pragma unroll 1
        for (int i = lane; i < KH; i += 32) {
            const int v = s.Iraw[i];
            st.I[(size_t)r * KH + i] = (long long)v;
            ginf += v;
        }
        for (int o = 16; o > 0; o >>= 1) ginf += __shfl_xor_sync(0xffffffffu, ginf, o);
#pragma unroll 1
        for (int i = lane; i < KS; i += 32) st.Sx[(size_t)r * KS + i] = (long long)s.Sx[i];
#pragma unroll 1
        for (int i = lane; i < K; i += 32) {
            st.cd[(size_t)r * K + i] = s.cd[i];
            st.ceff[(size_t)r * K + i] = s.c[i];
            st.maxEBM[(size_t)r * K + i] = s.maxEBM[i];
            st.lock[(size_t)r * K + i] = s.lock[i];
        }
        if (lane == 0) {
            for (int j = 0; j < 6; j++) ctr[j] = (restarted ? 0 : ctr[j]) + s.tally64[j];
            ctr[C_S] = sC;
            ctr[C_SWAP] += flips_total;
            ctr[C_GOOD] = good_attempt;
            ctr[C_EVPTR] = evptr;
            ctr[C_LEAPS] = leaps;
            ctr[C_GINF] = ginf;
            st.time[r] = t;
            st.epoch[r] = epoch;
        }
        __syncwarp();
    }
    if (prof && lane == 0)
        for (int k = 0; k < 8; k++) atomicAdd(&g_tau_phase_cycles[k], pc[k]);
    if (prof && lane == 0) {  // timing tap: when this warp ran out of work (ns on the global timer) -- the spread over the CTAs
        unsigned long long now;  // is the tail of the launch (slots 8: latest, 9: sum, 10: warps, 11: earliest)
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        atomicMax(&g_tau_phase_cycles[8], now);
        atomicAdd(&g_tau_phase_cycles[9], now & 0xffffffffffull);
        atomicAdd(&g_tau_phase_cycles[10], 1ull);
        atomicMin(&g_tau_phase_cycles[11], now);
        if (blockIdx.x < 512) {
            atomicMin(&g_tau_cta_end[2 * blockIdx.x], now);
            atomicMax(&g_tau_cta_end[2 * blockIdx.x + 1], now);
        }
    }
    // ---- lockstep tail: this warp is out of replicates; keep answering the generation barriers until every
    // warp is.  A warp announces itself after the last barrier of its last generation and before the first
    // barrier of the next; the counter is read between the first and the second barrier of a generation, where
    // no announcement can be in flight, so all idle warps take the same decision.
    if (gsync) {
        __syncwarp();
        if (lane == 0) atomicAdd(done_warps, 1);
        for (;;) {
            TW_GEN_SYNC();
            const bool all = *(volatile int *)done_warps >= gmembers;
            if (gsync == 1) TW_GEN_SYNC();
            if (gsync & 2) TW_GEN_SYNC();
            if (gsync & 4) TW_GEN_SYNC();
            if (all) break;
        }
    }
#undef TW_GEN_SYNC
#undef TW_MARK
}

}  // namespace vg
