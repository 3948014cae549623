// Backward coalescent replay (reference GetGenealogy, src/_BirthDeath.pyx:743-1000).
//
// One WARP per replicate.  The replay is inherently sequential per replicate, so the warp runs the
// scalar logic redundantly in all lanes (identical loads, identical stores -> one transaction) and
// uses the lanes for the parts that are parallel: prefetching 32 log rows at a time with one coalesced
// load, scanning the dense tau-leap count rows for non-zero records with __ballot_sync, bulk copies of
// lineage vectors, and the final parent/child deme comparison.
//
// Live lineages: the reference keeps vector<vector<vector<ssize_t>>> liveBranchesS[K][H] (:747,775-783).
// Here each (deme, haplotype) cell is a growable int32 vector inside a per-replicate arena in HBM:
// header (offset, size, capacity); growth doubles the capacity by bump allocation; when the active half
// of the arena is exhausted, all vectors are compacted into the other half (capacity 2*size), which
// always fits because at most n_samples lineages are alive.  Element order inside a vector is kept
// exactly as std::vector would have it (push_back / swap-with-last / pop_back), so with the same
// random stream the parent arrays are bit-identical to the reference's.
//
// Random stream: Philox4x32-10 keyed by the replicate seed (throughput mode), or an injected stream
// (parity taps): fp64 uniforms, or raw 64-bit words consumed exactly like numpy's PCG64 bit generator
// (next_double = (w >> 11) * 2^-53; 32-bit draws take the low half first and buffer the high half),
// which also drives the numpy-compatible hypergeometric sampler used for tau-leap logs (:885,931,949,955).
#include <cuda_runtime.h>
#include <algorithm>
#include <string>
#include <vector>
#include "../../include/vgsim_b200.h"
#include "common.cuh"
#include "logrec.cuh"
#include "host.h"
#include "genrng.cuh"

namespace vg {

// ---- per-replicate lineage store
struct GenArgs {
    const long long *node_off;   // [R+1]
    int *parent, *pop;
    double *time;
    int *nl;                     // scratch list (newLineages of one tau record), same offsets as nodes
    const long long *arena_off;  // [R+1]; per replicate 2*X ints
    int *arena;
    int *hdr;                    // [R][KH][3]
    const long long *mut_off, *mig_off;  // [R+1]
    int *mut_node, *mut_hap, *mut_nhap;
    double *mut_time;
    int *mig_node, *mig_old, *mig_new;
    double *mig_time;
    int *n_nodes, *mut_n, *mig_n;  // [R]
    const unsigned long long *new_seeds;  // [R] or null
    const double *ustream;                // injected stream (doubles or raw words) or null
    const long long *uoff;                // [R+1]
    long long *uused;                     // [R] words/doubles consumed
    int raw_words;
};

struct Lin {
    int *hdr;    // [KH][3]
    int *arena;  // replicate base
    int X;       // half size
    int half;    // active half
    int bump;    // next free slot (absolute inside the replicate arena)
    int KH;
    int err;

    __device__ __forceinline__ int size(int cell) const { return hdr[3 * cell + 1]; }
    __device__ __forceinline__ int get(int cell, int i) const { return arena[hdr[3 * cell] + i]; }
    __device__ __forceinline__ void set(int cell, int i, int v) { arena[hdr[3 * cell] + i] = v; }
    __device__ __forceinline__ void pop(int cell) { hdr[3 * cell + 1] -= 1; }
    // swap-with-last removal, exactly `v[i] = v[n-1]; v.pop_back()`
    __device__ __forceinline__ void remove_at(int cell, int i) {
        int off = hdr[3 * cell], n = hdr[3 * cell + 1];
        arena[off + i] = arena[off + n - 1];
        hdr[3 * cell + 1] = n - 1;
    }
    __device__ void compact() {
        const int lane = threadIdx.x & 31;
        int other = 1 - half;
        int nb = other * X;
        __syncwarp();
        for (int c = 0; c < KH; c++) {
            int off = hdr[3 * c], n = hdr[3 * c + 1];
            int ncap = n > 0 ? (2 * n > 4 ? 2 * n : 4) : 0;
            for (int i = lane; i < n; i += 32) arena[nb + i] = arena[off + i];
            __syncwarp();
            hdr[3 * c] = nb;
            hdr[3 * c + 2] = ncap;
            nb += ncap;
            __syncwarp();
        }
        half = other;
        bump = nb;
    }
    __device__ void grow(int cell) {
        const int lane = threadIdx.x & 31;
        int cap = hdr[3 * cell + 2];
        int ncap = cap > 0 ? 2 * cap : 4;
        if (bump + ncap > (half + 1) * X) {
            compact();
            if (hdr[3 * cell + 1] < hdr[3 * cell + 2]) return;
            cap = hdr[3 * cell + 2];
            ncap = cap > 0 ? 2 * cap : 4;
            if (bump + ncap > (half + 1) * X) {
                err |= ERR_ARENA;
                return;
            }
        }
        int off = hdr[3 * cell], n = hdr[3 * cell + 1];
        __syncwarp();
        for (int i = lane; i < n; i += 32) arena[bump + i] = arena[off + i];
        __syncwarp();
        hdr[3 * cell] = bump;
        hdr[3 * cell + 2] = ncap;
        bump += ncap;
    }
    __device__ __forceinline__ void push(int cell, int v) {
        if (hdr[3 * cell + 1] >= hdr[3 * cell + 2]) {
            grow(cell);
            if (err) return;
        }
        int n = hdr[3 * cell + 1];
        arena[hdr[3 * cell] + n] = v;
        hdr[3 * cell + 1] = n + 1;
    }
};

struct Out {
    int *parent, *pop;
    double *time;
    int n, cap;
    int *mut_node, *mut_hap, *mut_nhap;
    double *mut_time;
    int mut_n, mut_cap;
    int *mig_node, *mig_old, *mig_new;
    double *mig_time;
    int mig_n, mig_cap;
    int err;
    __device__ __forceinline__ int new_node(int deme, double t) {
        if (n >= cap) {
            err |= ERR_BADLOG;
            return cap - 1;
        }
        parent[n] = -1;
        pop[n] = deme;
        time[n] = t;
        return n++;
    }
    __device__ __forceinline__ void add_mutation(int node, int hap, int nhap, double t) {
        if (mut_n >= mut_cap) {
            err |= ERR_SIDE_TABLE;
            return;
        }
        mut_node[mut_n] = node;
        mut_hap[mut_n] = hap;
        mut_nhap[mut_n] = nhap;
        mut_time[mut_n] = t;
        mut_n++;
    }
    __device__ __forceinline__ void add_migration(int node, double t, int oldp, int newp) {
        if (mig_n >= mig_cap) {
            err |= ERR_SIDE_TABLE;
            return;
        }
        mig_node[mig_n] = node;
        mig_time[mig_n] = t;
        mig_old[mig_n] = oldp;
        mig_new[mig_n] = newp;
        mig_n++;
    }
};

__global__ void __launch_bounds__(128) genealogy_kernel(DevState st, GenArgs ga) {
    const Dims D = st.D;
    const int H = D.H;
    const int lane = threadIdx.x & 31;
    const int wpc = blockDim.x >> 5;
    const int nwarps = gridDim.x * wpc;
    for (int r = blockIdx.x * wpc + (threadIdx.x >> 5); r < st.R; r += nwarps) {
        const long long *ctr = st.counters + (size_t)r * NCOUNT;
        const long long sC = ctr[C_S];
        if (sC < 2) {  // reference: "Less than two cases were sampled..." and exit (:760-763)
            ga.n_nodes[r] = 0;
            ga.mut_n[r] = 0;
            ga.mig_n[r] = 0;
            continue;
        }
        const double *pp = st.params + (size_t)st.rep_pp[r] * D.blob;
        long long *I = st.I + (size_t)r * D.K * H;  // rewound in place like the reference (quirk Q9)
        Lin L;
        L.hdr = ga.hdr + (size_t)r * D.K * H * 3;
        L.arena = ga.arena + ga.arena_off[r];
        L.X = (int)((ga.arena_off[r + 1] - ga.arena_off[r]) / 2);
        L.half = 0;
        L.bump = 0;
        L.KH = D.K * H;
        L.err = 0;
        for (int i = lane; i < L.KH * 3; i += 32) L.hdr[i] = 0;
        __syncwarp();
        Out O;
        O.parent = ga.parent + ga.node_off[r];
        O.pop = ga.pop + ga.node_off[r];
        O.time = ga.time + ga.node_off[r];
        O.n = 0;
        O.cap = (int)(ga.node_off[r + 1] - ga.node_off[r]);
        O.mut_node = ga.mut_node + ga.mut_off[r];
        O.mut_hap = ga.mut_hap + ga.mut_off[r];
        O.mut_nhap = ga.mut_nhap + ga.mut_off[r];
        O.mut_time = ga.mut_time + ga.mut_off[r];
        O.mut_n = 0;
        O.mut_cap = (int)(ga.mut_off[r + 1] - ga.mut_off[r]);
        O.mig_node = ga.mig_node + ga.mig_off[r];
        O.mig_old = ga.mig_old + ga.mig_off[r];
        O.mig_new = ga.mig_new + ga.mig_off[r];
        O.mig_time = ga.mig_time + ga.mig_off[r];
        O.mig_n = 0;
        O.mig_cap = (int)(ga.mig_off[r + 1] - ga.mig_off[r]);
        O.err = 0;
        int *nl = ga.nl + ga.node_off[r];
        GRng g;
        g.err = 0;
        g.has32 = 0;
        g.b32 = 0;
        g.have = 0;
        g.ctr = 0;
        g.buf = make_uint4(0, 0, 0, 0);
        g.ud = nullptr;
        g.uw = nullptr;
        g.pos = g.end = 0;
        if (ga.ustream) {
            g.mode = ga.raw_words ? 2 : 1;
            g.ud = ga.ustream;
            g.uw = reinterpret_cast<const unsigned long long *>(ga.ustream);
            g.pos = ga.uoff[r];
            g.end = ga.uoff[r + 1];
        } else {
            g.mode = 0;
            unsigned long long seed = ga.new_seeds ? ga.new_seeds[r] : st.seeds[r];
            g.key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32) ^ (ga.new_seeds ? 0x9e3779b9u : 0x7f4a7c15u));
        }
        int clamped = 0, bad = 0;

        const double *ev_time = st.ev_time + (size_t)r * st.ev_cap;
        const unsigned long long *ev_desc = st.ev_desc + (size_t)r * st.ev_cap;
        const long long nev = ctr[C_EVPTR];
        for (long long hi = nev; hi > 0 && !bad; hi -= 32) {
            // rows hi-1, hi-2, ... : lane j holds row hi-1-j
            long long mine = hi - 1 - lane;
            double tl = 0.0;
            unsigned long long dl = 0;
            if (mine >= 0) {
                tl = ev_time[mine];
                dl = ev_desc[mine];
            }
            int cnt = hi < 32 ? (int)hi : 32;
            for (int j = 0; j < cnt; j++) {
                const double et = __shfl_sync(0xffffffffu, tl, j);
                const unsigned long long d = __shfl_sync(0xffffffffu, dl, j);
                int ty, eh, ep, enh, enp;
                unpack_event(d, ty, eh, ep, enh, enp);
                if (ty == EV_BIRTH) {  // :797-818
                    const int cell = ep * H + eh;
                    const int lbs = L.size(cell);
                    const long long lbs_e = I[cell];
                    double p = ((double)lbs * ((double)lbs - 1.0)) / (double)lbs_e / ((double)lbs_e - 1.0);
                    if (g.next_double() < p) {
                        int n1 = (int)floor((double)lbs * g.next_double());
                        int n2 = (int)floor((double)(lbs - 1) * g.next_double());
                        if (n2 >= n1) n2 += 1;
                        int id1 = L.get(cell, n1), id2 = L.get(cell, n2);
                        int id3 = O.new_node(ep, et);
                        L.set(cell, n1, id3);
                        L.remove_at(cell, n2);
                        O.parent[id1] = id3;
                        O.parent[id2] = id3;
                    }
                    I[cell] = lbs_e - 1;
                } else if (ty == EV_DEATH) {  // :819-820
                    I[ep * H + eh] += 1;
                } else if (ty == EV_SAMPLING) {  // :821-827
                    I[ep * H + eh] += 1;
                    int id = O.new_node(ep, et);
                    L.push(ep * H + eh, id);
                } else if (ty == EV_MUTATION) {  // :828-839
                    const int cnew = ep * H + enh, cold = ep * H + eh;
                    const int lbs = L.size(cnew);
                    double p = (double)lbs / (double)I[cnew];
                    if (g.next_double() < p) {
                        int n1 = (int)floor((double)lbs * g.next_double());
                        int id1 = L.get(cnew, n1);
                        L.remove_at(cnew, n1);
                        L.push(cold, id1);
                        O.add_mutation(id1, eh, enh, et);
                    }
                    I[cnew] -= 1;
                    I[cold] += 1;
                } else if (ty == EV_SUSCCHANGE) {
                } else if (ty == EV_MIGRATION) {  // :842-868  (ep = source deme, enp = target deme)
                    const int ct = enp * H + eh, cs = ep * H + eh;
                    const int lbs = L.size(ct);
                    double p = (double)lbs / (double)I[ct];
                    if (g.next_double() < p) {
                        int nt = (int)floor((double)lbs * g.next_double());
                        const int lbss = L.size(cs);
                        double p1 = (double)lbss / (double)I[cs];
                        if (g.next_double() < p1) {
                            int ns = (int)floor((double)lbss * g.next_double());
                            int idt = L.get(ct, nt), ids = L.get(cs, ns);
                            int id3 = O.new_node(ep, et);
                            L.set(cs, ns, id3);
                            L.remove_at(ct, nt);
                            O.parent[idt] = id3;
                            O.parent[ids] = id3;
                            O.add_migration(idt, et, ep, enp);
                        } else {
                            int idt = L.get(ct, nt);
                            L.remove_at(ct, nt);
                            L.push(cs, idt);
                        }
                    }
                    I[ct] -= 1;
                } else if (ty == EV_MULTITYPE) {  // :869-993
                    const long long leap = unpack_multi(d);
                    // one record (channel rc, count num) of the leap: :869-993
                    // The reference's pair / lineage hypergeometrics assume lineages <= individuals in every cell.  Its own
                    // approximation can break that (a BIRTH record that draws fewer coalescences than the rewind of `num`
                    // births needs leaves more lineages than individuals): the next draw then has a negative `bad` count
                    // or asks for more than the urn holds -- numpy raises there.  Here the arguments are brought back
                    // into range (flag 16), so that every index drawn below stays inside its lineage vector.
                    auto hyp = [&](long long good, long long bad_n, long long sample) -> long long {
                        if (bad_n < 0) {
                            bad_n = 0;
                            clamped++;
                        }
                        if (sample > good + bad_n) {
                            sample = good + bad_n;
                            clamped++;
                        }
                        const long long k = hypergeometric(g, good, bad_n, sample);
                        return k < 0 ? 0 : (k > good ? good : k);
                    };
                    auto record = [&](int rc, long long num) {
                    int mty, mh, mp, mnh, mnp;
                    decode_record(rc, D, pp, mty, mh, mp, mnh, mnp);
                    const int cell = mp * H + mh;  // the cell that receives the parked (new) lineages
                    int nnl = 0;
                    if (mty == EV_BIRTH) {  // :879-915
                        int lbs = L.size(cell);
                        const long long lbs_e = I[cell];
                        long long k = 0;
                        if (lbs != 0)
                            k = hyp((long long)(((double)lbs * ((double)lbs - 1.0)) / 2.0),
                                               ((lbs_e * (lbs_e - 1)) / 2) - (((long long)lbs * (lbs - 1)) / 2), num);
                        for (long long i = 0; i < k; i++) {
                            if (lbs < 2) {  // the reference runs into UB here; clamp and count
                                clamped++;
                                break;
                            }
                            int n1 = (int)floor((double)lbs * g.next_double());
                            int n2 = (int)floor((double)(lbs - 1) * g.next_double());
                            if (n2 >= n1) n2 += 1;
                            int id1 = L.get(cell, n1), id2 = L.get(cell, n2);
                            int id3 = O.new_node(mp, et);
                            nl[nnl++] = id3;
                            if (n1 == lbs - 1) {
                                L.pop(cell);
                                L.set(cell, n2, L.get(cell, lbs - 2));
                                L.pop(cell);
                            } else if (n2 == lbs - 1) {
                                L.pop(cell);
                                L.set(cell, n1, L.get(cell, lbs - 2));
                                L.pop(cell);
                            } else {
                                L.set(cell, n1, L.get(cell, lbs - 1));
                                L.pop(cell);
                                L.set(cell, n2, L.get(cell, lbs - 2));
                                L.pop(cell);
                            }
                            O.parent[id1] = id3;
                            O.parent[id2] = id3;
                            lbs -= 2;
                        }
                        I[cell] -= num;
                    } else if (mty == EV_DEATH) {  // :916-917
                        I[cell] += num;
                    } else if (mty == EV_SAMPLING) {  // :918-925
                        I[cell] += num;
                        for (long long i = 0; i < num; i++) nl[nnl++] = O.new_node(mp, et);
                    } else if (mty == EV_MUTATION) {  // :926-941
                        const int cnew = mp * H + mnh;
                        int lbs = L.size(cnew);
                        long long k = 0;
                        if (lbs != 0) k = hyp(lbs, I[cnew] - lbs, num);
                        for (long long i = 0; i < k; i++) {
                            int n1 = (int)floor((double)lbs * g.next_double());
                            int id1 = L.get(cnew, n1);
                            L.remove_at(cnew, n1);
                            nl[nnl++] = id1;
                            O.add_mutation(id1, mh, mnh, et);
                            lbs -= 1;
                        }
                        I[cnew] -= num;
                        I[cell] += num;
                    } else if (mty == EV_MIGRATION) {  // :944-982  (mp = source, mnp = target)
                        const int ct = mnp * H + mh;
                        int lbs = L.size(ct);
                        if (lbs != 0) {
                            long long k = hyp(lbs, I[ct] - lbs, num);
                            int lbss = L.size(cell);
                            long long k2 = 0;
                            if (!(k == 0 || lbss == 0)) k2 = hyp(lbss, I[cell] - lbss, k);
                            for (long long i = 0; i < k2; i++) {
                                int nt = (int)floor((double)lbs * g.next_double());
                                int ns = (int)floor((double)lbss * g.next_double());
                                int idt = L.get(ct, nt), ids = L.get(cell, ns);
                                int id3 = O.new_node(mp, et);
                                L.remove_at(cell, ns);
                                L.remove_at(ct, nt);
                                nl[nnl++] = id3;
                                O.parent[idt] = id3;
                                O.parent[ids] = id3;
                                O.add_migration(idt, et, mp, mnp);
                                lbss -= 1;
                                lbs -= 1;
                            }
                            for (long long i = 0; i < k - k2; i++) {
                                int nt = (int)floor((double)lbs * g.next_double());
                                nl[nnl++] = L.get(ct, nt);
                                L.remove_at(ct, nt);
                                lbs -= 1;
                            }
                        }
                        I[ct] -= num;
                    }
                    // merge the parked lineages back, last parked first (:987-993; only this record's
                    // receiving cell can hold any — untouched cells have nothing parked and no delta)
                    for (int i = nnl - 1; i >= 0; i--) L.push(cell, nl[i]);
                    if (g.err | L.err | O.err) bad = 1;
                    };
                    const long long dbase = st.dense_base[r];
                    if (leap < dbase) {
                        // archived leap: its non-zero counts are (channel, count) pairs in ascending channel order
                        const int *soff = st.sp_off + (size_t)r * (st.leap_cap + 1);
                        const int2 *ent = st.sp_ent + (size_t)r * st.sp_cap;
                        const int e0 = soff[leap], e1 = soff[leap + 1];
                        for (int eb = e0; eb < e1 && !bad; eb += 32) {
                            const int2 mine = eb + lane < e1 ? __ldcs(ent + eb + lane) : make_int2(0, 0);
                            const int nn = e1 - eb < 32 ? e1 - eb : 32;
                            for (int k = 0; k < nn; k++) {
                                const int rc = __shfl_sync(0xffffffffu, mine.x, k), rn = __shfl_sync(0xffffffffu, mine.y, k);
                                record(rc, (long long)rn);
                                if (bad) break;
                            }
                        }
                    } else {
                    const int *row = st.tau_counts + ((size_t)r * st.dense_cap + (leap - dbase)) * D.Pp;
                    // the row is scanned in ascending channel order, 128 counts (one int4 per lane) per step; eight steps'
                    // worth of loads (4 KB per warp) are in flight at a time -- one dependent 128-byte load per step made
                    // the scan latency-bound (11 s for 32 world-shape replicates x 1,200 leaps of 493,400 channels)
                    const int4 *row4 = reinterpret_cast<const int4 *>(row);
                    const int n16 = D.Pp >> 2;
                    int4 pre[8];
                    for (int base4 = 0; base4 < n16 && !bad; base4 += 32) {
                        if ((base4 & 255) == 0) {
#pragma unroll
                            for (int u = 0; u < 8; u++) {
                                const int j4 = base4 + u * 32 + lane;
                                pre[u] = j4 < n16 ? __ldcs(row4 + j4) : make_int4(0, 0, 0, 0);
                            }
                        }
                        const int4 v_l = pre[0];
#pragma unroll
                        for (int u = 0; u < 7; u++) pre[u] = pre[u + 1];
                        unsigned nzmask = __ballot_sync(0xffffffffu, (v_l.x | v_l.y | v_l.z | v_l.w) != 0);
                        while (nzmask) {
                            int b = __ffs(nzmask) - 1;
                            nzmask &= nzmask - 1;
                            const int q0 = __shfl_sync(0xffffffffu, v_l.x, b), q1 = __shfl_sync(0xffffffffu, v_l.y, b),
                                      q2 = __shfl_sync(0xffffffffu, v_l.z, b), q3 = __shfl_sync(0xffffffffu, v_l.w, b);
                            for (int e4 = 0; e4 < 4; e4++) {
                            const long long num = e4 == 0 ? q0 : e4 == 1 ? q1 : e4 == 2 ? q2 : q3;
                            if (num == 0) continue;
                            record((base4 + b) * 4 + e4, num);
                            if (bad) break;
                            }  // e4
                            if (bad) break;
                        }
                    }
                    }
                } else {
                    bad = 1;
                    O.err |= ERR_BADLOG;
                }
                if (g.err | L.err | O.err) bad = 1;
                if (bad) break;
            }
        }
        __syncwarp();
        // ---- post-pass (:998-1000): a Migrations row for every node whose parent sits in another deme
        const int nn = O.n;
        const int lim = (int)(sC * 2 - 2) < nn ? (int)(sC * 2 - 2) : nn;
        for (int base = 0; base < lim; base += 32) {
            int i = base + lane;
            int flag = 0, par = -1;
            if (i < lim) {
                par = O.parent[i];
                if (par >= 0 && O.pop[par] != O.pop[i]) flag = 1;
            }
            unsigned m = __ballot_sync(0xffffffffu, flag);
            int slot = O.mig_n + __popc(m & ((1u << lane) - 1));
            if (flag) {
                if (slot < O.mig_cap) {
                    O.mig_node[slot] = i;
                    O.mig_time[slot] = O.time[i];
                    O.mig_old[slot] = O.pop[par];
                    O.mig_new[slot] = O.pop[i];
                }
            }
            O.mig_n += __popc(m);
            if (O.mig_n > O.mig_cap) {
                O.mig_n = O.mig_cap;
                O.err |= ERR_SIDE_TABLE;
            }
        }
        ga.n_nodes[r] = O.n;
        ga.mut_n[r] = O.mut_n;
        ga.mig_n[r] = O.mig_n;
        if (ga.uused) ga.uused[r] = g.pos - (ga.ustream ? ga.uoff[r] : 0);
        int e = L.err | O.err | (g.err ? ERR_STREAM : 0) | (clamped ? ERR_CLAMPED : 0);
        if (e) st.err[r] |= e;
        __syncwarp();
    }
}

}  // namespace vg

using namespace vg;

namespace {

void free_gen(Handle *h) {
    GenealogyBuffers &G = h->gen;
    void *ptrs[] = {G.node_off, G.parent, G.pop, G.time, G.mut_off, G.mig_off, G.mut_n, G.mig_n, G.mut_node, G.mut_hap,
                    G.mut_nhap, G.mut_time, G.mig_node, G.mig_old, G.mig_new, G.mig_time, G.arena_off, G.arena,
                    G.cell_hdr, G.n_nodes, G.scratch};
    for (void *p : ptrs) dfree(h, p);
    G = GenealogyBuffers();
}

// One replay of every replicate's log into new output buffers whose side tables are `table_scale` times the default
// size; `ga` brings the caller's seeds or uniform stream.  *overflow: the side tables of some replicate overflowed (its
// error bit is cleared again).
int replay(Handle *h, const std::vector<long long> &ctr, long long table_scale, GenArgs ga, bool *overflow) {
    const Dims &D = h->D;
    const int R = h->R;
    free_gen(h);
    GenealogyBuffers &G = h->gen;
    G.h_node_off.assign(R + 1, 0);
    G.h_mut_off.assign(R + 1, 0);
    G.h_mig_off.assign(R + 1, 0);
    std::vector<long long> arena_off(R + 1, 0);
    const long long KH = (long long)D.K * D.H;
    for (int r = 0; r < R; r++) {
        long long sC = ctr[(size_t)r * NCOUNT + C_S];
        long long nodes = sC >= 2 ? 2 * sC - 1 : 0;
        G.h_node_off[r + 1] = G.h_node_off[r] + nodes;
        G.h_mut_off[r + 1] = G.h_mut_off[r] + (sC >= 2 ? (8 * sC + 64) * table_scale : 0);
        G.h_mig_off[r + 1] = G.h_mig_off[r] + (sC >= 2 ? (3 * sC + 8) * table_scale : 0);
        arena_off[r + 1] = arena_off[r] + (sC >= 2 ? 2 * (2 * sC + 4 * KH) : 0);
        if (2 * sC + 4 * KH > 1000000000LL) return fail("sample count too large for int32 lineage arena");
    }
    G.total_nodes = G.h_node_off[R];
    if (dalloc(h, &G.node_off, R + 1) || dalloc(h, &G.mut_off, R + 1) || dalloc(h, &G.mig_off, R + 1) ||
        dalloc(h, &G.arena_off, R + 1) || dalloc(h, &G.parent, G.total_nodes) || dalloc(h, &G.pop, G.total_nodes) ||
        dalloc(h, &G.time, G.total_nodes) || dalloc(h, &G.scratch, G.total_nodes) || dalloc(h, &G.arena, arena_off[R]) ||
        dalloc(h, &G.cell_hdr, (size_t)R * KH * 3) || dalloc(h, &G.n_nodes, R) || dalloc(h, &G.mut_n, R) ||
        dalloc(h, &G.mig_n, R) || dalloc(h, &G.mut_node, G.h_mut_off[R]) || dalloc(h, &G.mut_hap, G.h_mut_off[R]) ||
        dalloc(h, &G.mut_nhap, G.h_mut_off[R]) || dalloc(h, &G.mut_time, G.h_mut_off[R]) ||
        dalloc(h, &G.mig_node, G.h_mig_off[R]) || dalloc(h, &G.mig_old, G.h_mig_off[R]) ||
        dalloc(h, &G.mig_new, G.h_mig_off[R]) || dalloc(h, &G.mig_time, G.h_mig_off[R]))
        return 1;
    CK(cudaMemcpyAsync(G.node_off, G.h_node_off.data(), (R + 1) * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(G.mut_off, G.h_mut_off.data(), (R + 1) * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(G.mig_off, G.h_mig_off.data(), (R + 1) * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(G.arena_off, arena_off.data(), (R + 1) * 8, cudaMemcpyHostToDevice, h->stream));
    ga.node_off = G.node_off;
    ga.parent = G.parent;
    ga.pop = G.pop;
    ga.time = G.time;
    ga.nl = G.scratch;
    ga.arena_off = G.arena_off;
    ga.arena = G.arena;
    ga.hdr = G.cell_hdr;
    ga.mut_off = G.mut_off;
    ga.mig_off = G.mig_off;
    ga.mut_node = G.mut_node;
    ga.mut_hap = G.mut_hap;
    ga.mut_nhap = G.mut_nhap;
    ga.mut_time = G.mut_time;
    ga.mig_node = G.mig_node;
    ga.mig_old = G.mig_old;
    ga.mig_new = G.mig_new;
    ga.mig_time = G.mig_time;
    ga.n_nodes = G.n_nodes;
    ga.mut_n = G.mut_n;
    ga.mig_n = G.mig_n;
    int wpc = 4;
    int grid = (R + wpc - 1) / wpc;
    int maxgrid = h->num_sms * 16;
    if (grid > maxgrid) grid = maxgrid;
    genealogy_kernel<<<grid, wpc * 32, 0, h->stream>>>(h->st, ga);
    h->launches++;
    CK(cudaGetLastError());
    std::vector<int> errs(R);
    CK(cudaMemcpyAsync(errs.data(), h->st.err, (size_t)R * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    *overflow = false;
    for (int &v : errs)
        if (v & ERR_SIDE_TABLE) {
            *overflow = true;
            v &= ~ERR_SIDE_TABLE;
        }
    if (*overflow) {
        CK(cudaMemcpyAsync(h->st.err, errs.data(), (size_t)R * 4, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    return 0;
}

// *n = counts[r] of one of the genealogy's per-replicate counts (n_nodes, mut_n, mig_n)
int gen_count(Handle *h, int r, const int *counts, int *n) {
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(n, counts + r, 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

}  // namespace

extern "C" {

int vgsim_genealogy(vgsim_handle h, const uint64_t *seeds, const double *uniform_stream, const int64_t *stream_offsets,
                    int raw_words) {
    CK(cudaSetDevice(h->device));
    if (!h->st.first_simulation) return fail("nothing was simulated");
    if (uniform_stream && !stream_offsets) return fail("stream_offsets is required with uniform_stream");
    const int R = h->R;
    std::vector<long long> ctr((size_t)R * NCOUNT);
    CK(cudaMemcpyAsync(ctr.data(), h->st.counters, ctr.size() * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    GenArgs ga{};
    ga.raw_words = raw_words;
    Scratch<unsigned long long> dseeds;
    Scratch<double> dstream;
    Scratch<long long> doff, dused;
    if (seeds) {
        if (dseeds.alloc(R)) return 1;
        CK(cudaMemcpyAsync(dseeds, seeds, (size_t)R * 8, cudaMemcpyHostToDevice, h->stream));
        ga.new_seeds = dseeds;
    }
    if (uniform_stream) {
        const long long n = stream_offsets[R];
        if (dstream.alloc(n) || doff.alloc(R + 1) || dused.alloc(R)) return 1;
        CK(cudaMemcpyAsync(dstream, uniform_stream, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(doff, stream_offsets, (size_t)(R + 1) * 8, cudaMemcpyHostToDevice, h->stream));
        ga.ustream = dstream;
        ga.uoff = doff;
        ga.uused = dused;
    }
    // The mutation / migration side tables grow with rate x branch length, not with the sample count (the reference
    // appends to std::vectors, src/models.pxi): start from a size that covers the usual case and, if a replicate
    // overflows, run the replay again with 8x larger tables.  The replay rewinds the infectious counts in place (quirk
    // Q9), so they are saved first and put back before a retry.
    const size_t I_n = (size_t)R * h->D.K * h->D.H;
    Scratch<long long> I_saved;
    if (I_saved.alloc(I_n)) return 1;
    CK(cudaMemcpyAsync(I_saved, h->st.I, I_n * 8, cudaMemcpyDeviceToDevice, h->stream));
    for (long long attempt = 0, table_scale = 1;; attempt++, table_scale *= 8) {
        if (attempt > 0) CK(cudaMemcpyAsync(h->st.I, I_saved, I_n * 8, cudaMemcpyDeviceToDevice, h->stream));
        bool overflow = false;
        if (replay(h, ctr, table_scale, ga, &overflow)) return 1;
        if (!overflow) break;
        if (attempt >= 3) return fail("genealogy side tables overflow even at 512x the default capacity");
    }
    h->gen.valid = true;
    return 0;
}

int64_t vgsim_tree_size(vgsim_handle h, int r) {
    if (check_replicate(h, r)) return -1;
    if (!h->gen.valid) return 0;
    return h->gen.h_node_off[r + 1] - h->gen.h_node_off[r];
}

int vgsim_get_tree(vgsim_handle h, int r, int64_t *parent, int64_t *pop, double *time) {
    if (!h->gen.valid) return fail("genealogy was not simulated");
    if (check_replicate(h, r)) return 1;
    const long long n = h->gen.h_node_off[r + 1] - h->gen.h_node_off[r], off = h->gen.h_node_off[r];
    if (n == 0) return 0;
    int used = 0;
    if (gen_count(h, r, h->gen.n_nodes, &used)) return 1;
    std::vector<int> a(n), b(n);
    CK(cudaMemcpyAsync(a.data(), h->gen.parent + off, n * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(b.data(), h->gen.pop + off, n * 4, cudaMemcpyDeviceToHost, h->stream));
    if (time) CK(cudaMemcpyAsync(time, h->gen.time + off, n * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (long long i = 0; i < n; i++) {
        // nodes never created (incomplete coalescence) read as the reference's zero-initialised arrays
        if (parent) parent[i] = i < used ? a[i] : 0;
        if (pop) pop[i] = i < used ? b[i] : 0;
        if (time && i >= used) time[i] = 0.0;
    }
    return 0;
}

int64_t vgsim_num_mutations(vgsim_handle h, int r) {
    int n = 0;
    if (check_replicate(h, r) || (h->gen.valid && gen_count(h, r, h->gen.mut_n, &n))) return -1;
    return n;
}

int vgsim_get_mutations(vgsim_handle h, int r, int64_t *node, int64_t *AS, int64_t *DS, int64_t *site, double *time) {
    if (!h->gen.valid) return fail("genealogy was not simulated");
    int n = 0;
    if (check_replicate(h, r) || gen_count(h, r, h->gen.mut_n, &n)) return 1;
    if (n == 0) return 0;
    long long off = h->gen.h_mut_off[r];
    std::vector<int> a(n), b(n), c(n);
    CK(cudaMemcpyAsync(a.data(), h->gen.mut_node + off, n * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(b.data(), h->gen.mut_hap + off, n * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(c.data(), h->gen.mut_nhap + off, n * 4, cudaMemcpyDeviceToHost, h->stream));
    if (time) CK(cudaMemcpyAsync(time, h->gen.mut_time + off, n * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < n; i++) {
        // Mutations.AddMutation (src/models.pxi:12-26): site counted from the least-significant base-4 digit
        long long x = std::llabs((long long)c[i] - b[i]), s = 0;
        while (x >= 4) {
            x /= 4;
            s++;
        }
        long long digit4 = 1;
        for (long long k = 0; k < s; k++) digit4 *= 4;
        if (node) node[i] = a[i];
        if (DS) DS[i] = (c[i] / digit4) % 4;
        if (AS) AS[i] = (b[i] / digit4) % 4;
        if (site) site[i] = s;
    }
    return 0;
}

int64_t vgsim_num_migrations(vgsim_handle h, int r) {
    int n = 0;
    if (check_replicate(h, r) || (h->gen.valid && gen_count(h, r, h->gen.mig_n, &n))) return -1;
    return n;
}

int vgsim_get_migrations(vgsim_handle h, int r, int64_t *node, double *time, int64_t *old_pop, int64_t *new_pop) {
    if (!h->gen.valid) return fail("genealogy was not simulated");
    int n = 0;
    if (check_replicate(h, r) || gen_count(h, r, h->gen.mig_n, &n)) return 1;
    if (n == 0) return 0;
    long long off = h->gen.h_mig_off[r];
    std::vector<int> a(n), b(n), c(n);
    CK(cudaMemcpyAsync(a.data(), h->gen.mig_node + off, n * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(b.data(), h->gen.mig_old + off, n * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(c.data(), h->gen.mig_new + off, n * 4, cudaMemcpyDeviceToHost, h->stream));
    if (time) CK(cudaMemcpyAsync(time, h->gen.mig_time + off, n * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < n; i++) {
        if (node) node[i] = a[i];
        if (old_pop) old_pop[i] = b[i];
        if (new_pop) new_pop[i] = c[i];
    }
    return 0;
}

}  // extern "C"
