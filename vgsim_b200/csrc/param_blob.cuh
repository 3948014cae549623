// Parameter blob of one point (Dims::o_* layout) derived from its source arrays: the derived constants of UpdateAllRates
// (reference :279-351) in fp64 and the reference's summation order.  One derivation for vgsim_upload_params (host) and
// param_grid_kernel (device): the blob of a point is the same bits on either path.
#pragma once
#include "common.cuh"

namespace vg {

// The source arrays of vgsim_upload_params, in its argument order; a parameter grid's patches index their
// concatenation (vgsim_upload_param_grid).
enum { F_B, F_D, F_S, F_MRATE, F_HMT, F_SIGMA, F_SUSC, F_T, F_M, F_CD, F_CDB, F_CDA, F_STARTLD, F_ENDLD, F_SM, F_SIZES, NSRC };

__host__ __device__ inline long long src_len(const Dims &D, int f) {
    const long long H = D.H, U = D.U, S = D.S, K = D.K;
    switch (f) {
        case F_MRATE: return H * U;
        case F_HMT: return H * U * 3;
        case F_SIGMA: return H * S;
        case F_T: return S * S;
        case F_M: return K * K;
        default: return f <= F_SUSC ? H : K;
    }
}
// offset of field f in the concatenation (f = NSRC: its length)
__host__ __device__ inline long long src_off(const Dims &D, int f) {
    long long o = 0;
    for (int g = 0; g < f; g++) o += src_len(D, g);
    return o;
}

// One point's source arrays in the reference's layouts (include/vgsim_b200.h); I is the element type of suscType and
// sizes (int64 on the host, fp64 in the grid kernel's assembled copy, which holds them exactly).
template <class I>
struct Src {
    const double *b, *d, *s, *mRate, *hapMutType, *sigma, *T, *m, *cd, *cdBefore, *cdAfter, *startLD, *endLD, *sm;
    const I *suscType, *sizes;
};

// Rounding-explicit arithmetic: device code would otherwise contract a * b + c into one FMA and the two paths would
// differ in the last bit.
__host__ __device__ __forceinline__ double rn_add(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
__host__ __device__ __forceinline__ double rn_sub(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
__host__ __device__ __forceinline__ double rn_mul(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
__host__ __device__ __forceinline__ double rn_div(double a, double b) {
#ifdef __CUDA_ARCH__
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}

// The entries of haplotype i; returns max_s b[i] * sigma[i][s] (at least 0), whose maximum over i is the blob's maxB.
template <class I>
__host__ __device__ inline double blob_hap(const Dims &D, const Src<I> &P, double *blob, int i) {
    const int U = D.U, S = D.S, H = D.H;
    blob[D.o_b + i] = P.b[i];
    blob[D.o_d + i] = P.d[i];
    blob[D.o_sr + i] = P.s[i];
    blob[D.o_g + i] = (double)P.suscType[i];
    double tq = 0.0;
    for (int u = 0; u < U; u++) {
        const double *w = &P.hapMutType[((size_t)i * U + u) * 3];
        const double mr = P.mRate[(size_t)i * U + u];
        blob[D.o_mu + i * U + u] = mr;
        for (int k = 0; k < 3; k++) {
            double q = rn_div(rn_mul(mr, w[k]), rn_add(rn_add(w[0], w[1]), w[2]));  // (:2400-2401)
            blob[D.o_q + (i * U + u) * 3 + k] = q;
            blob[D.o_w + (i * U + u) * 3 + k] = w[k];
            tq = rn_add(tq, q);
        }
    }
    blob[D.o_tmq + i] = tq;
    double maxB = 0.0;
    for (int sn = 0; sn < S; sn++) {
        const double sg = P.sigma[(size_t)i * S + sn];
        blob[D.o_sigT + sn * H + i] = sg;
        if (rn_mul(P.b[i], sg) > maxB) maxB = rn_mul(P.b[i], sg);
    }
    return maxB;
}

// The entries of susceptibility group s1: row s1 of T and its sum.
template <class I>
__host__ __device__ inline void blob_group(const Dims &D, const Src<I> &P, double *blob, int s1) {
    const int S = D.S;
    double tc = 0;
    for (int s2 = 0; s2 < S; s2++) {
        blob[D.o_T + s1 * S + s2] = P.T[(size_t)s1 * S + s2];
        tc = rn_add(tc, P.T[(size_t)s1 * S + s2]);
    }
    blob[D.o_Tc + s1] = tc;
}

// The entries of deme p1: row p1 of the migration matrix with its diagonal filled in as 1 - (off-diagonal sum, in
// target order, like close_migration_matrix), the actual size A[p1] and the per-deme vectors.  Only off-diagonals of the
// source matrix are read.
template <class I>
__host__ __device__ inline void blob_deme(const Dims &D, const Src<I> &P, double *blob, int p1) {
    const int K = D.K;
    double stay = 1.0;
    for (int p2 = 0; p2 < K; p2++)
        if (p2 != p1) stay = rn_sub(stay, P.m[(size_t)p1 * K + p2]);
    double A = 0.0;
    for (int p2 = 0; p2 < K; p2++) {
        if (p2 == p1) continue;
        A = rn_add(A, rn_mul(P.m[(size_t)p2 * K + p1], (double)P.sizes[p2]));
    }
    A = rn_add(A, rn_mul(stay, (double)P.sizes[p1]));
    for (int q = 0; q < K; q++) blob[D.o_m + p1 * K + q] = q == p1 ? stay : P.m[(size_t)p1 * K + q];
    blob[D.o_A + p1] = A;
    blob[D.o_sm + p1] = P.sm[p1];
    blob[D.o_cd0 + p1] = P.cd[p1];
    blob[D.o_cdB + p1] = P.cdBefore[p1];
    blob[D.o_cdA + p1] = P.cdAfter[p1];
    blob[D.o_startN + p1] = rn_mul(P.startLD[p1], (double)P.sizes[p1]);
    blob[D.o_endN + p1] = rn_mul(P.endLD[p1], (double)P.sizes[p1]);
    blob[D.o_size + p1] = (double)P.sizes[p1];
}

}  // namespace vg
