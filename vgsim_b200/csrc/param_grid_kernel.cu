// Parameter grids on the device (vgsim_upload_param_grid): one CTA per point assembles the point's source arrays from the
// base point and one patch per axis, checks them, and derives its blob with the host upload's own code (param_blob.cuh).
#include <cuda_runtime.h>
#include "handle.h"
#include "param_blob.cuh"

namespace vg {

static constexpr int GRID_THREADS = 256;

// The source arrays of point g.first_point + i in this CTA's slot: the base, then the patch of every axis in axis order
// (axis 0 slowest).  Ends with a barrier.
static __device__ void assemble(const GridArgs &g, long long nsrc, double *slot, int i) {
    for (long long k = threadIdx.x; k < nsrc; k += blockDim.x) slot[k] = g.base[k];
    __syncthreads();
    const long long pt = g.first_point + i;
    long long start = 0;
    for (int a = 0; a < g.n_axes; a++) {
        long long stride = 1;
        for (int b = a + 1; b < g.n_axes; b++) stride *= g.axis_len[b];
        const long long j = start + (pt / stride) % g.axis_len[a];
        for (long long k = g.off[j] + threadIdx.x; k < g.off[j + 1]; k += blockDim.x) slot[g.idx[k]] = g.val[k];
        start += g.axis_len[a];
        __syncthreads();
    }
}

static __device__ Src<double> src_at(const Dims &D, const double *slot) {
    Src<double> P;
    P.b = slot + src_off(D, F_B);
    P.d = slot + src_off(D, F_D);
    P.s = slot + src_off(D, F_S);
    P.mRate = slot + src_off(D, F_MRATE);
    P.hapMutType = slot + src_off(D, F_HMT);
    P.sigma = slot + src_off(D, F_SIGMA);
    P.suscType = slot + src_off(D, F_SUSC);
    P.T = slot + src_off(D, F_T);
    P.m = slot + src_off(D, F_M);
    P.cd = slot + src_off(D, F_CD);
    P.cdBefore = slot + src_off(D, F_CDB);
    P.cdAfter = slot + src_off(D, F_CDA);
    P.startLD = slot + src_off(D, F_STARTLD);
    P.endLD = slot + src_off(D, F_ENDLD);
    P.sm = slot + src_off(D, F_SM);
    P.sizes = slot + src_off(D, F_SIZES);
    return P;
}

// Pass 1 (WRITE = false) checks every point, records its broken rules (GRID_ERR_* bits) in g.err and raises g.flag;
// pass 2 writes the blobs only when no point failed, so that a failed call leaves the device blobs as they were.
template <bool WRITE>
__global__ void __launch_bounds__(GRID_THREADS) param_grid_kernel(DevState st, GridArgs g) {
    if (WRITE && *g.flag) return;
    const Dims &D = st.D;
    const long long nsrc = src_off(D, NSRC);
    double *slot = g.slots + (size_t)blockIdx.x * nsrc;
    const Src<double> P = src_at(D, slot);
    __shared__ int bits;
    __shared__ double wmax[GRID_THREADS / 32];
    for (int i = blockIdx.x; i < g.n_points; i += gridDim.x) {
        assemble(g, nsrc, slot, i);
        if (!WRITE) {
            if (threadIdx.x == 0) bits = 0;
            __syncthreads();
            int e = 0;
            for (int h = threadIdx.x; h < D.H; h += blockDim.x) {
                const double v = P.suscType[h];
                if (!(v >= 0 && v < D.S && v == floor(v))) e |= GRID_ERR_SUSC;
            }
            for (int p = threadIdx.x; p < D.K; p += blockDim.x) {
                const double v = P.sizes[p];
                if (!(v >= 1 && v <= 2147483647.0 && v == floor(v))) e |= GRID_ERR_SIZES;
                // close_migration_matrix's two rules, its sums in its order
                double leaving = 0.0, stay = 1.0;
                for (int q = 0; q < D.K; q++)
                    if (q != p) {
                        leaving = rn_add(leaving, P.m[(size_t)p * D.K + q]);
                        stay = rn_sub(stay, P.m[(size_t)p * D.K + q]);
                    }
                if (leaving > 1) e |= GRID_ERR_MIG_SUM;
                if (stay <= 1e-15) e |= GRID_ERR_MIG_DIAG;
            }
            if (e) atomicOr(&bits, e);
            __syncthreads();
            if (threadIdx.x == 0) {
                g.err[i] = bits;
                if (bits) atomicOr(g.flag, 1);
            }
            continue;
        }
        double *blob = const_cast<double *>(st.params) + (size_t)(g.dst_pp0 + i) * D.blob;
        for (int k = threadIdx.x; k < D.blob; k += blockDim.x) blob[k] = 0.0;  // the entries no field fills stay 0
        __syncthreads();
        double mb = 0.0;
        for (int h = threadIdx.x; h < D.H; h += blockDim.x) {
            const double v = blob_hap(D, P, blob, h);
            if (v > mb) mb = v;
        }
        for (int s1 = threadIdx.x; s1 < D.S; s1 += blockDim.x) blob_group(D, P, blob, s1);
        for (int p = threadIdx.x; p < D.K; p += blockDim.x) blob_deme(D, P, blob, p);
        for (int o = 16; o > 0; o >>= 1) {
            const double v = __shfl_xor_sync(0xffffffffu, mb, o);
            if (v > mb) mb = v;
        }
        if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = mb;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < GRID_THREADS / 32; w++)
                if (wmax[w] > mb) mb = wmax[w];
            blob[D.o_maxB] = mb;
        }
        __syncthreads();  // the slot is refilled for the next point
    }
}

// Live contact density of every replicate mapped to a grid point: that point's uploaded cd (a first upload's semantics).
__global__ void grid_cd_kernel(DevState st, GridArgs g) {
    if (*g.flag) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= st.R * st.D.K) return;
    const int r = i / st.D.K, p = i - r * st.D.K, pp = st.rep_pp[r];
    if (pp >= g.dst_pp0 && pp < g.dst_pp0 + g.n_points) st.cd[i] = st.params[(size_t)pp * st.D.blob + st.D.o_cd0 + p];
}

int param_grid_slots(int num_sms, int n_points) { return n_points < 4 * num_sms ? n_points : 4 * num_sms; }

cudaError_t launch_param_grid(const DevState &st, const GridArgs &g, cudaStream_t stream) {
    param_grid_kernel<false><<<g.nslots, GRID_THREADS, 0, stream>>>(st, g);
    param_grid_kernel<true><<<g.nslots, GRID_THREADS, 0, stream>>>(st, g);
    const int n = st.R * st.D.K;
    grid_cd_kernel<<<(n + 255) / 256, 256, 0, stream>>>(st, g);
    return cudaGetLastError();
}

}  // namespace vg
