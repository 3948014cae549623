// Lineages through time of every replicate's genealogy on a time grid shared by all replicates.
//
// L_r(t_j) = #{ node i : time[i] >= t_j and (parent[i] < 0 or time[parent[i]] < t_j) }: the branch above node i is
// alive at the grid points in (time[parent], time[i]] (a root's branch from -inf).  One warp per replicate over the
// genealogy's node arrays (GenealogyBuffers): every node binary-searches the grid once, j(i) = #{ j : t_j <= time[i] }
// into the per-node scratch; then each branch adds +1 at j(parent) (0 for a root) and -1 at j(i) into the warp's
// difference array in shared memory (int32[T + 1]), and a warp prefix sum writes the row.  Roofline: the tree
// (4 + 8 + 4 bytes per node, the scratch written and read once) + 8 T bytes per replicate.
#include "common.cuh"
#include "handle.h"

namespace vg {

extern __shared__ __align__(16) unsigned char ltt_smem[];

#define LTT_MAX_POINTS 32768  // int32[T + 1] per warp must fit one SM's shared memory with one warp per CTA

int ltt_max_points() { return LTT_MAX_POINTS; }

__host__ __device__ static inline int ltt_stride(int npoints) { return (npoints + 1 + 3) & ~3; }  // ints per warp, 16-byte aligned

__global__ void ltt_kernel(const int R, const long long *node_off, const int *parent, const double *time,
                           const int *n_nodes, int *scratch, const double *times, const int T, long long *out) {
    const int lane = threadIdx.x & 31, wpc = blockDim.x >> 5;
    int *d = reinterpret_cast<int *>(ltt_smem) + (size_t)(threadIdx.x >> 5) * ltt_stride(T);
    for (int r = blockIdx.x * wpc + (threadIdx.x >> 5); r < R; r += gridDim.x * wpc) {
        long long *o = out + (size_t)r * T;
        const int n = n_nodes[r];
        if (n == 0) {  // no tree: a row of zeros
            for (int j = lane; j < T; j += 32) o[j] = 0;
            continue;
        }
        const int *par = parent + node_off[r];
        const double *tm = time + node_off[r];
        int *jn = scratch + node_off[r];
        for (int j = lane; j <= T; j += 32) d[j] = 0;
        for (int i = lane; i < n; i += 32) {  // upper bound: first grid index with t_j > time[i]
            const double t = tm[i];
            int lo = 0, hi = T;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (__ldg(times + mid) <= t)
                    lo = mid + 1;
                else
                    hi = mid;
            }
            jn[i] = lo;
        }
        __syncwarp();
        for (int i = lane; i < n; i += 32) {
            const int p = par[i];
            atomicAdd(&d[p < 0 ? 0 : jn[p]], 1);
            atomicAdd(&d[jn[i]], -1);
        }
        __syncwarp();
        int carry = 0;
        for (int j0 = 0; j0 < T; j0 += 32) {  // inclusive warp scan, 32 points at a time
            const int j = j0 + lane;
            int v = j < T ? d[j] : 0;
#pragma unroll
            for (int w = 1; w < 32; w <<= 1) {
                const int u = __shfl_up_sync(0xffffffffu, v, w);
                if (lane >= w) v += u;
            }
            v += carry;
            if (j < T) o[j] = v;
            carry = __shfl_sync(0xffffffffu, v, 31);
        }
        __syncwarp();
    }
}

cudaError_t launch_ltt(const DevState &st, const long long *node_off, const int *parent, const double *time,
                       const int *n_nodes, int *scratch, const double *times, int npoints, long long *out,
                       cudaStream_t stream, int num_sms) {
    const size_t per_warp = (size_t)ltt_stride(npoints) * 4;
    int wpc = (int)((227 * 1024) / per_warp);
    if (wpc > 8) wpc = 8;
    if (wpc < 1) return cudaErrorInvalidValue;
    const size_t smem = (size_t)wpc * per_warp;
    cudaError_t e = cudaFuncSetAttribute(ltt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int per_sm = 1;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ltt_kernel, wpc * 32, smem);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    int grid = (st.R + wpc - 1) / wpc;
    if (grid > num_sms * per_sm) grid = num_sms * per_sm;
    ltt_kernel<<<grid, wpc * 32, smem, stream>>>(st.R, node_off, parent, time, n_nodes, scratch, times, npoints, out);
    return cudaGetLastError();
}

}  // namespace vg
