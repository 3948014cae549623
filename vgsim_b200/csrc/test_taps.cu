// Test taps for the device samplers (include/vgsim_b200.h: vgsim_test_poisson).
#include <cuda_runtime.h>
#include <string>
#include "../../include/vgsim_b200.h"
#include "common.cuh"
#include "host.h"
#include "samplers.cuh"
#include "genrng.cuh"
#include "choose.cuh"

namespace vg {
__global__ void poisson_tap_kernel(const double *lam, long long n, uint64_t seed, long long *out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    // same addressing as the tau kernel: 4 draws share one Philox block (chunk = i/4, lane = i%4)
    PhiloxCtx ctx;
    ctx.key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    ctx.c0 = (uint32_t)(i >> 2);
    ctx.c1 = (uint32_t)(i >> 34);
    ctx.c2 = 0x5eedu;
    double l = lam[i];
    long long v = 0;
    if (l > 0.0) {
        uint4 w = ctx.draw(0u);
        v = poisson_draw(l, pick_word(w, (int)(i & 3)), ctx, (int)(i & 3));
    }
    out[i] = v;
}
}  // namespace vg

extern "C" int vgsim_test_poisson(const double *lam, int64_t n, uint64_t seed, int64_t *out) {
    vg::Scratch<double> dl;
    vg::Scratch<long long> dout;
    if (dl.alloc(n) || dout.alloc(n)) return 1;
    CK(cudaMemcpy(dl, lam, n * 8, cudaMemcpyHostToDevice));
    vg::poisson_tap_kernel<<<(unsigned)((n + 255) / 256), 256>>>(dl, n, seed, dout);
    CK(cudaGetLastError());
    CK(cudaMemcpy(out, dout, n * 8, cudaMemcpyDeviceToHost));
    return 0;
}

namespace vg {
__global__ void hyper_tap_kernel(const long long *good, const long long *bad, const long long *sample, long long n,
                                 const unsigned long long *words, long long n_words, long long *out, long long *used) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    GRng g;
    g.mode = 2;
    g.ud = nullptr;
    g.uw = words;
    g.pos = 0;
    g.end = n_words;
    g.err = 0;
    g.has32 = 0;
    g.b32 = 0;
    g.have = 0;
    g.ctr = 0;
    for (long long i = 0; i < n; i++) out[i] = hypergeometric(g, good[i], bad[i], sample[i]);
    *used = g.err ? -1 : g.pos;
}
}  // namespace vg

// sequential draws from an injected raw-word stream (numpy PCG64 semantics), for draw-for-draw parity
extern "C" int vgsim_test_hypergeometric(const int64_t *good, const int64_t *bad, const int64_t *sample, int64_t n,
                                         const uint64_t *raw_words, int64_t n_words, int64_t *out, int64_t *words_used) {
    vg::Scratch<long long> dg, db, ds, dout, dused;
    vg::Scratch<unsigned long long> dw;
    if (dg.alloc(n) || db.alloc(n) || ds.alloc(n) || dout.alloc(n) || dused.alloc(1) || dw.alloc(n_words)) return 1;
    CK(cudaMemcpy(dg, good, n * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(db, bad, n * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ds, sample, n * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dw, raw_words, n_words * 8, cudaMemcpyHostToDevice));
    vg::hyper_tap_kernel<<<1, 32>>>(dg, db, ds, n, dw, n_words, dout, dused);
    CK(cudaGetLastError());
    CK(cudaMemcpy(out, dout, n * 8, cudaMemcpyDeviceToHost));
    long long u = 0;
    CK(cudaMemcpy(&u, dused, 8, cudaMemcpyDeviceToHost));
    if (words_used) *words_used = u;
    return 0;
}

// ---- cumulative search tap (choose.cuh): one warp per query
namespace vg {
__global__ void choose_tap_kernel(const double *w, int n, const double *x, int m, int skip, int small, long long *idx,
                                  double *before, double *wsel, double *resid) {
    const int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (q >= m) return;
    const Pick p = small ? small_pick([&](int i) { return i == skip ? 0.0 : w[i]; }, n, x[q])
                         : warp_pick([&](int i) { return w[i]; }, n, x[q], skip);
    if ((threadIdx.x & 31) == 0) {
        idx[q] = p.i;
        before[q] = p.before;
        wsel[q] = p.w;
        resid[q] = p.i >= 0 ? p.resid(x[q]) : -1.0;
    }
}
}  // namespace vg

extern "C" int vgsim_test_choose(const double *w, int n, const double *x, int m, int skip, int small, int64_t *idx,
                                 double *before, double *wsel, double *resid) {
    vg::Scratch<double> dw, dx, db, dws, dr;
    vg::Scratch<long long> di;
    if (dw.alloc(n) || dx.alloc(m) || db.alloc(m) || dws.alloc(m) || dr.alloc(m) || di.alloc(m)) return 1;
    CK(cudaMemcpy(dw, w, (size_t)n * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dx, x, (size_t)m * 8, cudaMemcpyHostToDevice));
    vg::choose_tap_kernel<<<(m + 3) / 4, 128>>>(dw, n, dx, m, skip, small, di, db, dws, dr);
    CK(cudaGetLastError());
    CK(cudaMemcpy(idx, di, (size_t)m * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(before, db, (size_t)m * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(wsel, dws, (size_t)m * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(resid, dr, (size_t)m * 8, cudaMemcpyDeviceToHost));
    return 0;
}
