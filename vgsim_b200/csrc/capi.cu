// C ABI of libvgsim_b200.so (include/vgsim_b200.h): host-side plumbing around the sm_100a kernels.
#include <cuda_runtime.h>
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>
#include <vector>
#include "../../include/vgsim_b200.h"
#include "common.cuh"
#include "host.h"
#include "param_blob.cuh"

using namespace vg;

static thread_local std::string g_err;
int vg::fail(const std::string &m) {
    g_err = m;
    return 1;
}

extern "C" {

const char *vgsim_last_error(void) { return g_err.c_str(); }
int vgsim_version(void) { return 100; }

int vgsim_create(int sites, int K, int S, int n_replicates, int n_param_points, int device, vgsim_handle *out) {
    if (sites < 0 || sites > 9) return fail("number of sites must be in [0, 9] (18-bit haplotype field of the packed event)");
    if (K < 1 || K > 4096) return fail("populations number must be in [1, 4096]");
    if (S < 1 || S > 64) return fail("number of susceptible groups must be in [1, 64]");
    if (n_replicates < 1 || n_param_points < 1) return fail("replicates and parameter points must be >= 1");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(std::string("no CUDA device available (the vgsim_b200 hot path has no CPU fallback): ") +
                    cudaGetErrorString(e));
    if (device < 0) CK(cudaGetDevice(&device));
    CK(cudaSetDevice(device));
    std::unique_ptr<vgsim_handle_s, int (*)(vgsim_handle)> owner(new vgsim_handle_s(), vgsim_destroy);  // on failure
    vgsim_handle_s *h = owner.get();
    h->device = device;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    h->num_sms = prop.multiProcessorCount;
    h->D = make_dims(sites, K, S);
    const Dims &D = h->D;
    if ((long long)K * (K - 1) * S * D.H + (long long)K * D.PD > 2000000000LL)
        return fail("too many reaction channels for 32-bit channel indices");
    h->R = n_replicates;
    h->n_pp = n_param_points;
    h->hp.resize(n_param_points);
    h->rep_pp_host.assign(n_replicates, 0);
    for (int i = 0; i < Handle::NTIMER; i++) {
        CK(cudaEventCreate(&h->ev_ring0[i]));
        CK(cudaEventCreate(&h->ev_ring1[i]));
    }
    DevState &st = h->st;
    memset(&st, 0, sizeof(st));
    st.D = D;
    st.R = n_replicates;
    st.n_pp = n_param_points;
    size_t R = n_replicates;
    double *params;
    int *rep_pp;
    uint64_t *seeds;
    if (dalloc(h, &params, (size_t)n_param_points * D.blob) || dalloc(h, &rep_pp, R) || dalloc(h, &seeds, R) ||
        dalloc(h, &st.I, R * K * D.H) || dalloc(h, &st.Sx, R * K * S) || dalloc(h, &st.initI, R * K * D.H) ||
        dalloc(h, &st.initSx, R * K * S) || dalloc(h, &st.cd, R * K) || dalloc(h, &st.lock, R * K) ||
        dalloc(h, &st.eff, R * K * K) || dalloc(h, &st.ceff, R * K) || dalloc(h, &st.maxEBM, R * K) ||
        dalloc(h, &st.time, R) || dalloc(h, &st.counters, R * NCOUNT) || dalloc(h, &st.epoch, R) ||
        dalloc(h, &st.err, R) || dalloc(h, &st.loc_n, R) || dalloc(h, &st.ev_base, R) || dalloc(h, &st.dense_base, R) ||
        dalloc(h, &st.sp_n, R) || dalloc(h, &st.rate_tot, 2 * R))
        return 1;
    st.params = params;
    st.rep_pp = rep_pp;
    st.seeds = seeds;
    st.loc_cap = 64 + 16 * K;  // a deme flips its lockdown on and off a few times per wave; overflow sets a sticky error bit
    if (dalloc(h, &st.loc_sp, R * st.loc_cap) || dalloc(h, &st.loc_t, R * st.loc_cap) ||
        dalloc(h, &h->summaries, R * VGSIM_NSUMMARY) || dalloc(h, &h->tau_order, 2 * R) || dalloc(h, &h->work, 4))
        return 1;
    // default state: everyone susceptible in group 0, sizes 1e6 (reference :201-204)
    std::vector<long long> Sx(R * K * S, 0);
    for (size_t i = 0; i < R * K; i++) Sx[i * S] = 1000000;
    CK(cudaMemcpyAsync(st.Sx, Sx.data(), Sx.size() * 8, cudaMemcpyHostToDevice, h->stream));
    std::vector<uint64_t> sd(R);
    for (size_t i = 0; i < R; i++) sd[i] = i;
    CK(cudaMemcpyAsync(seeds, sd.data(), R * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    *out = owner.release();
    return 0;
}

int vgsim_destroy(vgsim_handle h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    for (void *p : h->allocs) cudaFree(p);
    h->allocs.clear();
    for (int i = 0; i < Handle::NTIMER; i++) {
        if (h->ev_ring0[i]) cudaEventDestroy(h->ev_ring0[i]);
        if (h->ev_ring1[i]) cudaEventDestroy(h->ev_ring1[i]);
    }
    delete h;
    return 0;
}

int vgsim_set_stream(vgsim_handle h, void *cuda_stream) {
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    h->stream = (cudaStream_t)cuda_stream;
    return 0;
}

int vgsim_set_seeds(vgsim_handle h, const uint64_t *seeds) {
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync((void *)h->st.seeds, seeds, (size_t)h->R * 8, cudaMemcpyHostToDevice, h->stream));
    HOST_SYNC(h);
    return 0;
}

__global__ void seed_cd_kernel(DevState st) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= st.R * st.D.K) return;
    int r = i / st.D.K, p = i - r * st.D.K;
    st.cd[i] = st.params[(size_t)st.rep_pp[r] * st.D.blob + st.D.o_cd0 + p];
}

int vgsim_set_replicate_params(vgsim_handle h, const int32_t *map) {
    for (int r = 0; r < h->R; r++)
        if (map[r] < 0 || map[r] >= h->n_pp) return fail("replicate_to_param entry out of range");
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync((void *)h->st.rep_pp, map, (size_t)h->R * 4, cudaMemcpyHostToDevice, h->stream));
    h->rep_pp_host.assign(map, map + h->R);
    // Before the first simulation the live contact density of every replicate follows its (new) parameter point, so the
    // order of vgsim_upload_params and vgsim_set_replicate_params does not matter; afterwards it is run state (a deme
    // may be in lockdown) and is left alone.
    if (!h->st.first_simulation) {
        seed_cd_kernel<<<(h->R * h->D.K + 255) / 256, 256, 0, h->stream>>>(h->st);
        h->launches++;
        CK(cudaGetLastError());
    }
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

static Src<long long> src_view(const HostParams &P) {
    Src<long long> v;
    v.b = P.b.data(), v.d = P.d.data(), v.s = P.s.data(), v.mRate = P.mRate.data(), v.hapMutType = P.hapMutType.data();
    v.sigma = P.sigma.data(), v.T = P.T.data(), v.m = P.m.data(), v.cd = P.cd.data(), v.cdBefore = P.cdBefore.data();
    v.cdAfter = P.cdAfter.data(), v.startLD = P.startLD.data(), v.endLD = P.endLD.data(), v.sm = P.sm.data();
    v.suscType = P.suscType.data(), v.sizes = P.sizes.data();
    return v;
}

// The fp64 fields of HostParams in vgsim_upload_params order (nullptr: the int64 fields suscType and sizes).
static void double_fields(HostParams &P, std::vector<double> *f[NSRC]) {
    std::vector<double> *t[NSRC] = {&P.b, &P.d, &P.s, &P.mRate, &P.hapMutType, &P.sigma, nullptr, &P.T,
                                    &P.m, &P.cd, &P.cdBefore, &P.cdAfter, &P.startLD, &P.endLD, &P.sm, nullptr};
    std::copy(t, t + NSRC, f);
}

static std::vector<double> flatten(const Dims &D, HostParams &P) {
    std::vector<double> *f[NSRC];
    double_fields(P, f);
    std::vector<double> out;
    out.reserve(src_off(D, NSRC));
    for (int k = 0; k < NSRC; k++) {
        if (f[k])
            out.insert(out.end(), f[k]->begin(), f[k]->end());
        else
            for (long long x : k == F_SUSC ? P.suscType : P.sizes) out.push_back((double)x);
    }
    return out;
}

// Host record of parameter point pp; a grid point's is rebuilt from its grid's base and patches at the first use.
static HostParams &host_params(Handle *h, int pp) {
    HostParams &P = h->hp[pp];
    if (!P.grid) return P;
    const ParamGrid &g = *P.grid;
    const Dims &D = h->D;
    std::vector<double> src(g.base);
    long long start = 0, stride = 1;
    for (int len : g.axis_len) stride *= len;
    for (int len : g.axis_len) {
        stride /= len;
        const long long j = start + (P.grid_point / stride) % len;
        for (long long k = g.off[j]; k < g.off[j + 1]; k++) src[g.idx[k]] = g.val[k];
        start += len;
    }
    std::vector<double> *f[NSRC];
    double_fields(P, f);
    for (int k = 0; k < NSRC; k++) {
        const double *a = src.data() + src_off(D, k), *e = a + src_len(D, k);
        if (f[k])
            f[k]->assign(a, e);
        else
            (k == F_SUSC ? P.suscType : P.sizes).assign(a, e);
    }
    P.grid.reset();
    return P;
}

__global__ void set_cd_kernel(DevState st, int pp, const int *mask, const double *cdv) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= st.R * st.D.K) return;
    int r = i / st.D.K, p = i - r * st.D.K;
    if (st.rep_pp[r] == pp && mask[p]) st.cd[i] = cdv[p];
}

int vgsim_upload_params(vgsim_handle h, int pp, const double *b, const double *d, const double *s,
                        const double *mRate, const double *hapMutType, const double *sigma, const int64_t *suscType,
                        const double *T, const double *m, const double *contact_density, const double *cd_before,
                        const double *cd_after, const double *startLD, const double *endLD,
                        const double *sampling_multiplier, const int64_t *sizes, const int32_t *cd_reset_mask) {
    if (pp < 0 || pp >= h->n_pp) return fail("parameter point out of range");
    CK(cudaSetDevice(h->device));
    const Dims &D = h->D;
    const int K = D.K, H = D.H, S = D.S, U = D.U;
    HostParams &P = host_params(h, pp);
    auto cp = [](std::vector<double> &v, const double *src, size_t n, double dflt) {
        if (src)
            v.assign(src, src + n);
        else if (v.size() != n)
            v.assign(n, dflt);
    };
    cp(P.b, b, H, 2.0);
    cp(P.d, d, H, 1.0);
    cp(P.s, s, H, 0.01);
    cp(P.mRate, mRate, (size_t)H * U, 0.01);
    cp(P.hapMutType, hapMutType, (size_t)H * U * 3, 1.0);
    if (sigma)
        P.sigma.assign(sigma, sigma + (size_t)H * S);
    else if (P.sigma.size() != (size_t)H * S) {
        P.sigma.assign((size_t)H * S, 0.0);
        for (int i = 0; i < H; i++) P.sigma[(size_t)i * S] = 1.0;
    }
    if (suscType)
        P.suscType.assign(suscType, suscType + H);
    else if (P.suscType.size() != (size_t)H)
        P.suscType.assign(H, 0);
    cp(P.T, T, (size_t)S * S, 0.0);
    cp(P.m, m, (size_t)K * K, 0.0);
    cp(P.cd, contact_density, K, 1.0);
    cp(P.cdBefore, cd_before, K, 1.0);
    cp(P.cdAfter, cd_after, K, 0.0);
    cp(P.startLD, startLD, K, 1.0);
    cp(P.endLD, endLD, K, 1.0);
    cp(P.sm, sampling_multiplier, K, 1.0);
    if (sizes)
        P.sizes.assign(sizes, sizes + K);
    else if (P.sizes.size() != (size_t)K)
        P.sizes.assign(K, 1000000);
    for (int i = 0; i < H; i++)
        if (P.suscType[i] < 0 || P.suscType[i] >= S) return fail("susceptibility type out of range");
    for (int p = 0; p < K; p++)
        if (P.sizes[p] <= 0 || P.sizes[p] > 2147483647LL)
            return fail("population sizes must be in [1, 2^31-1] (compartment counts are int32 on the device)");

    std::vector<double> blob(D.blob, 0.0);
    const Src<long long> src = src_view(P);
    double maxB = 0.0;
    for (int i = 0; i < H; i++) maxB = std::max(maxB, blob_hap(D, src, blob.data(), i));
    for (int s1 = 0; s1 < S; s1++) blob_group(D, src, blob.data(), s1);
    for (int p = 0; p < K; p++) blob_deme(D, src, blob.data(), p);
    blob[D.o_maxB] = maxB;
    CK(cudaMemcpyAsync((void *)(h->st.params + (size_t)pp * D.blob), blob.data(), (size_t)D.blob * 8,
                       cudaMemcpyHostToDevice, h->stream));
    // live contact density: first upload sets every deme, later uploads only the masked ones
    std::vector<int> mask(K, 1);
    if (P.uploaded && cd_reset_mask)
        for (int p = 0; p < K; p++) mask[p] = cd_reset_mask[p] != 0;
    else if (P.uploaded && !contact_density)
        std::fill(mask.begin(), mask.end(), 0);
    Scratch<int> dmask;
    Scratch<double> dcd;
    if (dmask.alloc(K) || dcd.alloc(K)) return 1;
    CK(cudaMemcpyAsync(dmask, mask.data(), K * 4, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(dcd, P.cd.data(), K * 8, cudaMemcpyHostToDevice, h->stream));
    int n = h->R * K;
    set_cd_kernel<<<(n + 255) / 256, 256, 0, h->stream>>>(h->st, pp, dmask, dcd);
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    P.uploaded = true;
    return 0;
}

int vgsim_upload_param_grid(vgsim_handle h, int base_pp, int n_axes, const int32_t *axis_len, const int64_t *patch_off,
                            const int64_t *patch_idx, const double *patch_val, int64_t first_point, int dst_pp0,
                            int n_points) {
    if (base_pp < 0 || base_pp >= h->n_pp) return fail("base parameter point out of range");
    if (n_points < 1 || dst_pp0 < 0 || dst_pp0 > h->n_pp - n_points) return fail("destination parameter points out of range");
    if (n_axes < 0) return fail("number of axes must be >= 0");
    HostParams &B = host_params(h, base_pp);
    if (!B.uploaded) return fail("base parameter point was not uploaded (vgsim_upload_params)");
    const Dims &D = h->D;
    auto g = std::make_shared<ParamGrid>();
    long long total = 1, nv = 0;
    for (int a = 0; a < n_axes; a++) {
        if (axis_len[a] < 1) return fail("axis lengths must be >= 1");
        if (total > (1LL << 62) / axis_len[a]) return fail("the grid has more than 2^62 points");
        total *= axis_len[a];
        nv += axis_len[a];
    }
    if (first_point < 0 || first_point > total - n_points) return fail("grid points out of range");
    if (patch_off[0] != 0) return fail("patch offsets must start at 0");
    for (long long j = 0; j < nv; j++)
        if (patch_off[j + 1] < patch_off[j]) return fail("patch offsets must not decrease");
    const long long nsrc = src_off(D, NSRC), ne = patch_off[nv];
    for (long long k = 0; k < ne; k++)
        if (patch_idx[k] < 0 || patch_idx[k] >= nsrc) return fail("patch index out of range");
    g->base = flatten(D, B);
    g->axis_len.assign(axis_len, axis_len + n_axes);
    g->off.assign(patch_off, patch_off + nv + 1);
    g->idx.assign(patch_idx, patch_idx + ne);
    g->val.assign(patch_val, patch_val + ne);
    CK(cudaSetDevice(h->device));
    GridArgs a;
    a.n_axes = n_axes;
    a.first_point = first_point;
    a.dst_pp0 = dst_pp0;
    a.n_points = n_points;
    a.nslots = param_grid_slots(h->num_sms, n_points);
    Scratch<double> dbase, dval, dslots;
    Scratch<int> dlen, derr, dflag;
    Scratch<long long> doff, didx;
    if (dbase.alloc(nsrc) || dlen.alloc(n_axes) || doff.alloc(nv + 1) || didx.alloc(ne) || dval.alloc(ne) ||
        dslots.alloc((size_t)a.nslots * nsrc) || derr.alloc(n_points) || dflag.alloc(1))
        return 1;
    CK(cudaMemcpyAsync(dbase, g->base.data(), nsrc * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(dlen, axis_len, (size_t)n_axes * 4, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(doff, patch_off, (nv + 1) * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(didx, patch_idx, ne * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(dval, patch_val, ne * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemsetAsync(dflag, 0, 4, h->stream));
    a.base = dbase, a.axis_len = dlen, a.off = doff, a.idx = didx, a.val = dval, a.slots = dslots, a.err = derr;
    a.flag = dflag;
    cudaError_t e = launch_param_grid(h->st, a, h->stream);
    if (e != cudaSuccess) return fail(std::string("parameter grid kernels: ") + cudaGetErrorString(e));
    h->launches += 3;
    std::vector<int> err(n_points);
    CK(cudaMemcpyAsync(err.data(), derr, (size_t)n_points * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < n_points; i++) {
        if (!err[i]) continue;
        const int b = err[i];
        return fail("parameter grid point " + std::to_string(first_point + i) + ": " +
                    (b & GRID_ERR_SUSC ? "susceptibility type out of range"
                     : b & GRID_ERR_SIZES ? "population sizes must be in [1, 2^31-1]"
                     : b & GRID_ERR_MIG_SUM ? "the migration probabilities out of a population sum to more than 1"
                                            : "a population's probability of staying (diagonal of the migration matrix) "
                                              "must be more than 1e-15"));
    }
    for (int i = 0; i < n_points; i++) {
        HostParams &P = h->hp[dst_pp0 + i];
        P = HostParams();
        P.uploaded = true;
        P.grid = g;
        P.grid_point = first_point + i;
    }
    return 0;
}

int vgsim_get_params(vgsim_handle h, int pp, double *blob_out) {
    if (pp < 0 || pp >= h->n_pp) return fail("parameter point out of range");
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(blob_out, h->st.params + (size_t)pp * h->D.blob, (size_t)h->D.blob * 8, cudaMemcpyDeviceToHost,
                       h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int vgsim_set_state(vgsim_handle h, const int64_t *Sx, const int64_t *I) {
    CK(cudaSetDevice(h->device));
    const Dims &D = h->D;
    if (Sx) CK(cudaMemcpyAsync(h->st.Sx, Sx, (size_t)h->R * D.K * D.S * 8, cudaMemcpyHostToDevice, h->stream));
    if (I) CK(cudaMemcpyAsync(h->st.I, I, (size_t)h->R * D.K * D.H * 8, cudaMemcpyHostToDevice, h->stream));
    HOST_SYNC(h);
    return 0;
}

int vgsim_set_state_dev(vgsim_handle h, const int64_t *dSx, const int64_t *dI) {
    CK(cudaSetDevice(h->device));
    const Dims &D = h->D;
    if (dSx) CK(cudaMemcpyAsync(h->st.Sx, dSx, (size_t)h->R * D.K * D.S * 8, cudaMemcpyDeviceToDevice, h->stream));
    if (dI) CK(cudaMemcpyAsync(h->st.I, dI, (size_t)h->R * D.K * D.H * 8, cudaMemcpyDeviceToDevice, h->stream));
    return 0;
}

int vgsim_state_dev(vgsim_handle h, void **dSx, void **dI) {
    if (dSx) *dSx = h->st.Sx;
    if (dI) *dI = h->st.I;
    return 0;
}

__global__ void reset_kernel(DevState st) {  // one warp per replicate
    const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (r >= st.R) return;
    const int K = st.D.K;
    for (int i = lane; i < NCOUNT; i += 32) st.counters[(size_t)r * NCOUNT + i] = 0;
    for (int p = lane; p < K; p += 32) {
        st.lock[(size_t)r * K + p] = 0;
        st.cd[(size_t)r * K + p] = st.params[(size_t)st.rep_pp[r] * st.D.blob + st.D.o_cd0 + p];
    }
    if (lane == 0) {
        st.time[r] = 0.0;
        st.epoch[r] = 0;
        st.err[r] = 0;
        st.loc_n[r] = 0;
        st.ev_base[r] = 0;
        st.dense_base[r] = 0;
        st.sp_n[r] = 0;
    }
}

int vgsim_set_async(vgsim_handle h, int on) {
    h->async_host = on != 0;
    return 0;
}

int vgsim_wait(vgsim_handle h) {
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int vgsim_reset(vgsim_handle h) {
    CK(cudaSetDevice(h->device));
    DevState &st = h->st;
    const size_t R = h->R;
    // one kernel: counters, clocks, epochs, error bits, lockdown records / flags, recycled-row counts to zero; live contact
    // density back to the uploaded value of each replicate's parameter point (device side: no host sync)
    reset_kernel<<<((int)R * 32 + 255) / 256, 256, 0, h->stream>>>(st);
    h->launches++;
    CK(cudaGetLastError());
    h->ev_bound = 0;
    h->leap_bound = 0;
    h->dense_bound = 0;
    st.first_simulation = 0;
    h->gen.valid = false;
    return 0;
}

__global__ void recycle_log_kernel(DevState st) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= st.R) return;
    st.ev_base[r] += st.counters[(size_t)r * NCOUNT + C_EVPTR];
    st.counters[(size_t)r * NCOUNT + C_EVPTR] = 0;
    st.counters[(size_t)r * NCOUNT + C_LEAPS] = 0;
    st.dense_base[r] = 0;
    st.sp_n[r] = 0;
}

int vgsim_recycle_log(vgsim_handle h) {
    CK(cudaSetDevice(h->device));
    recycle_log_kernel<<<(h->R + 255) / 256, 256, 0, h->stream>>>(h->st);
    h->launches++;
    CK(cudaGetLastError());
    h->ev_bound = 0;
    h->leap_bound = 0;
    h->dense_bound = 0;
    h->gen.valid = false;
    return 0;
}

int vgsim_get_state(vgsim_handle h, int64_t *Sx, int64_t *I, double *cd, int64_t *lock) {
    CK(cudaSetDevice(h->device));
    const Dims &D = h->D;
    if (Sx) CK(cudaMemcpyAsync(Sx, h->st.Sx, (size_t)h->R * D.K * D.S * 8, cudaMemcpyDeviceToHost, h->stream));
    if (I) CK(cudaMemcpyAsync(I, h->st.I, (size_t)h->R * D.K * D.H * 8, cudaMemcpyDeviceToHost, h->stream));
    if (cd) CK(cudaMemcpyAsync(cd, h->st.cd, (size_t)h->R * D.K * 8, cudaMemcpyDeviceToHost, h->stream));
    std::vector<int> lk;
    if (lock) {
        lk.resize((size_t)h->R * D.K);
        CK(cudaMemcpyAsync(lk.data(), h->st.lock, lk.size() * 4, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));  // converted on the host below
    }
    HOST_SYNC(h);
    if (lock)
        for (size_t i = 0; i < lk.size(); i++) lock[i] = lk[i];
    return 0;
}

}  // extern "C"

// grow a per-replicate 2-D device buffer [R][old_cap*w] -> [R][new_cap*w], keeping the first `keep` rows
template <class T>
static int grow2d(Handle *h, T **buf, long long old_cap, long long new_cap, long long keep, size_t w) {
    T *nb;
    if (dalloc(h, &nb, (size_t)h->R * new_cap * w)) return 1;
    if (*buf && keep > 0)
        CK(cudaMemcpy2DAsync(nb, new_cap * w * sizeof(T), *buf, old_cap * w * sizeof(T), keep * w * sizeof(T), h->R,
                             cudaMemcpyDeviceToDevice, h->stream));
    if (*buf) {
        CK(cudaStreamSynchronize(h->stream));
        dfree(h, *buf);
    }
    *buf = nb;
    return 0;
}

static int ensure_ev_cap(Handle *h, long long need) {
    DevState &st = h->st;
    if (need <= st.ev_cap) return 0;
    long long nc = std::max(need, std::min(st.ev_cap + st.ev_cap / 2, need + (1LL << 16)));  // blocked runs: not one regrow per block
    nc = (nc + 1) & ~1LL;  // even: every replicate's rows start 16-byte aligned for the vector copies of vgsim_resample
    if (grow2d(h, &st.ev_time, st.ev_cap, nc, h->ev_bound, 1)) return 1;
    if (grow2d(h, &st.ev_desc, st.ev_cap, nc, h->ev_bound, 1)) return 1;
    st.ev_cap = nc;
    return 0;
}
static int ensure_leap_cap(Handle *h, long long need) {  // tau_tt and the archive's offsets: all leaps of a replicate
    DevState &st = h->st;
    if (need <= st.leap_cap) return 0;
    long long nc = std::max(need, std::min(st.leap_cap + st.leap_cap / 2, need + (1LL << 16)));
    if (grow2d(h, &st.tau_tt, st.leap_cap, nc, h->leap_bound, 2)) return 1;
    // sp_off rows have one more entry than there are leaps: grow with the row strides old_cap + 1 -> new_cap + 1
    {
        int *nb;
        if (dalloc(h, &nb, (size_t)h->R * (nc + 1))) return 1;
        if (st.sp_off && h->leap_bound > 0)
            CK(cudaMemcpy2DAsync(nb, (nc + 1) * 4, st.sp_off, (st.leap_cap + 1) * 4, (h->leap_bound + 1) * 4, h->R,
                                 cudaMemcpyDeviceToDevice, h->stream));
        if (st.sp_off) {
            CK(cudaStreamSynchronize(h->stream));
            dfree(h, st.sp_off);
        }
        st.sp_off = nb;
    }
    st.leap_cap = nc;
    return 0;
}
static int ensure_dense_cap(Handle *h, long long need) {  // dense count rows: the leaps not archived yet
    DevState &st = h->st;
    if (need <= st.dense_cap) return 0;
    if (grow2d(h, &st.tau_counts, st.dense_cap, need, h->dense_bound, (size_t)st.D.Pp)) return 1;
    st.dense_cap = need;
    return 0;
}

// The host-side bounds grow by `iterations` per call (the device decides how many rows a replicate really writes); at a
// point where the stream is idle anyway they are brought back to the true maxima, so that the next call sizes the log
// for what is there plus what it may add -- a direct call of 10^7 iterations that stopped after 1,500 events must not
// make every later call carry 10^7 rows of capacity per replicate.
static int tighten_bounds(Handle *h) {
    const size_t R = h->R;
    std::vector<long long> ctr(R * NCOUNT), base(R);
    CK(cudaMemcpyAsync(ctr.data(), h->st.counters, R * NCOUNT * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(base.data(), h->st.dense_base, R * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    long long ev = 0, lp = 0, dn = 0;
    for (size_t r = 0; r < R; r++) {
        ev = std::max(ev, ctr[r * NCOUNT + C_EVPTR]);
        lp = std::max(lp, ctr[r * NCOUNT + C_LEAPS]);
        dn = std::max(dn, ctr[r * NCOUNT + C_LEAPS] - base[r]);
    }
    h->ev_bound = std::min(h->ev_bound, ev);
    h->leap_bound = std::min(h->leap_bound, lp);
    h->dense_bound = std::min(h->dense_bound, dn);
    return 0;
}

static int prepare(Handle *h, int tau_mode) {
    if (!h->hp[0].uploaded) return fail("parameters were not uploaded (vgsim_upload_params)");
    int first = h->st.first_simulation == 0;
    cudaError_t e = launch_prepare(h->st, first, tau_mode, h->stream);
    if (e != cudaSuccess) return fail(std::string("prepare kernel: ") + cudaGetErrorString(e));
    e = launch_refresh(h->st, h->stream);
    if (e != cudaSuccess) return fail(std::string("refresh kernel: ") + cudaGetErrorString(e));
    h->launches += 2;
    h->st.first_simulation = 1;
    h->gen.valid = false;
    return 0;
}

static void next_timer(Handle *h) {
    h->timer_id++;
    h->ev_k0 = h->ev_ring0[h->timer_id % Handle::NTIMER];
    h->ev_k1 = h->ev_ring1[h->timer_id % Handle::NTIMER];
}

static SimArgs make_args(int64_t iterations, int64_t sample_size, float t, int64_t attempts) {
    SimArgs a;
    a.iterations = iterations;
    a.sample_size = sample_size;
    a.time = t;
    a.has_time = !(t == -1.0f);
    a.attempts = attempts < 1 ? 1 : attempts;
    a.cont = 0;
    return a;
}

// the parameter point every replicate uses, or -1 when they differ
static int uniform_pp(const Handle *h) {
    int u = h->rep_pp_host.empty() ? 0 : h->rep_pp_host[0];
    for (int v : h->rep_pp_host)
        if (v != u) u = -1;
    return u;
}

static int check_tau_shape(const Handle *h) {
    if (tau_fits(h->D, uniform_pp(h))) return 0;
    const Dims &D = h->D;
    return fail("tau-leaping: one replicate of this shape (" + std::to_string(D.U) + " sites = " + std::to_string(D.H) +
                " haplotypes, " + std::to_string(D.K) + " demes, " + std::to_string(D.S) +
                " susceptibility groups) exceeds one SM's shared memory, which the tau kernels need; simulate this shape "
                "with the direct method (vgsim_simulate_direct)");
}

// Warp slices of the large-state direct kernel: one per resident warp (at most 16 per SM) that the batch can use, capped
// so that they take at most half of the device memory that is free (the slices already held count as free).  Grown,
// never shrunk.  nwarps: slices available.
static int dl_slices(Handle *h, const DLLayout &L, int &nwarps) {
    size_t fr = 0, tot = 0;
    CK(cudaMemGetInfo(&fr, &tot));
    const size_t slice = (size_t)L.slice * 8;
    const size_t fit = (fr / 2 + h->dl_slices_n * 8) / slice;
    size_t nw = std::min<size_t>(std::min<size_t>(h->R, (size_t)h->num_sms * 16), fit);
    if (nw < 1)
        return fail("direct kernel: one replicate's state (" + std::to_string(slice >> 20) +
                    " MB of rate trees) exceeds half of the free device memory");
    if (h->dl_slices_n < nw * L.slice) {
        dfree(h, h->dl_slices);
        h->dl_slices = nullptr;
        h->dl_slices_n = 0;
        if (dalloc(h, &h->dl_slices, nw * L.slice)) return 1;
        h->dl_slices_n = nw * L.slice;
    }
    nwarps = (int)(h->dl_slices_n / L.slice < nw ? h->dl_slices_n / L.slice : nw);
    return 0;
}

// the large-state direct kernel runs the shapes whose rate hierarchy does not fit the shared-memory kernel, and every
// shape with vgsim_set_direct_variant bit 0
static bool direct_large(const Handle *h, int upp) { return (h->direct_variant & 1) || !direct_fits_shared(h->D, upp); }

extern "C" {

// one launch of the tau kernel for `iterations` more leaps per replicate.  tau_mode 1: a call of SimulatePopulation_tau
// (FirstInfection when nobody is infectious, :2302-2303); 2: the continuation of one (vgsim_simulate_tau_blocks).
static int tau_call(Handle *h, int64_t iterations, int64_t sample_size, float epidemic_time, int64_t attempts, int tau_mode,
                    bool timed) {
    if (ensure_ev_cap(h, h->ev_bound + iterations) || ensure_leap_cap(h, h->leap_bound + iterations) ||
        ensure_dense_cap(h, h->dense_bound + iterations))
        return 1;
    if (prepare(h, tau_mode)) return 1;
    SimArgs a = make_args(iterations, sample_size, epidemic_time, attempts);
    a.cont = tau_mode == 2;
    if (timed) {
        next_timer(h);
        CK(cudaEventRecord(h->ev_k0, h->stream));
    }
    cudaError_t e = launch_tau(h->st, a, h->stream, h->num_sms, h->tau_variant, uniform_pp(h), h->tau_order,
                                &h->tau_fixed_shape);
    if (e != cudaSuccess) return fail(std::string("tau kernel: ") + cudaGetErrorString(e));
    if (timed) {
        CK(cudaEventRecord(h->ev_k1, h->stream));
        h->ev_valid = true;
    }
    h->launches++;
    h->ev_bound += iterations;
    h->leap_bound += iterations;
    h->dense_bound += iterations;
    return 0;
}

int vgsim_simulate_tau(vgsim_handle h, int64_t iterations, int64_t sample_size, float epidemic_time,
                       int64_t attempts) {
    CK(cudaSetDevice(h->device));
    if (iterations < 0) return fail("iterations must be >= 0");
    if (check_tau_shape(h)) return 1;
    return tau_call(h, iterations, sample_size, epidemic_time, attempts, 1, true);
}

// One SimulatePopulation_tau call of `iterations` leaps run as blocks of `leap_block` leaps; the dense rows of a finished
// block go to the sparse archive before the next block starts, so the dense log never holds more than one block per
// replicate.  The blocks are one call to the reference's eyes: FirstInfection only before the first, the stop conditions
// carry over, the run ends when no replicate used up its block.  The timer pair spans the whole run (tau kernels and
// the archive passes between them).
int vgsim_simulate_tau_blocks(vgsim_handle h, int64_t iterations, int64_t sample_size, float epidemic_time, int64_t attempts,
                              int64_t leap_block) {
    CK(cudaSetDevice(h->device));
    if (iterations < 0) return fail("iterations must be >= 0");
    if (leap_block < 1) return fail("leap_block must be >= 1");
    if (check_tau_shape(h)) return 1;
    // the extinction retry looks at the call's `iterations > 100` (:2331): a block must not hide that from the kernel
    if (iterations > 100 && leap_block <= 100) leap_block = 101;
    next_timer(h);
    cudaEvent_t k0 = h->ev_k0, k1 = h->ev_k1;
    CK(cudaEventRecord(k0, h->stream));
    if (tighten_bounds(h)) return 1;
    int64_t done = 0;
    bool first = true;
    while (done < iterations || first) {
        const int64_t n = std::min<int64_t>(leap_block, iterations - done);
        if (tau_call(h, n, sample_size, epidemic_time, first ? attempts : 1, first ? 1 : 2, false)) return 1;
        first = false;
        done += n;
        if (done >= iterations) break;
        if (tighten_bounds(h)) return 1;
        if (h->dense_bound < n) break;  // no replicate used up its block: every one of them met a stop condition
        if (vgsim_archive_tau_log(h)) return 1;
    }
    // the last block as well: the readers of the log (genealogy replay, curves) then never scan a dense row -- at the world
    // shape the rows of one block are 6-50 GB, the whole archive of the run a few hundred MB
    if (vgsim_archive_tau_log(h)) return 1;
    CK(cudaEventRecord(k1, h->stream));
    h->ev_k0 = k0;
    h->ev_k1 = k1;
    h->ev_valid = true;
    return 0;
}

// The dense rows of every replicate go into the sparse archive (non-zero counts only, ascending channel order, 8 bytes
// each) and the dense capacity is free again: long tau runs proceed in leap blocks without the log growing by
// 4P bytes per leap (4,096 T3 replicates x 1,200 leaps would be 520 GB; 256 world-shape replicates x 2,000 leaps 1 TB).
// Genealogy, curves and the exporters read archived leaps from the archive, the others from their dense rows.
int vgsim_archive_tau_log(vgsim_handle h) {
    CK(cudaSetDevice(h->device));
    DevState &st = h->st;
    if (h->dense_bound == 0 || st.dense_cap == 0) return 0;
    const size_t R = h->R;
    if (h->arch_cnt_cap < R * st.dense_cap) {
        if (h->arch_cnt) dfree(h, h->arch_cnt);
        h->arch_cnt = nullptr;
        h->arch_cnt_cap = 0;
        if (dalloc(h, &h->arch_cnt, R * st.dense_cap)) return 1;
        h->arch_cnt_cap = R * st.dense_cap;
    }
    if (!h->arch_need && dalloc(h, &h->arch_need, R)) return 1;
    int *cnt = h->arch_cnt, *need = h->arch_need;
    cudaError_t e = launch_archive_count(st, cnt, need, h->stream);
    h->launches += 2;
    std::vector<int> hneed(R), hn(R);
    if (e == cudaSuccess) e = cudaMemcpyAsync(hneed.data(), need, R * 4, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(hn.data(), st.sp_n, R * 4, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) return fail(std::string("archive (count): ") + cudaGetErrorString(e));
    long long want = 0, keep = 0;
    for (size_t r = 0; r < R; r++) {
        want = std::max(want, (long long)hn[r] + hneed[r]);
        keep = std::max(keep, (long long)hn[r]);
    }
    if (want > 2147483647LL) return fail("archive: more than 2^31 entries in one replicate");
    if (want > st.sp_cap) {
        // room for the blocks to come: the archive of a growing epidemic grows faster than linearly
        long long nc = std::max(2 * want, (long long)1024);
        if (grow2d(h, &st.sp_ent, st.sp_cap, nc, keep, 1)) return 1;
        st.sp_cap = nc;
    }
    e = launch_archive_write(st, cnt, need, h->stream);
    h->launches += 2;
    if (e != cudaSuccess) return fail(std::string("archive (write): ") + cudaGetErrorString(e));
    h->dense_bound = 0;
    return 0;
}

int vgsim_archive_stats(vgsim_handle h, int64_t *entries_total, int64_t *entries_max, int64_t *leaps_archived) {
    CK(cudaSetDevice(h->device));
    const size_t R = h->R;
    std::vector<int> n(R);
    std::vector<long long> base(R);
    CK(cudaMemcpyAsync(n.data(), h->st.sp_n, R * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(base.data(), h->st.dense_base, R * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    int64_t tot = 0, mx = 0, la = 0;
    for (size_t r = 0; r < R; r++) {
        tot += n[r];
        mx = std::max<int64_t>(mx, n[r]);
        la += base[r];
    }
    if (entries_total) *entries_total = tot;
    if (entries_max) *entries_max = mx;
    if (leaps_archived) *leaps_archived = la;
    return 0;
}

int vgsim_simulate_direct(vgsim_handle h, int64_t iterations, int64_t sample_size, float epidemic_time,
                          int64_t attempts) {
    CK(cudaSetDevice(h->device));
    if (iterations < 0) return fail("iterations must be >= 0");
    if (ensure_ev_cap(h, h->ev_bound + iterations)) return 1;
    if (prepare(h, 0)) return 1;
    SimArgs a = make_args(iterations, sample_size, epidemic_time, attempts);
    const int upp = uniform_pp(h);
    const bool large = direct_large(h, upp);
    const DLLayout L = dl_layout(h->D);
    int nwarps = 0;
    if (large && dl_slices(h, L, nwarps)) return 1;
    next_timer(h);
    CK(cudaEventRecord(h->ev_k0, h->stream));
    cudaError_t e = large ? launch_direct_large(h->st, a, L, h->dl_slices, nwarps, h->num_sms, h->stream, h->work)
                          : launch_direct(h->st, a, h->stream, h->num_sms, upp, h->work);
    if (e != cudaSuccess) return fail(std::string("direct kernel: ") + cudaGetErrorString(e));
    CK(cudaEventRecord(h->ev_k1, h->stream));
    h->ev_valid = true;
    h->launches++;
    h->ev_bound += iterations;
    return 0;
}

int vgsim_synchronize(vgsim_handle h) {
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    if (tighten_bounds(h)) return 1;
    std::vector<int> err(h->R);
    CK(cudaMemcpy(err.data(), h->st.err, (size_t)h->R * 4, cudaMemcpyDeviceToHost));
    int all = 0;
    for (int v : err) all |= v;
    if (all) {
        g_err = "device error flags: " + std::to_string(all);
        if (all & ERR_ZERO_WEIGHT) g_err += " [zero weight sampled]";
        if (all & ERR_LOCKDOWN_OVERFLOW) g_err += " [lockdown record overflow]";
        if (all & ERR_ARENA) g_err += " [lineage arena exhausted]";
        if (all & ERR_STREAM) g_err += " [injected uniform stream exhausted]";
        if (all & ERR_CLAMPED) g_err += " [tau-log coalescences clamped]";
        if (all & ERR_COUNT_OVERFLOW) g_err += " [compartment count overflow]";
        if (all & ERR_BADLOG) g_err += " [bad event log]";
        if (all & ERR_TAU_STUCK) g_err += " [tau leap infeasible after 80 halvings]";
        if (all & ERR_SIDE_TABLE) g_err += " [genealogy side table overflow]";
        // reported once: later synchronize calls must not raise (or warn) again for the same condition
        CK(cudaMemsetAsync(h->st.err, 0, (size_t)h->R * 4, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    return all;
}

int64_t vgsim_prop_num(vgsim_handle h) { return h->D.P; }

int vgsim_propensities(vgsim_handle h, int replicate, double *out, double *dI, double *dS, double *tau) {
    CK(cudaSetDevice(h->device));
    if (check_replicate(h, replicate)) return 1;
    if (!h->hp[0].uploaded) return fail("parameters were not uploaded");
    if (check_tau_shape(h)) return 1;
    const Dims &D = h->D;
    // like PrintPropensities: UpdateAllRates on the CURRENT state (no FirstInfection, no lockdown check)
    cudaError_t e = launch_refresh(h->st, h->stream);
    if (e != cudaSuccess) return fail(std::string("refresh kernel: ") + cudaGetErrorString(e));
    Scratch<double> buf;
    size_t n = (size_t)D.P + (size_t)D.K * D.H + (size_t)D.K * D.S + 1;
    if (buf.alloc(n)) return 1;
    e = launch_propensities(h->st, replicate, buf, buf + D.P, buf + D.P + D.K * D.H, buf + n - 1, h->stream);
    h->launches += 2;
    if (e != cudaSuccess) return fail(std::string("propensity kernel: ") + cudaGetErrorString(e));
    std::vector<double> hb(n);
    CK(cudaMemcpyAsync(hb.data(), buf, n * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (out) memcpy(out, hb.data(), (size_t)D.P * 8);
    if (dI) memcpy(dI, hb.data() + D.P, (size_t)D.K * D.H * 8);
    if (dS) memcpy(dS, hb.data() + D.P + D.K * D.H, (size_t)D.K * D.S * 8);
    if (tau) *tau = hb[n - 1];
    return 0;
}

int vgsim_rates(vgsim_handle h, int replicate, double *A, double *eff, double *maxEBM, double *ev, double *hapPopRate,
                double *popRate, double *migPopRate, double *totals) {
    CK(cudaSetDevice(h->device));
    if (check_replicate(h, replicate)) return 1;
    if (!h->hp[0].uploaded) return fail("parameters were not uploaded");
    const Dims &D = h->D;
    const int K = D.K, H = D.H;
    cudaError_t e = launch_refresh(h->st, h->stream);
    if (e != cudaSuccess) return fail(std::string("refresh kernel: ") + cudaGetErrorString(e));
    size_t n = (size_t)K * H * 4 + (size_t)K * H + K + K + 2;
    Scratch<double> buf;
    if (buf.alloc(n)) return 1;
    Scratch<double> slice;
    if (direct_large(h, -1)) {  // the large-state kernel's trees, built as that kernel builds them
        const DLLayout L = dl_layout(D);
        if (slice.alloc(L.slice)) return 1;
        e = launch_rates_large(h->st, L, slice, replicate, buf, buf + K * H * 4, buf + K * H * 5, buf + K * H * 5 + K,
                               buf + K * H * 5 + 2 * K, h->stream);
    } else {
        e = launch_rates_tap(h->st, replicate, buf, buf + K * H * 4, buf + K * H * 5, buf + K * H * 5 + K,
                             buf + K * H * 5 + 2 * K, h->stream);
    }
    h->launches += 2;
    if (e != cudaSuccess) return fail(std::string("rates kernel: ") + cudaGetErrorString(e));
    std::vector<double> hb(n);
    CK(cudaMemcpyAsync(hb.data(), buf, n * 8, cudaMemcpyDeviceToHost, h->stream));
    int pp;
    CK(cudaMemcpyAsync(&pp, h->st.rep_pp + replicate, 4, cudaMemcpyDeviceToHost, h->stream));
    if (eff) CK(cudaMemcpyAsync(eff, h->st.eff + (size_t)replicate * K * K, (size_t)K * K * 8, cudaMemcpyDeviceToHost, h->stream));
    if (maxEBM) CK(cudaMemcpyAsync(maxEBM, h->st.maxEBM + (size_t)replicate * K, (size_t)K * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (A) CK(cudaMemcpy(A, h->st.params + (size_t)pp * D.blob + D.o_A, (size_t)K * 8, cudaMemcpyDeviceToHost));
    if (ev) memcpy(ev, hb.data(), (size_t)K * H * 4 * 8);
    if (hapPopRate) memcpy(hapPopRate, hb.data() + K * H * 4, (size_t)K * H * 8);
    if (popRate) memcpy(popRate, hb.data() + K * H * 5, (size_t)K * 8);
    if (migPopRate) memcpy(migPopRate, hb.data() + K * H * 5 + K, (size_t)K * 8);
    if (totals) memcpy(totals, hb.data() + K * H * 5 + 2 * K, 16);
    return 0;
}

int vgsim_get_counters(vgsim_handle h, int64_t *counters, double *current_time) {
    CK(cudaSetDevice(h->device));
    if (counters)
        CK(cudaMemcpyAsync(counters, h->st.counters, (size_t)h->R * NCOUNT * 8, cudaMemcpyDeviceToHost, h->stream));
    if (current_time) CK(cudaMemcpyAsync(current_time, h->st.time, (size_t)h->R * 8, cudaMemcpyDeviceToHost, h->stream));
    HOST_SYNC(h);
    return 0;
}

static int fetch_counters(Handle *h, int r, long long *c) {
    CK(cudaMemcpyAsync(c, h->st.counters + (size_t)r * NCOUNT, NCOUNT * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int vgsim_get_event_log(vgsim_handle h, int r, double *out, int64_t n) {
    CK(cudaSetDevice(h->device));
    if (check_replicate(h, r)) return 1;
    long long c[NCOUNT];
    if (fetch_counters(h, r, c)) return 1;
    if (n != c[C_EVPTR]) return fail("event count mismatch (expected counters[9])");
    if (n == 0) return 0;
    std::vector<double> t(n);
    std::vector<unsigned long long> d(n);
    CK(cudaMemcpyAsync(t.data(), h->st.ev_time + (size_t)r * h->st.ev_cap, n * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(d.data(), h->st.ev_desc + (size_t)r * h->st.ev_cap, n * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const long long P = h->D.P;
    for (int64_t i = 0; i < n; i++) {
        int type, hap, pop, nhap, npop;
        unpack_event(d[i], type, hap, pop, nhap, npop);
        out[i] = t[i];
        out[n + i] = type;
        if (type == EV_MULTITYPE) {
            long long leap = unpack_multi(d[i]);
            out[2 * n + i] = (double)(leap * P);
            out[3 * n + i] = (double)((leap + 1) * P);
            out[4 * n + i] = 0;
            out[5 * n + i] = 0;
        } else {
            out[2 * n + i] = hap;
            out[3 * n + i] = pop;
            out[4 * n + i] = nhap;
            out[5 * n + i] = (type == EV_BIRTH) ? h->D.H : npop;  // BIRTH rows carry the hapNum sentinel (:600)
        }
    }
    return 0;
}

int vgsim_get_tau_log(vgsim_handle h, int r, int64_t leaps, int32_t *counts, double *time_tau) {
    CK(cudaSetDevice(h->device));
    if (check_replicate(h, r)) return 1;
    long long c[NCOUNT];
    if (fetch_counters(h, r, c)) return 1;
    if (leaps != c[C_LEAPS]) return fail("leap count mismatch (expected counters[10])");
    if (leaps == 0) return 0;
    const Dims &D = h->D;
    const DevState &st = h->st;
    long long base = 0;
    CK(cudaMemcpyAsync(&base, st.dense_base + r, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (counts) {
        if (leaps > base)  // the leaps that still have their dense row
            CK(cudaMemcpy2DAsync(counts + (size_t)base * D.P, (size_t)D.P * 4, st.tau_counts + (size_t)r * st.dense_cap * D.Pp,
                                 (size_t)D.Pp * 4, (size_t)D.P * 4, leaps - base, cudaMemcpyDeviceToHost, h->stream));
        if (base > 0) {    // archived leaps: scatter the (channel, count) entries back into dense rows
            std::vector<int> off(base + 1);
            CK(cudaMemcpyAsync(off.data(), st.sp_off + (size_t)r * (st.leap_cap + 1), (base + 1) * 4, cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            std::vector<int2> ent(off[base]);
            if (off[base] > 0)
                CK(cudaMemcpyAsync(ent.data(), st.sp_ent + (size_t)r * st.sp_cap, (size_t)off[base] * 8, cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            memset(counts, 0, (size_t)base * D.P * 4);
            for (long long l = 0; l < base; l++)
                for (int k = off[l]; k < off[l + 1]; k++) counts[(size_t)l * D.P + ent[k].x] = ent[k].y;
        }
    }
    if (time_tau)
        CK(cudaMemcpyAsync(time_tau, st.tau_tt + (size_t)r * st.leap_cap * 2, leaps * 16, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int vgsim_get_multievents(vgsim_handle h, int r, int64_t n, int64_t *num, double *time, int64_t *type, int64_t *hap,
                          int64_t *pop, int64_t *nhap, int64_t *npop) {
    const Dims &D = h->D;
    if (n % D.P != 0) return fail("n must be leaps * P");
    int64_t L = n / D.P;
    std::vector<int32_t> cnt((size_t)n);
    std::vector<double> tt((size_t)L * 2);
    if (vgsim_get_tau_log(h, r, L, cnt.data(), tt.data())) return 1;
    const HostParams &P = host_params(h, h->rep_pp_host[r]);  // suscType of THIS replicate's parameter point (sweeps)
    const int K = D.K, H = D.H, S = D.S, U = D.U;
    int64_t k = 0;
    auto put = [&](int64_t nn, double t, int ty, int a, int b, int c, int d2) {
        if (num) num[k] = nn;
        if (time) time[k] = t;
        if (type) type[k] = ty;
        if (hap) hap[k] = a;
        if (pop) pop[k] = b;
        if (nhap) nhap[k] = c;
        if (npop) npop[k] = d2;
        k++;
    };
    for (int64_t l = 0; l < L; l++) {
        double t = tt[l * 2];
        const int32_t *c = cnt.data() + l * D.P;
        int64_t j = 0;
        for (int sp = 0; sp < K; sp++)
            for (int tp = 0; tp < K; tp++) {
                if (sp == tp) continue;
                for (int sn = 0; sn < S; sn++)
                    for (int hh = 0; hh < H; hh++) put(c[j++], t, EV_MIGRATION, hh, sp, sn, tp);
            }
        for (int p = 0; p < K; p++) {
            for (int ss = 0; ss < S; ss++)
                for (int ts = 0; ts < S; ts++)
                    if (ss != ts) put(c[j++], t, EV_SUSCCHANGE, ss, p, ts, 0);
            for (int hh = 0; hh < H; hh++) {
                int g = (int)P.suscType[hh];
                put(c[j++], t, EV_DEATH, hh, p, g, 0);
                put(c[j++], t, EV_SAMPLING, hh, p, g, 0);
                for (int u = 0; u < U; u++)
                    for (int i = 0; i < 3; i++) put(c[j++], t, EV_MUTATION, hh, p, mutate_hap(hh, u, i, U), 0);
                for (int sn = 0; sn < S; sn++) put(c[j++], t, EV_BIRTH, hh, p, sn, 0);
            }
        }
    }
    return 0;
}

static int lockdown_count(Handle *h, int r, int *n) {
    if (check_replicate(h, r)) return 1;
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(n, h->st.loc_n + r, 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}
int64_t vgsim_num_lockdowns(vgsim_handle h, int r) {
    int n = 0;
    return lockdown_count(h, r, &n) ? -1 : n;
}
int vgsim_get_lockdowns(vgsim_handle h, int r, int64_t *state, int64_t *pop, double *time) {
    int n = 0;
    if (lockdown_count(h, r, &n)) return 1;
    if (n == 0) return 0;
    std::vector<int> sp(n);
    CK(cudaMemcpyAsync(sp.data(), h->st.loc_sp + (size_t)r * h->st.loc_cap, n * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(time, h->st.loc_t + (size_t)r * h->st.loc_cap, n * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < n; i++) {
        state[i] = sp[i] & 1;
        pop[i] = sp[i] >> 1;
    }
    return 0;
}

}  // extern "C"

// Replicates whose replay state does not fit one SM's shared memory replay in device slices: one per resident warp (at
// most 16 per SM), at most half of the free device memory.  Nothing is allocated for a state that fits.
static int replay_slices(Handle *h, size_t slice_bytes, int rep_count, const char *what, Scratch<unsigned char> &slices,
                         int &nslices) {
    nslices = 0;
    if (slice_bytes <= 227 * 1024) return 0;
    size_t fr = 0, tot = 0;
    CK(cudaMemGetInfo(&fr, &tot));
    const size_t nw = std::min<size_t>(std::min<size_t>(rep_count, (size_t)h->num_sms * 16), fr / 2 / slice_bytes);
    if (nw < 1) return fail(std::string(what) + ": one replicate's counts exceed half of the free device memory");
    if (slices.alloc(nw * slice_bytes)) return 1;
    nslices = (int)nw;
    return 0;
}

// A handle-owned device buffer of at least n elements (contents not kept when it grows).
template <class T>
static int ensure_buf(Handle *h, T **buf, size_t &cap, size_t n) {
    if (n <= cap) return 0;
    dfree(h, *buf);
    *buf = nullptr;
    cap = 0;
    if (dalloc(h, buf, n)) return 1;
    cap = n;
    return 0;
}

// The caller's time grid: T >= 1 finite, strictly increasing values, at most max_points of them; copied to the handle's
// grid buffer.
static int upload_grid(Handle *h, const char *what, const double *times, int64_t T, int64_t max_points) {
    const std::string w(what);
    if (T < 1 || !times) return fail(w + ": the time grid needs at least one point");
    if (T > max_points) return fail(w + ": at most " + std::to_string(max_points) + " grid points (got " + std::to_string(T) + ")");
    for (int64_t j = 0; j < T; j++) {
        if (!std::isfinite(times[j])) return fail(w + ": grid time " + std::to_string(j) + " is not finite");
        if (j > 0 && !(times[j] > times[j - 1]))
            return fail(w + ": grid times must be strictly increasing (point " + std::to_string(j) + " is not after point " +
                        std::to_string(j - 1) + ")");
    }
    if (ensure_buf(h, &h->grid_buf, h->grid_cap, (size_t)T)) return 1;
    CK(cudaMemcpyAsync(h->grid_buf, times, (size_t)T * 8, cudaMemcpyHostToDevice, h->stream));
    return 0;
}

extern "C" {

int vgsim_trajectories_dev(vgsim_handle h, const double *times, int64_t T, void **dev_ptr) {
    CK(cudaSetDevice(h->device));
    // grid indices are int on the device, and so is the point count of the launch
    if (upload_grid(h, "trajectories", times, T, 1LL << 30)) return 1;
    const Dims &D = h->D;
    const size_t W = 2 * ((size_t)D.K + D.H);
    if (ensure_buf(h, &h->traj_buf, h->traj_cap, (size_t)h->R * T * W)) return 1;
    Scratch<unsigned char> d_slices;
    int nslices = 0;
    if (replay_slices(h, trajectories_slice_bytes(D), h->R, "trajectories", d_slices, nslices)) return 1;
    next_timer(h);
    CK(cudaEventRecord(h->ev_k0, h->stream));  // vgsim_last_kernel_ms then reports this kernel
    cudaError_t e = launch_trajectories(h->st, h->grid_buf, (int)T, h->traj_buf, h->stream, h->num_sms, d_slices, nslices);
    CK(cudaEventRecord(h->ev_k1, h->stream));
    h->ev_valid = true;
    h->launches++;
    if (e != cudaSuccess) return fail(std::string("trajectories: ") + cudaGetErrorString(e));
    if (nslices) CK(cudaStreamSynchronize(h->stream));  // the slices are freed on return
    if (dev_ptr) *dev_ptr = h->traj_buf;
    return 0;
}

int vgsim_trajectories(vgsim_handle h, const double *times, int64_t T, int64_t *out) {
    if (vgsim_trajectories_dev(h, times, T, nullptr)) return 1;
    const size_t W = 2 * ((size_t)h->D.K + h->D.H);
    CK(cudaMemcpyAsync(out, h->traj_buf, (size_t)h->R * T * W * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int vgsim_lineages_through_time_dev(vgsim_handle h, const double *times, int64_t T, void **dev_ptr) {
    CK(cudaSetDevice(h->device));
    const GenealogyBuffers &G = h->gen;
    if (!G.valid) return fail("lineages through time: no genealogy (call vgsim_genealogy after the last simulation)");
    if (upload_grid(h, "lineages through time", times, T, ltt_max_points())) return 1;
    if (ensure_buf(h, &h->ltt_buf, h->ltt_cap, (size_t)h->R * T)) return 1;
    next_timer(h);
    CK(cudaEventRecord(h->ev_k0, h->stream));
    cudaError_t e = launch_ltt(h->st, G.node_off, G.parent, G.time, G.n_nodes, G.scratch, h->grid_buf, (int)T, h->ltt_buf,
                               h->stream, h->num_sms);
    CK(cudaEventRecord(h->ev_k1, h->stream));
    h->ev_valid = true;
    h->launches++;
    if (e != cudaSuccess) return fail(std::string("lineages through time: ") + cudaGetErrorString(e));
    if (dev_ptr) *dev_ptr = h->ltt_buf;
    return 0;
}

int vgsim_lineages_through_time(vgsim_handle h, const double *times, int64_t T, int64_t *out) {
    if (vgsim_lineages_through_time_dev(h, times, T, nullptr)) return 1;
    CK(cudaMemcpyAsync(out, h->ltt_buf, (size_t)h->R * T * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int vgsim_resample(vgsim_handle h, const int32_t *source) {
    CK(cudaSetDevice(h->device));
    const int R = h->R;
    std::vector<int2> pairs;
    for (int r = 0; r < R; r++) {
        const int s = source[r];
        if (s < 0 || s >= R)
            return fail("resample: replicate " + std::to_string(r) + " copies from " + std::to_string(s) +
                        ": replicate out of range");
    }
    for (int r = 0; r < R; r++) {
        const int s = source[r];
        if (s == r) continue;
        if (source[s] != s)
            return fail("resample: replicate " + std::to_string(r) + " copies from " + std::to_string(s) +
                        ", which copies from " + std::to_string(source[s]) +
                        " (a replicate that is copied from must keep its own run)");
        pairs.push_back(make_int2(r, s));
    }
    // genealogy outputs are dropped as after a simulate call (for the identity map as well); the host bounds are maxima
    // over replicates and stay valid
    h->gen.valid = false;
    if (pairs.empty()) return 0;
    if (ensure_buf(h, &h->resample_pairs, h->resample_cap, pairs.size())) return 1;
    CK(cudaMemcpyAsync(h->resample_pairs, pairs.data(), pairs.size() * sizeof(int2), cudaMemcpyHostToDevice, h->stream));
    int n = 0;
    cudaError_t e = launch_resample(h->st, h->resample_pairs, (int)pairs.size(), h->ev_bound, h->leap_bound, h->dense_bound,
                                    h->stream, &n);
    h->launches += n;
    if (e != cudaSuccess) return fail(std::string("resample kernel: ") + cudaGetErrorString(e));
    return 0;
}

int vgsim_epidemic_curves(vgsim_handle h, int rep_first, int rep_count, int step_num, int64_t *infectious,
                          int64_t *susceptible, int64_t *removed, int64_t *sampled, double *time_points,
                          int32_t *last_point) {
    CK(cudaSetDevice(h->device));
    if (rep_first < 0 || rep_count < 1 || rep_first + rep_count > h->R) return fail("epidemic curves: replicate range out of bounds");
    if (step_num < 1) return fail("epidemic curves: step_num must be >= 1");
    const Dims &D = h->D;
    const size_t np = (size_t)rep_count * (step_num + 1), KH = (size_t)D.K * D.H, KS = (size_t)D.K * D.S;
    // every output the kernel is given is written in full: the buffers need no zero fill
    Scratch<long long> d_inf, d_sus, d_rem, d_smp;
    Scratch<double> d_tp;
    Scratch<int> d_lp;
    if ((infectious && d_inf.alloc(np * KH)) || (susceptible && d_sus.alloc(np * KS)) || (removed && d_rem.alloc(np * KH)) ||
        (sampled && d_smp.alloc(np * KH)) || (time_points && d_tp.alloc(np)) || (last_point && d_lp.alloc(rep_count)))
        return 1;
    Scratch<unsigned char> d_slices;
    int nslices = 0;
    if (replay_slices(h, curves_slice_bytes(D, removed || sampled), rep_count, "epidemic curves", d_slices, nslices)) return 1;
    next_timer(h);
    CK(cudaEventRecord(h->ev_k0, h->stream));  // vgsim_last_kernel_ms then reports this kernel
    cudaError_t e = launch_curves(h->st, rep_first, rep_count, step_num, d_inf, d_sus, d_rem, d_smp, d_tp, d_lp, h->stream,
                                  h->num_sms, d_slices, nslices);
    CK(cudaEventRecord(h->ev_k1, h->stream));
    h->ev_valid = true;
    h->launches++;
    if (e != cudaSuccess) return fail(std::string("epidemic curves: ") + cudaGetErrorString(e));
    if (infectious) CK(cudaMemcpyAsync(infectious, d_inf, np * KH * 8, cudaMemcpyDeviceToHost, h->stream));
    if (susceptible) CK(cudaMemcpyAsync(susceptible, d_sus, np * KS * 8, cudaMemcpyDeviceToHost, h->stream));
    if (removed) CK(cudaMemcpyAsync(removed, d_rem, np * KH * 8, cudaMemcpyDeviceToHost, h->stream));
    if (sampled) CK(cudaMemcpyAsync(sampled, d_smp, np * KH * 8, cudaMemcpyDeviceToHost, h->stream));
    if (time_points) CK(cudaMemcpyAsync(time_points, d_tp, np * 8, cudaMemcpyDeviceToHost, h->stream));
    if (last_point) CK(cudaMemcpyAsync(last_point, d_lp, (size_t)rep_count * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int64_t vgsim_launch_count(vgsim_handle h) { return h->launches; }

int vgsim_debug_tau_phases(vgsim_handle h, uint64_t *out16, int reset) {
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    CK(tau_phase_cycles((unsigned long long *)out16, reset));
    return 0;
}

int vgsim_debug_tau_cta_end(vgsim_handle h, uint64_t *out1024, int reset) {
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    CK(tau_cta_end((unsigned long long *)out1024, reset));
    return 0;
}

int vgsim_set_tau_variant(vgsim_handle h, int variant) {
    if (variant < 0 || variant > 127 || (variant & 12) == 12)
        return fail("tau variant must be 0..127 (bit 0: per-channel draws, bit 1: phase timing, bit 2: force the team kernel, bit 3: force the warp kernel, bit 4: free-running warps, bit 5: unsorted schedule, bit 6: runtime-shape warp kernel)");
    h->tau_variant = variant;
    return 0;
}

int vgsim_tau_fixed_shape(vgsim_handle h) { return h->tau_fixed_shape; }

int vgsim_set_direct_variant(vgsim_handle h, int variant) {
    if (variant < 0 || variant > 1) return fail("direct variant must be 0 or 1 (bit 0: the large-state kernel on every shape)");
    h->direct_variant = variant;
    return 0;
}

int vgsim_last_kernel_ms(vgsim_handle h, float *ms) {
    CK(cudaSetDevice(h->device));
    if (!h->ev_valid) return fail("no hot kernel was launched yet");
    CK(cudaEventSynchronize(h->ev_k1));
    CK(cudaEventElapsedTime(ms, h->ev_k0, h->ev_k1));
    return 0;
}

int64_t vgsim_last_kernel_id(vgsim_handle h) { return h->timer_id; }

int vgsim_kernel_ms(vgsim_handle h, int64_t id, float *ms) {
    CK(cudaSetDevice(h->device));
    if (id < 0 || id > h->timer_id || id + Handle::NTIMER <= h->timer_id) return fail("kernel timer id is not (or no longer) held");
    CK(cudaEventSynchronize(h->ev_ring1[id % Handle::NTIMER]));
    CK(cudaEventElapsedTime(ms, h->ev_ring0[id % Handle::NTIMER], h->ev_ring1[id % Handle::NTIMER]));
    return 0;
}

int vgsim_counters_dev(vgsim_handle h, void **counters, void **current_time) {
    if (counters) *counters = h->st.counters;
    if (current_time) *current_time = h->st.time;
    return 0;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
namespace vg {
// per-replicate summary vector: counters, final time, tree statistics (one warp per replicate).
// Node ids are assigned in creation order going BACKWARD in time (reference src/_BirthDeath.pyx:743-1000),
// so a parent's id is always larger than its children's: depths resolve in one descending sweep.
__global__ void summary_kernel(DevState st, const long long *node_off, const int *parent, const double *time,
                               const int *n_nodes, const int *mut_n, const int *mig_n, int *scratch_all, double *out) {
    const int lane = threadIdx.x & 31, wpc = blockDim.x >> 5;
    for (int r = blockIdx.x * wpc + (threadIdx.x >> 5); r < st.R; r += gridDim.x * wpc) {
        double *o = out + (size_t)r * VGSIM_NSUMMARY;
        for (int i = lane; i < VGSIM_NSUMMARY; i += 32) o[i] = 0.0;
        __syncwarp();
        if (lane < NCOUNT) o[lane] = (double)st.counters[(size_t)r * NCOUNT + lane];
        if (lane == 0) {
            o[12] = st.time[r];
            o[22] = st.rate_tot[2 * (size_t)r];
            o[23] = st.rate_tot[2 * (size_t)r + 1];
        }
        if (!node_off) continue;
        const int n = n_nodes[r];
        if (n == 0) continue;
        const int *par = parent + node_off[r];
        const double *tm = time + node_off[r];
        int *sc = scratch_all + node_off[r];
        double tmin = 1e300, tmax = -1e300, bl = 0.0;
        int roots = 0;
        for (int i = lane; i < n; i += 32) {
            double t = tm[i];
            tmin = fmin(tmin, t);
            tmax = fmax(tmax, t);
            int p = par[i];
            if (p >= 0) bl += t - tm[p]; else roots++;
            sc[i] = 0;
        }
        __syncwarp();
        // children per node (0 = leaf, i.e. created by a SAMPLING row; internal nodes have exactly 2)
        for (int i = lane; i < n; i += 32)
            if (par[i] >= 0) atomicAdd(&sc[par[i]], 1);
        __syncwarp();
        // leaf children per node in bits 2.. : a cherry is an internal node whose two children are leaves
        for (int i = lane; i < n; i += 32)
            if ((sc[i] & 3) == 0 && par[i] >= 0) atomicAdd(&sc[par[i]], 4);
        __syncwarp();
        int cherries = 0;
        for (int i = lane; i < n; i += 32) {
            int v = sc[i];
            if ((v >> 2) == 2) cherries++;
            sc[i] = (v & 3) == 0 ? 1 : 0;  // leaf bit; depth goes to bits 1..
        }
        __syncwarp();
        // depth (edges to the root) by a descending sweep, 32 nodes at a time; dependencies inside a chunk
        // are resolved by lane-to-lane shuffles.  Sackin index = sum of leaf depths.
        long long sackin = 0;
        for (int hi = n; hi > 0; hi -= 32) {
            const int lo = hi - 32;
            const int i = lo + lane;
            const bool live = i >= 0;
            int p = live ? par[i] : -1;
            int depth = 0;
            bool done = !live || p < 0;
            if (live && p >= hi) {
                depth = (sc[p] >> 1) + 1;
                done = true;
            }
            // (a chain inside a chunk is at most 32 long; the bound keeps a malformed tree -- a parent that is not
            // younger than its child -- from spinning for ever: its depths stay 0 and the error bit says so)
            for (int it = 0; it < 33 && __any_sync(0xffffffffu, !done); it++) {
                if (it == 32) {
                    if (lane == 0) st.err[r] |= ERR_BADLOG;
                    break;
                }
                int src = (!done) ? p - lo : lane;
                int pd = __shfl_sync(0xffffffffu, depth, src & 31);
                int pdone = __shfl_sync(0xffffffffu, (int)done, src & 31);
                if (!done && pdone) {
                    depth = pd + 1;
                    done = true;
                }
            }
            if (live) {
                int leaf = sc[i] & 1;
                sc[i] = (depth << 1) | leaf;
                if (leaf) sackin += depth;
            }
            __syncwarp();
        }
        for (int o2 = 16; o2 > 0; o2 >>= 1) {
            tmin = fmin(tmin, __shfl_xor_sync(0xffffffffu, tmin, o2));
            tmax = fmax(tmax, __shfl_xor_sync(0xffffffffu, tmax, o2));
            bl += __shfl_xor_sync(0xffffffffu, bl, o2);
            roots += __shfl_xor_sync(0xffffffffu, roots, o2);
            cherries += __shfl_xor_sync(0xffffffffu, cherries, o2);
            sackin += __shfl_xor_sync(0xffffffffu, sackin, o2);
        }
        if (lane == 0) {
            o[13] = (double)n;
            o[14] = tmax - tmin;   // tree height (latest sample to root)
            o[15] = bl;            // total branch length
            o[16] = (double)roots; // 1 when the genealogy coalesced completely
            o[17] = (double)mut_n[r];
            o[18] = (double)mig_n[r];
            o[19] = tmin;          // time of the root (TMRCA in absolute time)
            o[20] = (double)cherries;
            o[21] = (double)sackin;
        }
    }
}
}  // namespace vg

extern "C" {

int vgsim_summaries_dev(vgsim_handle h, void **dev_ptr) {
    CK(cudaSetDevice(h->device));
    const GenealogyBuffers &G = h->gen;
    int wpc = 4, grid = (h->R + wpc - 1) / wpc;
    if (grid > h->num_sms * 8) grid = h->num_sms * 8;
    summary_kernel<<<grid, wpc * 32, 0, h->stream>>>(h->st, G.valid ? G.node_off : nullptr, G.parent, G.time, G.n_nodes,
                                                      G.mut_n, G.mig_n, G.scratch, h->summaries);
    h->launches++;
    CK(cudaGetLastError());
    if (dev_ptr) *dev_ptr = h->summaries;
    return 0;
}

int vgsim_summaries(vgsim_handle h, double *out) {
    if (vgsim_summaries_dev(h, nullptr)) return 1;
    CK(cudaMemcpyAsync(out, h->summaries, (size_t)h->R * VGSIM_NSUMMARY * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int vgsim_set_event_log(vgsim_handle h, int r, const double *in, int64_t n, const int64_t *I_end) {
    CK(cudaSetDevice(h->device));
    if (check_replicate(h, r)) return 1;
    const Dims &D = h->D;
    if (ensure_ev_cap(h, n > h->ev_bound ? n : h->ev_bound)) return 1;
    std::vector<double> t(n);
    std::vector<unsigned long long> d(n);
    long long sC = 0, cnt[6] = {0, 0, 0, 0, 0, 0};
    for (int64_t i = 0; i < n; i++) {
        int ty = (int)in[n + i];
        if (ty < 0 || ty > 5) return fail("set_event_log accepts direct-method rows only (types 0..5)");
        t[i] = in[i];
        int hap = (int)in[2 * n + i], pop = (int)in[3 * n + i], nhap = (int)in[4 * n + i], npop = (int)in[5 * n + i];
        if (ty == EV_BIRTH) npop = 0;
        if (hap < 0 || hap >= (ty == EV_SUSCCHANGE ? D.S : D.H) || pop < 0 || pop >= D.K || nhap < 0 || npop < 0 ||
            npop >= D.K)
            return fail("event row out of range");
        d[i] = pack_event(ty, hap, pop, nhap, npop);
        cnt[ty]++;
        if (ty == EV_SAMPLING) sC++;
    }
    if (n) {
        CK(cudaMemcpyAsync(h->st.ev_time + (size_t)r * h->st.ev_cap, t.data(), n * 8, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->st.ev_desc + (size_t)r * h->st.ev_cap, d.data(), n * 8, cudaMemcpyHostToDevice, h->stream));
    }
    long long c[NCOUNT] = {cnt[0], cnt[1], cnt[2], cnt[3], cnt[4], cnt[5], 0, 0, 1, (long long)n, 0, 0};
    if (I_end) {
        for (int i = 0; i < D.K * D.H; i++) c[C_GINF] += I_end[i];
        CK(cudaMemcpyAsync(h->st.I + (size_t)r * D.K * D.H, I_end, (size_t)D.K * D.H * 8, cudaMemcpyHostToDevice, h->stream));
    }
    CK(cudaMemcpyAsync(h->st.counters + (size_t)r * NCOUNT, c, NCOUNT * 8, cudaMemcpyHostToDevice, h->stream));
    double tl = n ? t[n - 1] : 0.0;
    CK(cudaMemcpyAsync(h->st.time + r, &tl, 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (n > h->ev_bound) h->ev_bound = n;
    h->st.first_simulation = 1;
    h->gen.valid = false;
    return 0;
}

}  // extern "C"
