// Host-side handle behind the C ABI (include/vgsim_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <memory>
#include <string>
#include <vector>
#include "common.cuh"

namespace vg {

// One vgsim_upload_param_grid call: the base point's source arrays (concatenated in vgsim_upload_params order, fp64) and
// the patch tables, from which the host record of any of its points is rebuilt on demand.
struct ParamGrid {
    std::vector<double> base;
    std::vector<int> axis_len;
    std::vector<long long> off, idx;
    std::vector<double> val;
};

struct HostParams {  // host copy of one parameter point in the reference's layouts
    std::vector<double> b, d, s, mRate, hapMutType, sigma, T, m, cd, cdBefore, cdAfter, startLD, endLD, sm;
    std::vector<long long> suscType, sizes;
    bool uploaded = false;
    std::shared_ptr<const ParamGrid> grid;  // set: a grid point whose arrays above are not filled in yet
    long long grid_point = 0;               // its global index in the grid
};

// Arguments of the parameter-grid kernels (param_grid_kernel.cu); device pointers.
enum { GRID_ERR_SUSC = 1, GRID_ERR_SIZES = 2, GRID_ERR_MIG_SUM = 4, GRID_ERR_MIG_DIAG = 8 };
struct GridArgs {
    const double *base;  // [nsrc] the base point's source arrays, concatenated
    int n_axes;
    const int *axis_len;                  // [n_axes]
    const long long *off, *idx;           // [sum axis_len + 1], [off[sum]]
    const double *val;                    // [off[sum]]
    long long first_point;
    int dst_pp0, n_points;
    double *slots;  // [nslots][nsrc] one assembled point per CTA
    int nslots;
    int *err;       // [n_points] GRID_ERR_* bits of each point
    int *flag;      // [1] non-zero when any point failed
};

struct GenealogyBuffers {
    // per replicate outputs; node capacity = 2*sC-1
    long long *node_off = nullptr;     // [R+1] prefix offsets into the node arrays
    int *parent = nullptr, *pop = nullptr;
    double *time = nullptr;
    long long total_nodes = 0;
    // side tables
    long long *mut_off = nullptr, *mig_off = nullptr;  // [R+1] capacity offsets
    int *mut_n = nullptr, *mig_n = nullptr;            // [R] used
    int *mut_node = nullptr, *mut_hap = nullptr;       // hap | nhap packed separately
    int *mut_nhap = nullptr;
    double *mut_time = nullptr;
    int *mig_node = nullptr, *mig_old = nullptr, *mig_new = nullptr;
    double *mig_time = nullptr;
    // lineage arena
    long long *arena_off = nullptr;  // [R+1]
    int *arena = nullptr;
    int *cell_hdr = nullptr;         // [R][K*H][3] (offset, size, cap)
    int *n_nodes = nullptr;          // [R] nodes actually created
    int *scratch = nullptr;          // one int per node: newLineages scratch of the replay, then tree-shape scratch
    bool valid = false;
    std::vector<long long> h_node_off, h_mut_off, h_mig_off;
};

struct Handle {
    int device = 0;
    int num_sms = 148;
    cudaStream_t stream = 0;
    Dims D;
    int R = 0, n_pp = 0;
    DevState st;
    std::vector<HostParams> hp;
    long long ev_bound = 0, leap_bound = 0;  // host upper bounds of log rows / leaps per replicate
    long long dense_bound = 0;               // ... of leaps whose dense row has not been archived
    long long launches = 0;
    int tau_variant = 0;  // 0 = aggregated small groups (product), 1 = one Poisson draw per channel (parity tap)
    int direct_variant = 0;  // bit 0: the large-state direct kernel on every shape (parity tap)
    int tau_fixed_shape = 0;  // U << 16 | K << 8 | S of the compiled-in shape the last tau launch ran, 0: runtime shape
    double *dl_slices = nullptr;  // warp slices of the large-state direct kernel (allocated at its first call)
    size_t dl_slices_n = 0;       // doubles held
    bool state_set = false;
    bool async_host = false;  // vgsim_set_async: host-buffer copies are enqueued without blocking the calling thread
    GenealogyBuffers gen;
    double *summaries = nullptr;  // [R][VGSIM_NSUMMARY]
    int *work = nullptr;           // [4] atomic work counters of the kernels that hand out replicates dynamically
    int *tau_order = nullptr;      // [2R] scratch of the tau kernel's size-sorted schedule (weights, order)
    int *arch_cnt = nullptr, *arch_need = nullptr;  // scratch of vgsim_archive_tau_log: non-zero counts per dense row / per replicate
    size_t arch_cnt_cap = 0;
    std::vector<int> rep_pp_host;  // host copy of the replicate -> parameter point map
    // outputs of vgsim_trajectories / vgsim_lineages_through_time and the device copy of their grid: grown, never shrunk
    double *grid_buf = nullptr;
    long long *traj_buf = nullptr, *ltt_buf = nullptr;
    size_t grid_cap = 0, traj_cap = 0, ltt_cap = 0;
    int2 *resample_pairs = nullptr;  // (destination, source) pairs of the last vgsim_resample: grown, never shrunk
    size_t resample_cap = 0;
    // event pairs that bracket the hot kernels on the handle's stream: a ring, so that a pipelined driver can read the
    // duration of launch `id` after the fact (vgsim_kernel_ms) instead of blocking on every launch
    static const int NTIMER = 64;
    cudaEvent_t ev_ring0[NTIMER] = {}, ev_ring1[NTIMER] = {};
    long long timer_id = -1;  // id of the last hot-kernel launch
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr;  // the pair of the last launch
    bool ev_valid = false;
    std::vector<void *> allocs;
};

// 32-ary sum tree of the large-state direct kernel (direct_large_kernel.cu): level l has n[l] nodes at offset off[l]
// (doubles); size: doubles in all.  Depth 4 holds 2^20 leaves (H <= 4^9, K <= 4096).
#define TREE32_MAXD 4
struct Tree32 {
    int depth, size;
    int off[TREE32_MAXD], n[TREE32_MAXD];
};
// One warp slice of the large-state direct kernel, in doubles: K * nt haplotype trees, the deme tree, the per-deme
// vectors.
struct DLLayout {
    Tree32 th, tk;  // over the H haplotypes of a deme, over the K demes
    int nt;         // trees per deme: S + 2
    long long o_dtree, o_tm, o_Sx, o_root, o_totSus, o_imm, o_c, o_cd, o_maxEBM, o_lock, o_zs;
    long long slice;
};
DLLayout dl_layout(const Dims &D);

// kernels' host launchers (defined in the .cu files)
cudaError_t launch_tau(const DevState &st, const SimArgs &a, cudaStream_t stream, int num_sms, int variant, int uniform_pp,
                       int *order_buf, int *fixed_shape);
cudaError_t tau_phase_cycles(unsigned long long *out16, int reset);
cudaError_t tau_cta_end(unsigned long long *out1024, int reset);
cudaError_t launch_propensities(const DevState &st, int r, double *out, double *dI, double *dS, double *tau,
                                cudaStream_t stream);
cudaError_t launch_archive_count(const DevState &st, int *cnt, int *need, cudaStream_t stream);
cudaError_t launch_archive_write(const DevState &st, const int *cnt, const int *need, cudaStream_t stream);
cudaError_t launch_prepare(const DevState &st, int first, int tau_mode, cudaStream_t stream);
cudaError_t launch_refresh(const DevState &st, cudaStream_t stream);
cudaError_t launch_direct(const DevState &st, const SimArgs &a, cudaStream_t stream, int num_sms, int uniform_pp, int *work);
bool direct_fits_shared(const Dims &D, int uniform_pp);
cudaError_t launch_direct_large(const DevState &st, const SimArgs &a, const DLLayout &L, double *slices, int nwarps,
                                int num_sms, cudaStream_t stream, int *work);
// one replicate's curve slice in bytes; when it does not fit one SM's shared memory, launch_curves replays in gslices,
// a device scratch of nslices >= 1 such slices
size_t curves_slice_bytes(const Dims &D, bool tallies);
cudaError_t launch_curves(const DevState &st, int rep_first, int rep_count, int step_num, long long *inf, long long *sus,
                          long long *removed, long long *sampled, double *time_points, int *last_point,
                          cudaStream_t stream, int num_sms, unsigned char *gslices, int nslices);
// trajectories of every replicate on the grid times[npoints] (device), out[R][npoints][2K + 2H]; gslices as above, slices
// of trajectories_slice_bytes
size_t trajectories_slice_bytes(const Dims &D);
cudaError_t launch_trajectories(const DevState &st, const double *times, int npoints, long long *out, cudaStream_t stream,
                                int num_sms, unsigned char *gslices, int nslices);
// lineages through time of every replicate's genealogy on the grid times[npoints] (device), out[R][npoints]
int ltt_max_points();
cudaError_t launch_ltt(const DevState &st, const long long *node_off, const int *parent, const double *time,
                       const int *n_nodes, int *scratch, const double *times, int npoints, long long *out,
                       cudaStream_t stream, int num_sms);
cudaError_t launch_rates_tap(const DevState &st, int r, double *ev, double *hp, double *popRate, double *migPop,
                             double *totals, cudaStream_t stream);
cudaError_t launch_rates_large(const DevState &st, const DLLayout &L, double *slice, int r, double *ev, double *hp,
                               double *popRate, double *migPop, double *totals, cudaStream_t stream);
bool tau_fits(const Dims &D, int uniform_pp);
int param_grid_slots(int num_sms, int n_points);
cudaError_t launch_param_grid(const DevState &st, const GridArgs &g, cudaStream_t stream);
// the gather of vgsim_resample over pairs[ndst] (device); the bounds are the handle's host maxima of log rows, leaps and
// dense rows per replicate.  nlaunch: kernel launches enqueued (0 when ndst == 0)
cudaError_t launch_resample(const DevState &st, const int2 *pairs, int ndst, long long ev_bound, long long leap_bound,
                            long long dense_bound, cudaStream_t stream, int *nlaunch);

}  // namespace vg
