/* vgsim_b200 — C ABI of the B200-native VGsim hot path (libvgsim_b200.so).
 *
 * This is the drop-in boundary for the reference's Python->Cython call
 * `self.simulation.<method>()` (reference src/_interface.py:44-46,823,826,839): every entry point
 * below replaces one `BirthDeathModel` method or data member of the reference
 * (src/_BirthDeath.pyx, src/events.pxi, src/models.pxi), cited per function.  Plain pointers and
 * sizes only — no torch / numpy / CUDA types in any signature.  Every function returns 0 on
 * success, non-zero on failure; the message is available from vgsim_last_error().  The int64
 * count functions (vgsim_num_lockdowns, vgsim_tree_size, vgsim_num_mutations,
 * vgsim_num_migrations) return -1 on failure, e.g. for a replicate index outside [0, R), and 0
 * when there is nothing to count (no genealogy yet).  Every entry point that takes a replicate
 * index fails with "replicate out of range" outside [0, R).
 *
 * A handle owns R independent replicates of one model shape (sites U -> H = 4^U haplotypes,
 * K demes, S susceptibility groups) on one CUDA device: compartment state, per-replicate event
 * logs, the dense tau-leap log and genealogy outputs all live in HBM between calls (the reference
 * keeps the same things in numpy arrays inside the engine object).  Unless stated otherwise all
 * pointer arguments are HOST pointers; the *_dev getters hand out device pointers for zero-copy
 * consumers (e.g. torch via __cuda_array_interface__).
 *
 * Layouts are the reference's C-order arrays: b,d,s [H]; mRate [H][U]; hapMutType [H][U][3];
 * sigma (susceptibility) [H][S]; suscType [H]; T (suscepTransition) [S][S]; m (migrationRates)
 * [K][K]; per-deme vectors [K]; state Sx [R][K][S], I [R][K][H] (int64, like the reference).
 */
#ifndef VGSIM_B200_H
#define VGSIM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct vgsim_handle_s *vgsim_handle;

/* number of int64 counters per replicate returned by vgsim_get_counters */
#define VGSIM_NCOUNTERS 12
/* order: bCounter, dCounter, sCounter, mCounter, iCounter, migPlus, migNonPlus, swapLockdown,
 *        good_attempt, events.ptr (log rows), leaps (tau rows), globalInfectious
 * (reference src/_BirthDeath.pyx:127-135, 2048-2068) */

const char *vgsim_last_error(void);
int vgsim_version(void);

/* BirthDeathModel.__init__ (src/_BirthDeath.pyx:70-229): allocate R replicates and
 * n_param_points parameter blocks on CUDA device `device` (-1 = current device). */
int vgsim_create(int sites, int K, int S, int n_replicates, int n_param_points, int device, vgsim_handle *out);
int vgsim_destroy(vgsim_handle h);

/* Launch stream for all kernels/copies of this handle (a cudaStream_t passed as void*; NULL = the
 * legacy default stream).  Lets the caller time the kernels with events on its own stream. */
int vgsim_set_stream(vgsim_handle h, void *cuda_stream);

/* Pipelined batch drivers: with async on, the entry points that copy between HOST buffers and the device
 * (vgsim_set_seeds, vgsim_set_state, vgsim_get_state without the lockdown output, vgsim_get_counters) and vgsim_reset
 * only ENQUEUE their work on the handle's stream and return; the caller's buffers must be page-locked and stay
 * untouched until vgsim_wait (or vgsim_synchronize) returns.  Two handles on two streams then overlap the uploads and
 * read-backs of one batch with the kernels of the other (what bench.py's e2e number does).  Default: off (every call
 * blocks until its copy is complete, like the reference's synchronous methods). */
int vgsim_set_async(vgsim_handle h, int on);
/* Block until everything queued on the handle's stream has finished (no error-flag read-back). */
int vgsim_wait(vgsim_handle h);

/* Per-replicate seeds: replaces RndmWrapper(seed=(user_seed, attempt)) (src/_BirthDeath.pyx:74,403,2310).
 * Replicate r draws from the counter-based Philox4x32-10 stream keyed by seeds[r]; the attempt
 * index, step index and channel index form the counter, so results do not depend on how
 * replicates are sharded over GPUs. */
int vgsim_set_seeds(vgsim_handle h, const uint64_t *seeds /*[R]*/);

/* The `set_*` parameter block (src/_BirthDeath.pyx:1380-1702) of parameter point `pp`.
 * cd_reset_mask[K] (may be NULL = all ones): demes whose LIVE contact density is overwritten with
 * contact_density[] in every replicate (what set_contact_density does, :1633-1640); elsewhere the
 * per-replicate lockdown state keeps its value.  Derived constants of UpdateAllRates (:279-351:
 * diagonal of m, actual sizes, effective migration, max effective birth-migration, cumulative
 * immunity transitions, total mutation rates) are recomputed on the host in fp64 in the
 * reference's summation order and uploaded with the block. */
int vgsim_upload_params(vgsim_handle h, int pp, const double *b, const double *d, const double *s,
                        const double *mRate, const double *hapMutType, const double *sigma,
                        const int64_t *suscType, const double *T, const double *m,
                        const double *contact_density, const double *cd_before, const double *cd_after,
                        const double *startLD, const double *endLD, const double *sampling_multiplier,
                        const int64_t *sizes, const int32_t *cd_reset_mask);
/* Parameter grid (sweeps described by their axes): points [dst_pp0, dst_pp0 + n_points) become the points
 * first_point .. first_point + n_points - 1 of the row-major product of n_axes axes (axis 0 slowest, itertools.product
 * order), built on the device.  Point pp = (c_0, .., c_{n-1}) is the source arrays of the base point base_pp (which must
 * have been uploaded) with the patch of value c_a of every axis a written over them, in axis order.  Value j of the
 * concatenated axes (j = axis_len[0] + .. + axis_len[a-1] + c_a) patches entries patch_idx[patch_off[j] ..
 * patch_off[j+1]) with patch_val[..]; an index addresses the concatenation of the 16 source arrays of
 * vgsim_upload_params in its argument order (b, d, s, mRate, hapMutType, sigma, suscType, T, m, contact_density,
 * cd_before, cd_after, startLD, endLD, sampling_multiplier, sizes; suscType and sizes as fp64).  The diagonal of m is
 * not read: it is 1 - (row's off-diagonal sum), like vgsim_upload_params computes it.  Each point's blob is the same
 * bits vgsim_upload_params writes for the same arrays.  Every point is checked first: suscType an integer in [0, S),
 * sizes an integer in [1, 2^31-1], every row of m with an off-diagonal sum <= 1 and a diagonal > 1e-15 (the two rules of
 * the reference's migration setters).  A failing point fails the whole call with a message naming its grid index and
 * the rule; nothing is uploaded then.  Otherwise the live contact density of every replicate mapped to one of the
 * points is set to that point's contact_density (what a first vgsim_upload_params of the point does).  One stream
 * synchronisation per call; host cost O(sum axis_len + patches), device work O(n_points). */
int vgsim_upload_param_grid(vgsim_handle h, int base_pp, int n_axes, const int32_t *axis_len,
                            const int64_t *patch_off /*[sum axis_len + 1]*/, const int64_t *patch_idx,
                            const double *patch_val, int64_t first_point, int dst_pp0, int n_points);
/* Read tap: the device blob of parameter point pp (the derived constants the kernels read; its length follows from the
 * model shape, see Dims in csrc/common.cuh). */
int vgsim_get_params(vgsim_handle h, int pp, double *blob_out);
/* replicate -> parameter point map (default: all 0).  Parameter sweeps (BASELINE config 5).  Before the first simulate
 * call the live contact density of every replicate is (re)seeded from its point's uploaded value, whichever of
 * vgsim_upload_params / vgsim_set_replicate_params comes first; after it the map may still change, but contact
 * densities are run state (lockdowns) and are left alone. */
int vgsim_set_replicate_params(vgsim_handle h, const int32_t *replicate_to_param /*[R]*/);

/* susceptible / infectious compartments (src/_BirthDeath.pyx:150,178; set_susceptible/set_infectious
 * :1593-1627).  Before the first simulate call this is the initial state (FirstInfection, :234-242,
 * is applied on top by the first simulate call exactly like the reference does). */
int vgsim_set_state(vgsim_handle h, const int64_t *Sx /*[R][K][S]*/, const int64_t *I /*[R][K][H]*/);
int vgsim_get_state(vgsim_handle h, int64_t *Sx, int64_t *I, double *contact_density /*[R][K]*/,
                    int64_t *lockdown_on /*[R][K]*/);

/* Same as vgsim_set_state with DEVICE pointers (asynchronous on the handle's stream), and the device
 * pointers of the live compartment arrays Sx[R][K][S], I[R][K][H] (int64) for zero-copy consumers. */
int vgsim_set_state_dev(vgsim_handle h, const int64_t *dSx, const int64_t *dI);
int vgsim_state_dev(vgsim_handle h, void **dSx, void **dI);
/* Back to the state of a freshly constructed engine with the uploaded parameters kept: event logs,
 * counters, clocks, lockdown flags and genealogy are dropped (log capacity is retained and reused), the
 * next simulate call is a "first simulation" again (what re-running the reference's constructor +
 * setters does; batch drivers call it between independent batches, followed by vgsim_set_state). */
int vgsim_reset(vgsim_handle h);

/* Resampling and branching on the device: for every r with source[r] != r, replicate r's run becomes the run replicate
 * source[r] had before the call; replicates with source[r] == r are untouched.  Copied: I, Sx and the Restart snapshot,
 * live contact density, lockdown flags and records, effective migration, clock, rate totals, all counters, the Philox
 * epoch, error bits, the recycled-row count, the event log rows [0, events), the (time, tau) rows [0, leaps), the dense
 * rows not yet archived and the archive itself (used rows only, never whole capacities).  Not copied: the seed and the
 * parameter point -- r keeps its own, and its derived rates follow its point at the next simulate call or rate tap.  A
 * clone given its source's seed then continues exactly like the source; with its own seed it is an independent run from
 * the same history.
 * Rule: a replicate that is copied from keeps its own run, source[source[r]] == source[r] for every r (survivors keep
 * their slots, extra copies fill the slots of replicates that die), so the gather needs no staging memory.  A map that
 * breaks it, or an index outside [0, R) ("replicate out of range"), fails with a message naming r and its source, and
 * changes nothing.  Genealogy outputs are dropped as after a simulate call.  Whatever a replicate holds is copied: after
 * vgsim_genealogy, the rewound infectious counts.  Stream-ordered, no host synchronisation: one small copy of the map and
 * one kernel launch on the handle's stream; the identity map enqueues nothing.  Works before the first simulate call
 * (the configured state is copied) and on every shape vgsim_create accepts. */
int vgsim_resample(vgsim_handle h, const int32_t *source /*[R]*/);

/* Long runs in leap blocks: drop the event log / dense tau log of every replicate but keep compartments, clocks,
 * event counters, lockdown state and the Philox epoch, so that the next simulate call continues the same
 * trajectories into recycled log capacity (the reference can only grow its log, src/events.pxi:52-68; 4,096
 * replicates x 1,200 leaps of the T3 shape would be 520 GB).  A consumer (vgsim_epidemic_curves, vgsim_genealogy)
 * must have read the block first; events.ptr and the leap count restart at 0. */
int vgsim_recycle_log(vgsim_handle h);

/* Long runs with the whole log kept: move the dense count rows of every replicate (4P bytes per leap) into a sparse
 * archive -- the non-zero counts as (channel, count) pairs in ascending channel order, 8 bytes each -- and free the dense
 * capacity for the next block of leaps.  The event log, leap times, counters and state are untouched; vgsim_genealogy,
 * vgsim_epidemic_curves, vgsim_get_tau_log and vgsim_get_multievents read archived leaps from the archive and give the
 * same results as on the dense rows.  (The reference appends 56 bytes per channel and leap, zeros included,
 * src/_BirthDeath.pyx:2536-2593; the dense row stays the roofline yardstick, SURVEY 8(d).) */
int vgsim_archive_tau_log(vgsim_handle h);
/* Size of the archive: (channel, count) entries over all replicates, the largest replicate's, and the leaps archived. */
int vgsim_archive_stats(vgsim_handle h, int64_t *entries_total, int64_t *entries_max, int64_t *leaps_archived);

/* SimulatePopulation (src/_BirthDeath.pyx:396-429): batched direct Gillespie, one warp per
 * replicate.  `epidemic_time` is a C float like the reference's (quirk Q1); -1 = no limit;
 * sample_size -1 = no limit.  Appends up to `iterations` rows to each replicate's event log.
 * Every shape vgsim_create accepts runs: a shape whose rate hierarchy fits one SM's shared memory runs on the
 * shared-memory kernel, any other on the large-state kernel, which keeps each replicate's rates in 32-ary sum trees in
 * device memory (one slice per resident warp, allocated at its first call and held by the handle, at most half of the
 * free device memory).  The two kernels draw from independent streams: they agree in distribution, not draw for draw.
 * vgsim_set_direct_variant bit 0 runs the large-state kernel on every shape. */
int vgsim_simulate_direct(vgsim_handle h, int64_t iterations, int64_t sample_size, float epidemic_time,
                          int64_t attempts);
/* SimulatePopulation_tau (src/_BirthDeath.pyx:2293-2346): replicate-batched tau-leaping, one CTA
 * per replicate; appends up to `iterations` leaps (MULTITYPE rows + dense count blocks). */
int vgsim_simulate_tau(vgsim_handle h, int64_t iterations, int64_t sample_size, float epidemic_time,
                       int64_t attempts);
/* The same call run as blocks of `leap_block` leaps with vgsim_archive_tau_log between blocks: the dense rows never
 * exceed one block per replicate (a 2,000-leap run of the K = 100 world model would need 4 GB of dense rows per replicate).
 * One call to the reference's eyes: FirstInfection (:2302-2303) only before the first block, the stop conditions of
 * :2312 carry over, the run ends when no replicate used up its block.  leap_block is raised to 101 when iterations > 100
 * so that the extinction retry of :2331 sees the same condition in every block.  The last block is archived too. */
int vgsim_simulate_tau_blocks(vgsim_handle h, int64_t iterations, int64_t sample_size, float epidemic_time,
                              int64_t attempts, int64_t leap_block);
/* Block until everything queued on the handle's stream has finished; returns the sticky device
 * error flags of the last kernels (0 = ok). */
int vgsim_synchronize(vgsim_handle h);

/* Number of reaction channels P (src/_BirthDeath.pyx:2301). */
int64_t vgsim_prop_num(vgsim_handle h);

/* Deterministic parity taps.
 * vgsim_propensities = PrintPropensities (src/_BirthDeath.pyx:2615-2649): Propensities (:2351-2417)
 * + ChooseTau (:2432-2450) of replicate r's CURRENT state, computed by the tau kernel's own device
 * code; out[P] in positional channel order (SURVEY App. A.4), drift dI[K][H], dS[K][S], tau. */
int vgsim_propensities(vgsim_handle h, int replicate, double *out, double *dI, double *dS, double *tau);
/* vgsim_rates = the direct-method rate hierarchy after UpdateAllRates (:279-351) computed by the
 * direct kernel's device code: actual sizes A[K], eff[K][K], maxEBM[K], event rates ev[K][H][4],
 * hapPopRate[K][H], popRate[K], migPopRate[K], totals[2] = {totalRate, totalMigrationRate}.  On shapes that
 * vgsim_simulate_direct runs on the large-state kernel (and on every shape with vgsim_set_direct_variant bit 0) the
 * numbers come from that kernel's sum trees: hapPopRate[p,h] = c[p] sum_s Sx[p,s] b[h] sigma[s,h] I[p,h] + (d[h] +
 * sr[h] sm[p] + tm[h]) I[p,h], popRate and totalRate from the deme tree. */
int vgsim_rates(vgsim_handle h, int replicate, double *A, double *eff, double *maxEBM, double *ev,
                double *hapPopRate, double *popRate, double *migPopRate, double *totals);

/* counters[R][VGSIM_NCOUNTERS], current_time[R] (Stats, src/_BirthDeath.pyx:2048-2068). */
int vgsim_get_counters(vgsim_handle h, int64_t *counters, double *current_time);

/* Event log of one replicate in the reference's export_chain_events layout
 * (src/_BirthDeath.pyx:1849-1851; src/events.pxi:24-68): out[6][n] float64 = times, types,
 * haplotypes, populations, newHaplotypes, newPopulations; MULTITYPE rows carry the
 * [first, one-past-last) multi-event indices like the reference's.  n = counters[..][9]. */
int vgsim_get_event_log(vgsim_handle h, int replicate, double *out6xN, int64_t n);
/* Dense tau log of one replicate expanded to the reference's multiEvents SoA
 * (src/events.pxi:105-152): n = leaps * P records. Any output pointer may be NULL. */
int vgsim_get_multievents(vgsim_handle h, int replicate, int64_t n, int64_t *num, double *time,
                          int64_t *type, int64_t *hap, int64_t *pop, int64_t *nhap, int64_t *npop);
/* Raw dense tau log: counts[leaps][P] int32 and (time, tau)[leaps][2] float64. */
int vgsim_get_tau_log(vgsim_handle h, int replicate, int64_t leaps, int32_t *counts, double *time_tau);
/* Replace replicate r's event log with direct-method rows given in the 6 x n reference layout (the
 * working counterpart of the reference's broken set_chain_events, src/_BirthDeath.pyx:1705-1719),
 * and set its infectious counts I[K][H] to the state at the END of that log. */
int vgsim_set_event_log(vgsim_handle h, int replicate, const double *in6xN, int64_t n, const int64_t *I_end);

/* Lockdown records (src/models.pxi:49-66): n rows of (state, deme, time) for replicate r. */
int64_t vgsim_num_lockdowns(vgsim_handle h, int replicate);
int vgsim_get_lockdowns(vgsim_handle h, int replicate, int64_t *state, int64_t *pop, double *time);

/* GetGenealogy (src/_BirthDeath.pyx:743-1000) for every replicate with sCounter >= 2, one warp per
 * replicate.  seeds == NULL continues each replicate's forward key (reference quirk Q10), otherwise
 * seeds[R] re-keys the stream.  Parity tap: if uniform_stream != NULL, replicate r consumes
 * uniform_stream[stream_offsets[r] .. stream_offsets[r+1]) in order in place of Philox uniforms
 * (64-bit raw words when raw_words != 0: next_double = (w >> 11) * 2^-53, like numpy's PCG64). */
int vgsim_genealogy(vgsim_handle h, const uint64_t *seeds, const double *uniform_stream,
                    const int64_t *stream_offsets /*[R+1]*/, int raw_words);
/* Tree of replicate r: n = 2*sCounter-1 nodes; parent (root = -1), deme, absolute time
 * (self.tree, self.tree_pop, self.times; src/_BirthDeath.pyx:769-773). */
int64_t vgsim_tree_size(vgsim_handle h, int replicate);
int vgsim_get_tree(vgsim_handle h, int replicate, int64_t *parent, int64_t *pop, double *time);
/* Mutations (src/models.pxi:12-26) and Migrations (src/models.pxi:42-46) side tables. */
int64_t vgsim_num_mutations(vgsim_handle h, int replicate);
int vgsim_get_mutations(vgsim_handle h, int replicate, int64_t *node, int64_t *AS, int64_t *DS, int64_t *site,
                        double *time);
int64_t vgsim_num_migrations(vgsim_handle h, int replicate);
int vgsim_get_migrations(vgsim_handle h, int replicate, int64_t *node, double *time, int64_t *old_pop,
                         int64_t *new_pop);

/* Fixed-size per-replicate summary vector (device-resident; what the multi-GPU all-gather moves, together with the
 * time-resolved rows of vgsim_trajectories_dev and vgsim_lineages_through_time_dev when a sweep wants them):
 * counters, final time, and tree statistics when a genealogy exists.  out[R][VGSIM_NSUMMARY] f64:
 *   [0..11] the VGSIM_NCOUNTERS counters, [12] current time, [13] tree nodes (2n-1), [14] tree height,
 *   [15] total branch length, [16] roots (1 = fully coalesced), [17] mutation rows, [18] migration rows,
 *   [19] root time, [20] cherries, [21] Sackin index (sum of leaf depths), [22] totalRate and [23] totalMigrationRate as
 *   the last vgsim_simulate_direct call's incremental updates left them (UpdateRates, src/_BirthDeath.pyx:516-546; parity tap:
 *   vgsim_rates recomputes both from the state).
 * vgsim_summaries_dev returns the DEVICE pointer of the same buffer (valid until destroy). */
#define VGSIM_NSUMMARY 24
int vgsim_summaries(vgsim_handle h, double *out);
int vgsim_summaries_dev(vgsim_handle h, void **dev_ptr);

/* Epidemic curves of EVERY compartment of replicates [rep_first, rep_first + rep_count) in one pass over their
 * event logs (direct rows and MULTITYPE leaps); replaces get_data_infectious / get_data_susceptible
 * (src/_BirthDeath.pyx:1967-2045), which walk the whole log once per (deme, haplotype) query.
 * Grid: time_points[q][j] = j * currentTime / step_num, j = 0..step_num (:1968); the value at j is the state
 * after every log row with time <= time_points[j] (:1975-1978).  Host outputs, any may be NULL:
 *   infectious[rep_count][step_num+1][K*H], susceptible[..][K*S] : compartment counts;
 *   removed[..][K*H], sampled[..][K*H] : cumulative recoveries+samplings / samplings per infectious cell (the
 *   reference's Data / Sample arrays mix these in through an operator-precedence quirk; the Python wrapper rebuilds
 *   its exact output from them);
 *   last_point[rep_count] : index of the grid point that holds the last log row (the reference leaves later points
 *   zero, here they repeat the final state).
 * A replicate whose counts do not fit one SM's shared memory is replayed in a device scratch slice instead (one per
 * resident warp, freed on return, at most half of the free device memory); the results are the same. */
int vgsim_epidemic_curves(vgsim_handle h, int rep_first, int rep_count, int step_num, int64_t *infectious,
                          int64_t *susceptible, int64_t *removed, int64_t *sampled, double *time_points,
                          int32_t *last_point);

/* Trajectories of every replicate on ONE time grid shared by all of them, one pass over each event log (the walk of
 * vgsim_epidemic_curves: direct rows, dense MULTITYPE rows, archived leaps; replicates whose counts exceed one SM's shared
 * memory replay in device scratch slices).  times[T]: absolute times, finite, strictly increasing, 1 <= T <= 2^30.  Row
 * j of replicate r is the state after every log row with time <= times[j], starting from the state vgsim_epidemic_curves
 * starts from, as 2K + 2H int64 in this order:
 *   infectious per deme [K] (sum over haplotypes), infectious per haplotype [H] (sum over demes),
 *   samplings per deme [K] and per haplotype [H], cumulative since the start of the log.
 * A point with times[j] > currentTime[r] was not simulated for that replicate: every entry of its row is -1.
 * out[R][T][2K + 2H].  vgsim_trajectories_dev returns the DEVICE pointer of the same rows instead (a buffer owned by the
 * handle, grown when needed, valid until the next vgsim_trajectories* call or destroy); the rows are fixed-size per
 * replicate, so a multi-GPU all-gather can move them like the summaries.  vgsim_last_kernel_ms reports the kernel. */
int vgsim_trajectories(vgsim_handle h, const double *times, int64_t T, int64_t *out);
int vgsim_trajectories_dev(vgsim_handle h, const double *times, int64_t T, void **dev_ptr);

/* Lineages through time of every replicate's genealogy (after vgsim_genealogy; fails with a message before one, or after
 * a later simulate call) on the grid times[T] (same rules as vgsim_trajectories, T <= 32768):
 *   out[r][j] = #{ node i : time[i] >= times[j] and (parent[i] < 0 or time[parent[i]] < times[j]) }
 * with absolute node times as vgsim_get_tree returns them; every root of a forest counts its lineage.  A replicate
 * without a tree (summaries[13] == 0) gets a row of zeros.  out[R][T] int64; vgsim_lineages_through_time_dev returns the
 * DEVICE pointer of the same rows (owned by the handle, valid until the next vgsim_lineages_through_time* call or
 * destroy).  vgsim_last_kernel_ms reports the kernel. */
int vgsim_lineages_through_time(vgsim_handle h, const double *times, int64_t T, int64_t *out);
int vgsim_lineages_through_time_dev(vgsim_handle h, const double *times, int64_t T, void **dev_ptr);

/* Parity tap.  Variant 0 (default, product): per infectious cell the kernel draws ONE Poisson for the total of
 * its mutation channels and ONE for the total of its out-migration channels whenever that total's lambda is
 * <= 0.25 (mutation) / 0.5 (out-migration), and splits a non-zero total multinomially over the group's channels (independent Poissons
 * conditioned on their sum are multinomial, so the joint distribution is unchanged).  Variant 1 draws every
 * channel separately, exactly like the reference's GenerateEvents_tau (src/_BirthDeath.pyx:2454-2532);
 * tests compare both with theory and with each other.
 * Bits 2 and 3 pick the kernel mapping (scheduling only, same log bit for bit): by default a batch small enough to
 * be resident as 256-thread teams runs on the team kernel, larger batches on the warp-per-replicate kernel; bit 2
 * forces the former, bit 3 the latter.  Bits 4 and 5 switch off the warp kernel's lockstep generations and its
 * size-sorted replicate schedule (scheduling only as well; tests check that the log does not change).  Bit 6 runs the
 * warp kernel instance that reads the model dimensions at run time even where one with the shape compiled in exists
 * (same log bit for bit; see vgsim_tau_fixed_shape). */
int vgsim_set_tau_variant(vgsim_handle h, int variant);
/* Which warp kernel instance the last tau launch of this handle ran: U << 16 | K << 8 | S of the model shape it was
 * compiled for ((3, 10, 3) and (2, 10, 3) have one), 0 for an instance that reads the shape at run time (every
 * other shape, variant bit 6, the team kernel). */
int vgsim_tau_fixed_shape(vgsim_handle h);
/* Parity tap of the direct method.  Bit 0: vgsim_simulate_direct and vgsim_rates use the large-state kernel (sum
 * trees in device memory) on every shape, not only on shapes whose rate hierarchy exceeds one SM's shared memory.
 * Default 0.  Tests compare the two kernels in distribution and the trees with the reference's rates. */
int vgsim_set_direct_variant(vgsim_handle h, int variant);
/* Measurement tap: with bit 1 of the variant set, thread 0 of every CTA of the tau kernel accumulates the clock
 * cycles between consecutive barriers of the leap loop (critical path per phase: 0 row wipe + lists + Q,
 * 1 drifts + tau, 2 primary draws, 3 slow-path drain, 4 feasibility, 5 apply, 6 lockdown vote, 7 = #leaps)
 * summed over CTAs since the last reset.  out16[16]. */
int vgsim_debug_tau_phases(vgsim_handle h, uint64_t *out16, int reset);
/* Same tap, the tail of a launch: out1024[2b] / [2b+1] = global-timer ns at which the first / the last warp of CTA b
 * (b < 512) of the warp kernel ran out of replicates; slots 8-11 of vgsim_debug_tau_phases hold latest / sum / count /
 * earliest over all warps. */
int vgsim_debug_tau_cta_end(vgsim_handle h, uint64_t *out1024, int reset);

/* Launch accounting: kernels launched by this handle since creation. */
int64_t vgsim_launch_count(vgsim_handle h);
/* Device time of the LAST hot kernel (tau / direct / epidemic curves / trajectories / lineages through time), bracketed by CUDA events on the handle's
 * stream inside vgsim_simulate_* (replaces the reference's time.time() pair, src/_interface.py:821-827).
 * Blocks until that kernel has finished. */
int vgsim_last_kernel_ms(vgsim_handle h, float *ms);
/* The same for a pipelined driver: every hot-kernel launch gets an id (vgsim_last_kernel_id, right after the simulate call);
 * vgsim_kernel_ms reads the duration of launch `id` later (blocks until it has finished).  The last 64 launches are held. */
int64_t vgsim_last_kernel_id(vgsim_handle h);
int vgsim_kernel_ms(vgsim_handle h, int64_t id, float *ms);
/* Device pointers of counters[R][VGSIM_NCOUNTERS] (int64) and current_time[R] (fp64). */
int vgsim_counters_dev(vgsim_handle h, void **counters, void **current_time);

/* Test taps for the device samplers (Poisson: multiplication-free inversion / PTRS;
 * hypergeometric: numpy-compatible HYP/HRUA): n draws each from Philox keyed by `seed`. */
int vgsim_test_poisson(const double *lam, int64_t n, uint64_t seed, int64_t *out);
int vgsim_test_hypergeometric(const int64_t *good, const int64_t *bad, const int64_t *sample, int64_t n,
                              const uint64_t *raw_words, int64_t n_words, int64_t *out, int64_t *words_used);

/* Test tap for the cumulative search that replaces fastChoose / fastChoose_skip (src/fast_choose.pxi:18-52): m queries
 * x[q] in [0, sum w) over the same n weights; skip >= 0 leaves that index out (fastChoose_skip); small != 0 runs the
 * sequential every-lane variant used for the handful-of-weights levels.  Outputs per query: picked index (-1 when every
 * weight is zero), cumulative weight before it, its weight, and the reference's residual (x - before) / w. */
int vgsim_test_choose(const double *w, int n, const double *x, int m, int skip, int small, int64_t *idx,
                      double *before, double *wsel, double *resid);

#ifdef __cplusplus
}
#endif
#endif /* VGSIM_B200_H */
