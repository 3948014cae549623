"""Parameter sweeps: one replicate batch in which every replicate (or group of replicates) has its own parameter
point (BASELINE.json configs[4]: "ABC-style sweep: 65,536 replicates over R0/migration grid sharded across 8xB200").

The reference runs one `Simulator` per parameter point and process.  Here a sweep is ONE handle: `n_points`
parameter blobs are uploaded once (`vgsim_upload_params`), `vgsim_set_replicate_params` maps replicates to points,
and a single launch of each kernel advances all of them; a rank owns a contiguous range of the global point list
(`_shard.replicate_range`), replicate seeds are functions of the GLOBAL replicate id, and the only exchange is the
all-gather of fixed-size rows: the summaries, and where wanted the trajectories and lineages through time on a grid
shared by every replicate (`_shard.gather_summaries` moves any of them).
"""
import numpy as np

from . import _capi, _shard
from ._engine import BirthDeathModel


class Sweep:
    """`points`: list of callables, each taking a configured engine and changing it through the reference's setters
    (e.g. ``lambda e: (e.set_transmission_rate(0.3, None), e.set_total_migration_probability(1e-3))``)."""

    def __init__(self, dims, base_setup, points, replicates_per_point=1, seed=0, rank=0, world=1, device=None):
        self._open(dims, base_setup, len(points), replicates_per_point, seed, rank, world, device)
        for i in range(self.hi - self.lo):
            e = self.engine
            saved = {k: v.copy() for k, v in e.param_arrays().items()}
            points[self.lo + i](e)
            self.h.upload_params(i, e.param_arrays())
            self._restore(e, saved)
        self._seed_and_state(seed)

    @classmethod
    def grid(cls, dims, base_setup, axes, replicates_per_point=1, seed=0, rank=0, world=1, device=None):
        """The sweep over the row-major product of `axes` (axis 0 slowest, `itertools.product` order): the same points,
        rank slices, seeds and results as ``Sweep(dims, base_setup, [point(v0, v1, ..) for v0 in axes[0][1] for v1 in
        ...])`` where a point applies every axis's setter in axis order.  `axes`: list of ``(setter, values)``, where
        ``setter(engine, value)`` calls the reference's setters (e.g. ``lambda e, v: e.set_transmission_rate(v, None)``).

        Each axis value is resolved once on the host into a patch of the parameter arrays (`resolve_axes`); the points
        are assembled, checked and derived on the device (vgsim_upload_param_grid), so host work grows with the sum of
        the axis lengths, not their product."""
        axes = [(setter, list(values)) for setter, values in axes]
        self = cls.__new__(cls)
        self._open(dims, base_setup, int(np.prod([len(v) for _, v in axes], dtype=np.int64)), replicates_per_point,
                   seed, rank, world, device)
        off, idx, val = resolve_axes(self.engine, axes)
        self.h.upload_params(0, self.engine.param_arrays())
        self.h.upload_param_grid(0, [len(v) for _, v in axes], off, idx, val, self.lo, 0, self.hi - self.lo)
        self._seed_and_state(seed)
        return self

    def _open(self, dims, base_setup, n_global, replicates_per_point, seed, rank, world, device):
        U, K, S = dims
        self.n_global = n_global
        self.lo, self.hi = _shard.replicate_range(rank, world, self.n_global)
        self.rpp = int(replicates_per_point)
        n_pts = self.hi - self.lo
        self.R = n_pts * self.rpp
        self.engine = BirthDeathModel(U, K, S, seed, False, False, int(1e6), 0.0)   # host-side validation + arrays only
        base_setup(self.engine)
        self.h = _capi.Handle(U, K, S, self.R, n_pts, device)
        # the map first: an upload seeds the live contact density of the replicates that are mapped to its point
        self.h.set_replicate_params(np.repeat(np.arange(n_pts, dtype=np.int32), self.rpp))

    def _seed_and_state(self, seed):
        gid = np.arange(self.lo * self.rpp, self.hi * self.rpp, dtype=np.uint64)
        self.h.set_seeds((np.uint64(seed) + gid).astype(np.uint64))
        Sx, I = self.engine._susceptible, self.engine._infectious
        self.h.set_state(np.ascontiguousarray(np.broadcast_to(Sx, (self.R,) + Sx.shape)),
                         np.ascontiguousarray(np.broadcast_to(I, (self.R,) + I.shape)))

    @staticmethod
    def _restore(e, saved):
        """Put the base parameter arrays back (the engine's arrays are the live views the setters write into)."""
        live = e.param_arrays()
        names = dict(b="bRate", d="dRate", s="sRate", mRate="mRate", hapMutType="hapMutType", sigma="_susceptibility",
                     suscType="suscType", T="suscepTransition", m="migrationRates", cd="contactDensity",
                     cdBefore="contactDensityBeforeLockdown", cdAfter="contactDensityAfterLockdown", startLD="startLD",
                     endLD="endLD", sm="samplingMultiplier", sizes="sizes")
        for k, attr in names.items():
            getattr(e, attr)[...] = saved[k]
        del live

    def simulate(self, iterations, sample_size=None, epidemic_time=-1, method="direct", attempts=200):
        ss = iterations if sample_size is None else sample_size
        if method == "direct":
            self.h.simulate_direct(int(iterations), int(ss), float(epidemic_time), int(attempts))
        elif method == "tau":
            self.h.simulate_tau(int(iterations), int(ss), float(epidemic_time), int(attempts))
        else:
            raise ValueError("Unknown method. Choose between 'direct' and 'tau'.")

    def resample(self, source):
        """Replicate r of this rank continues the run of replicate source[r] of this rank (rank-local indices, one per
        replicate, points in order and replicates_per_point within each); r keeps its seed and parameter point, so a
        fork of one history maps into every point of the sweep (Handle.resample)."""
        self.h.resample(source)

    def genealogy(self, seed=None):
        self.h.genealogy(seed, None)

    def summaries(self):
        """[points on this rank, replicates_per_point, NSUMMARY] (include/vgsim_b200.h: vgsim_summaries)."""
        return self.h.summaries().reshape(self.hi - self.lo, self.rpp, _capi.NSUMMARY)

    def trajectories(self, times):
        """Trajectories on the shared grid `times` (Handle.trajectories), each array shaped [points on this rank,
        replicates_per_point, T, K or H]; -1 where a replicate's run ended before the grid point."""
        return {k: v.reshape((self.hi - self.lo, self.rpp) + v.shape[1:]) for k, v in self.h.trajectories(times).items()}

    def lineages_through_time(self, times):
        """[points on this rank, replicates_per_point, T] lineages through time of every replicate's genealogy."""
        return self.h.lineages_through_time(times).reshape(self.hi - self.lo, self.rpp, -1)

    def counters(self):
        return self.h.get_counters()


def _flat(e):
    """The engine's parameter arrays concatenated in vgsim_upload_params order, as float64."""
    a = e.param_arrays()
    return np.concatenate([np.asarray(a[k], np.float64).ravel() for k in _capi.SOURCE_FIELDS])


def _entry(e, j):
    """Name of entry j of `_flat`, e.g. 'm[0, 1]'."""
    for k in _capi.SOURCE_FIELDS:
        a = e.param_arrays()[k]
        if j < a.size:
            return "%s[%s]" % (k, ", ".join(str(int(i)) for i in np.unravel_index(j, a.shape)))
        j -= a.size
    raise IndexError(j)


def _patch(e, setter, value, before):
    """(indices, values) of the entries of `_flat` that setter(e, value) changes relative to `before` (the engine's
    current arrays, which are put back afterwards).  Entries are compared bit for bit."""
    saved = {k: v.copy() for k, v in e.param_arrays().items()}
    try:
        setter(e, value)
        after = _flat(e)
    finally:
        Sweep._restore(e, saved)
    j = np.flatnonzero(after.view(np.int64) != before.view(np.int64))
    return j, after[j]


def resolve_axes(engine, axes):
    """Patch tables of vgsim_upload_param_grid for `axes` over the engine's parameters: (patch_off, patch_idx,
    patch_val), one patch per axis value in axis order.  Each value's setter runs once, on the base parameters.

    The patches stand for sequential setter calls only when the axes do not interact, so the axes are refused with a
    ValueError naming both when two axes write the same entry, or when an axis's patch changes while another axis is at
    its first or last value (a setter that reads what the other writes).  The diagonal of the migration matrix is left
    out of both checks: the blob derivation recomputes it from the off-diagonals the way close_migration_matrix does.
    Combinations a setter refuses (the migration row rules) are checked per point on the device."""
    base = _flat(engine)
    patches = [[_patch(engine, setter, v, base) for v in values] for setter, values in axes]
    K = engine.popNum
    m0 = sum(engine.param_arrays()[k].size for k in _capi.SOURCE_FIELDS[:_capi.SOURCE_FIELDS.index("m")])
    diag = m0 + np.arange(K) * (K + 1)

    def off_diag(p):
        keep = ~np.isin(p[0], diag)
        return p[0][keep], p[1][keep]

    written = [np.unique(np.concatenate([off_diag(p)[0] for p in ps])) for ps in patches]
    for a in range(len(axes)):
        for b in range(a + 1, len(axes)):
            both = np.intersect1d(written[a], written[b])
            if both.size:
                raise ValueError("Sweep.grid: axes %d and %d both write %s" % (a, b, _entry(engine, both[0])))
    for b, (setter_b, values_b) in enumerate(axes):
        for vb in (values_b[0], values_b[-1]):
            saved = {k: v.copy() for k, v in engine.param_arrays().items()}
            try:
                setter_b(engine, vb)
                state = _flat(engine)
                for a, (setter_a, values_a) in enumerate(axes):
                    if a == b:
                        continue
                    for ia, va in enumerate(values_a):
                        try:
                            j, x = off_diag(_patch(engine, setter_a, va, state))
                        except ValueError:
                            continue   # an inadmissible combination: the device refuses that point
                        j0, x0 = off_diag(patches[a][ia])
                        if not (np.array_equal(j, j0) and np.array_equal(x.view(np.int64), x0.view(np.int64))):
                            raise ValueError("Sweep.grid: axis %d depends on axis %d (its patch for value %r changes "
                                             "when axis %d is %r)" % (a, b, va, b, vb))
            finally:
                Sweep._restore(engine, saved)
    off = np.zeros(sum(len(v) for _, v in axes) + 1, np.int64)
    flat = [p for ps in patches for p in ps]
    off[1:] = np.cumsum([len(j) for j, _ in flat])
    idx = np.concatenate([j for j, _ in flat] + [np.zeros(0, np.int64)]).astype(np.int64)
    val = np.concatenate([x for _, x in flat] + [np.zeros(0)])
    return off, idx, val
