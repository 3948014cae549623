"""Sweep.grid on the host: the axes resolve into patches that compose like sequential setter calls, the grid defines
the same global point list and rank slices as the callable Sweep, and interacting axes are refused.  The handle is
replaced by a recorder that composes the grid's points on the host the way vgsim_upload_param_grid documents it, so
no GPU is needed."""
import numpy as np
import pytest

from scenarios import SCENARIOS
from vgsim_b200 import _capi, sweep as sweep_mod
from vgsim_b200._engine import BirthDeathModel as Eng
from vgsim_b200.sweep import Sweep, resolve_axes

B = np.linspace(1.2, 4.0, 5) * 0.1
MIG = np.logspace(-4, -1, 3)
AXES = [(lambda e, v: e.set_transmission_rate(v, None), B), (lambda e, v: e.set_total_migration_probability(v), MIG)]


def mk(b, m):
    def f(e):
        e.set_transmission_rate(float(b), None)
        e.set_total_migration_probability(float(m))
    return f


class Recorder:
    """Stands in for _capi.Handle: keeps every point's source arrays (concatenated, fp64) and the other uploads."""

    def __init__(self, sites, K, S, replicates=1, param_points=1, device=None):
        self.K, self.R, self.n_pp = K, replicates, param_points
        self.src = [None] * param_points

    def set_replicate_params(self, m):
        self.map = np.array(m)

    def upload_params(self, pp, a):
        self.src[pp] = np.concatenate([np.asarray(a[k], np.float64).ravel() for k in _capi.SOURCE_FIELDS])

    def upload_param_grid(self, base_pp, axis_len, off, idx, val, first_point, dst_pp0, n_points):
        base = self.src[base_pp].copy()
        for i in range(n_points):
            x, rem, start = base.copy(), first_point + i, np.cumsum([0] + list(axis_len))
            coords = np.unravel_index(rem, tuple(axis_len)) if len(axis_len) else ()
            for a, c in enumerate(coords):
                j = start[a] + c
                x[idx[off[j]:off[j + 1]]] = val[off[j]:off[j + 1]]
            self.src[dst_pp0 + i] = x

    def set_seeds(self, s):
        self.seeds = np.array(s)

    def set_state(self, Sx, I):
        self.state = (Sx.copy(), I.copy())


@pytest.fixture
def recorder(monkeypatch):
    monkeypatch.setattr(sweep_mod._capi, "Handle", Recorder)


def m_offset(dims):
    U, K, S = dims
    e = Eng(U, K, S, 1, False, False, int(1e6), 0.0)
    a = e.param_arrays()
    return sum(a[k].size for k in _capi.SOURCE_FIELDS[:_capi.SOURCE_FIELDS.index("m")])


def closed(x, mo, K):
    """x with the migration diagonal recomputed from the off-diagonals (what the blob derivation does)."""
    x = x.copy()
    m = x[mo:mo + K * K].reshape(K, K)
    for p in range(K):
        stay = 1.0
        for q in range(K):
            if q != p:
                stay -= m[p, q]
        m[p, p] = stay
    return x


@pytest.mark.parametrize("world", [1, 3, 8])
def test_grid_matches_the_callable_list(recorder, world):
    dims, setup = SCENARIOS["table3_k10"]
    pts = [mk(b, m) for b in B for m in MIG]
    mo = m_offset(dims)
    for rank in range(world):
        g = Sweep.grid(dims, setup, AXES, replicates_per_point=2, seed=11, rank=rank, world=world)
        c = Sweep(dims, setup, pts, replicates_per_point=2, seed=11, rank=rank, world=world)
        assert (g.n_global, g.lo, g.hi, g.R) == (c.n_global, c.lo, c.hi, c.R)
        assert np.array_equal(g.h.seeds, c.h.seeds) and np.array_equal(g.h.map, c.h.map)
        assert all(np.array_equal(a, b) for a, b in zip(g.h.state, c.h.state))
        for pp in range(g.hi - g.lo):
            assert np.array_equal(closed(g.h.src[pp], mo, dims[1]).view(np.int64), c.h.src[pp].view(np.int64))


def test_patch_is_the_callable_diff():
    dims, setup = SCENARIOS["w"]
    e = Eng(*dims, 1, False, False, int(1e6), 0.0)
    setup(e)
    base = sweep_mod._flat(e)
    off, idx, val = resolve_axes(e, [(lambda e, v: e.set_sampling_multiplier(v, 3), [0.5, 2.0]),
                                     (lambda e, v: e.set_npi(list(v), None), [(0.2, 0.02, 0.001)])])
    assert np.array_equal(sweep_mod._flat(e), base)            # the base is left as it was
    assert list(np.diff(off)) == [1, 1, 3 * dims[1]]
    for j, f in enumerate([lambda x: x.set_sampling_multiplier(0.5, 3), lambda x: x.set_sampling_multiplier(2.0, 3),
                           lambda x: x.set_npi([0.2, 0.02, 0.001], None)]):
        x = Eng(*dims, 1, False, False, int(1e6), 0.0)
        setup(x)
        f(x)
        want = sweep_mod._flat(x)
        changed = np.flatnonzero(want != base)
        assert np.array_equal(idx[off[j]:off[j + 1]], changed)
        assert np.array_equal(val[off[j]:off[j + 1]], want[changed])


def test_two_axes_writing_one_entry_are_refused(recorder):
    dims, setup = SCENARIOS["t3small"]
    axes = [(lambda e, v: e.set_total_migration_probability(v), [0.01, 0.02]),
            (lambda e, v: e.set_migration_probability(v, 0, 1), [0.001, 0.002])]
    with pytest.raises(ValueError, match=r"axes 0 and 1 both write m\[0, 1\]"):
        Sweep.grid(dims, setup, axes)


def test_dependent_axes_are_refused(recorder):
    dims, setup = SCENARIOS["t3small"]

    def sampling_mode(e):
        setup(e)
        e._sampling_probability = True
    # in sampling-probability mode set_sampling_rate splits d + s, which the recovery-rate axis writes
    axes = [(lambda e, v: e.set_sampling_rate(v, None), [0.1, 0.3]), (lambda e, v: e.set_recovery_rate(v, None), [0.1, 0.2])]
    with pytest.raises(ValueError, match="axes 0 and 1"):
        Sweep.grid(dims, sampling_mode, axes)
    # an axis that reads (but does not write) what another axis writes
    axes = [(lambda e, v: e.set_transmission_rate(v, None), [0.2, 0.4]),
            (lambda e, v: e.set_sampling_rate(v * e.bRate[0], None), [0.01, 0.02])]
    with pytest.raises(ValueError, match="axis 1 depends on axis 0"):
        Sweep.grid(dims, setup, axes)


def test_migration_diagonal_is_exempt(recorder):
    """Two axes on the same migration row both rewrite its diagonal; the diagonal is recomputed from the off-diagonals,
    so the grid is accepted and equals the callable list."""
    dims, setup = SCENARIOS["t3small"]
    V0, V1 = [0.01, 0.05, 0.1], [0.02, 0.2]
    axes = [(lambda e, v: e.set_migration_probability(v, 0, 1), V0), (lambda e, v: e.set_migration_probability(v, 0, 2), V1)]
    g = Sweep.grid(dims, setup, axes)

    def pt(a, b):
        return lambda e: (e.set_migration_probability(a, 0, 1), e.set_migration_probability(b, 0, 2))
    c = Sweep(dims, setup, [pt(a, b) for a in V0 for b in V1])
    mo = m_offset(dims)
    off, idx, _ = resolve_axes(g.engine, axes)
    assert mo in idx[off[0]:off[1]] and mo in idx[off[3]:off[4]]     # m[0, 0] is in the patches of both axes
    for pp in range(len(V0) * len(V1)):
        assert np.array_equal(closed(g.h.src[pp], mo, dims[1]).view(np.int64), c.h.src[pp].view(np.int64))
