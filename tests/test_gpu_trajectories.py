"""Trajectories and lineages through time on a time grid shared by every replicate (vgsim_trajectories,
vgsim_lineages_through_time).

Oracles: a numpy replay of the exported log (get_chain_events + the MULTITYPE records of get_multievents) from the state
the curves kernel starts from, the existing epidemic curves on a grid equal to the reference's, and the definition of
lineages through time evaluated on the tree get_tree returns.  Every comparison is exact."""
import ctypes

import numpy as np
import pytest
import torch

from scenarios import SCENARIOS
from test_gpu_curves import first_infection, run
from test_gpu_tau import make_engine, warm_state
from vgsim_b200 import _capi
from vgsim_b200._capi import VgsimError
from vgsim_b200.sweep import Sweep

pytestmark = pytest.mark.gpu
BIRTH, DEATH, SAMPLING, MUTATION, SUSCCHANGE, MIGRATION, MULTITYPE = range(7)


def _entries(e, r):
    """Per compartment change of replicate r's log, in log order: (time, deme, haplotype, infectious delta, samplings)."""
    chain = e.get_chain_events(r)
    t, ty = chain[0], chain[1].astype(np.int64)
    hap, pop, nhap, npop = (chain[k].astype(np.int64) for k in (2, 3, 4, 5))
    num = np.ones(len(t), np.int64)
    row = np.arange(len(t))
    multi = np.flatnonzero(ty == MULTITYPE)
    if multi.size:  # expand each MULTITYPE row into its non-zero records
        m = e.get_multievents(r)
        idx = np.concatenate([np.arange(int(chain[2][i]), int(chain[3][i])) for i in multi])
        rows = np.repeat(multi, [int(chain[3][i] - chain[2][i]) for i in multi])
        keep = m["num"][idx] != 0
        idx, rows = idx[keep], rows[keep]
        direct = ty != MULTITYPE
        row = np.concatenate([row[direct], rows])
        order = np.argsort(row, kind="stable")
        row = row[order]
        ty = np.concatenate([ty[direct], m["type"][idx]])[order]
        hap = np.concatenate([hap[direct], m["hap"][idx]])[order]
        pop = np.concatenate([pop[direct], m["pop"][idx]])[order]
        nhap = np.concatenate([nhap[direct], m["nhap"][idx]])[order]
        npop = np.concatenate([npop[direct], m["npop"][idx]])[order]
        num = np.concatenate([num[direct], m["num"][idx]])[order]
    tt = t[row]
    out = []
    for sel, d, h, sign, smp in ((ty == BIRTH, pop, hap, 1, 0), (ty == DEATH, pop, hap, -1, 0),
                                 (ty == SAMPLING, pop, hap, -1, 1), (ty == MUTATION, pop, hap, -1, 0),
                                 (ty == MUTATION, pop, nhap, 1, 0), (ty == MIGRATION, npop, hap, 1, 0)):
        k = np.flatnonzero(sel)
        out.append((k, d[k], h[k], sign * num[k], smp * num[k]))
    k = np.concatenate([o[0] for o in out])
    order = np.argsort(k, kind="stable")
    cat = [np.concatenate([o[i] for o in out])[order] for i in range(1, 5)]
    return (tt[k[order]],) + tuple(cat)


def replay(e, r, I0, grid):
    """[T, 2K + 2H] rows of replicate r on `grid`, replayed on the host."""
    K, H = e.popNum, e.hapNum
    t, d, h, dinf, dsmp = _entries(e, r)
    ct = float(e.counters()["time"][r])
    I = I0.astype(np.int64).copy()
    sd, sh = np.zeros(K, np.int64), np.zeros(H, np.int64)
    rows, done = [], 0
    for g in grid:
        cut = int(np.searchsorted(t, g, side="right"))
        np.add.at(I, (d[done:cut], h[done:cut]), dinf[done:cut])
        np.add.at(sd, d[done:cut], dsmp[done:cut])
        np.add.at(sh, h[done:cut], dsmp[done:cut])
        done = cut
        row = np.concatenate([I.sum(axis=1), I.sum(axis=0), sd, sh])
        rows.append(np.full_like(row, -1) if g > ct else row)
    return np.stack(rows)


def as_rows(traj):
    return np.concatenate([traj[k] for k in ("infectious_deme", "infectious_hap", "sampled_deme", "sampled_hap")], axis=2)


def grid_for(e, R):
    """Before the first row, at row times (direct and leap rows), between the replicates' end times, after all of them."""
    ct = e.counters()["time"]
    pts = [-0.5, 0.0]
    for r in (0, R - 1):
        t = e.get_chain_events(r)[0]
        if len(t):
            pts += [t[len(t) // 3], t[(2 * len(t)) // 3], t[-1]]
    pts += [float(np.median(ct)), float(ct.min()), float(ct.max()), float(ct.max()) + 1.0, float(ct.max()) * 2 + 3.0]
    pts += list(np.linspace(0.0, float(ct.max()) * 1.2, 9))
    return np.unique(np.asarray(pts, np.float64))


def check_replay(e, I0, R):
    grid = grid_for(e, R)
    got = e.trajectories(grid)
    K, H = e.popNum, e.hapNum
    assert got["infectious_deme"].shape == (R, len(grid), K) and got["sampled_hap"].shape == (R, len(grid), H)
    rows = as_rows(got)
    ct = e.counters()["time"]
    assert np.all((rows == -1).all(axis=2) == (grid[None, :] > ct[:, None]))   # the -1 rule, row by row
    assert (rows >= 0).any(axis=2).sum() > 0
    for r in range(R):
        np.testing.assert_array_equal(rows[r], replay(e, r, I0, grid), err_msg="replicate %d" % r)
    assert e._handle.last_kernel_ms() > 0.0
    return grid, rows


@pytest.mark.parametrize("name,seed,direct_t,tau_leaps,tau_t", [("s9", 11, 5.0, 0, None), ("t3small", 5, 50.0, 60, 62.0),
                                                               ("example", 1234, 45.0, 50, 55.0), ("s7", 7, 7.0, 0, None)])
def test_trajectories_equal_log_replay(name, seed, direct_t, tau_leaps, tau_t):
    """Direct rows (s9; s7 with lockdowns), direct + dense tau rows (t3small, example)."""
    R = 4
    e, Sx0, I0 = run(name, seed, R, direct_t, tau_leaps, tau_t)
    if tau_leaps:
        assert (e.counters()["leaps"] > 0).all()
    check_replay(e, I0, R)


def test_trajectories_on_tau_only_log():
    """A log of tau leaps only (t3small from a warm state)."""
    R = 3
    Sx0, I0 = warm_state("t3small", 5, 60.0)
    e = make_engine("t3small", 5, replicates=R)
    e._susceptible[...] = Sx0
    e._infectious[...] = I0
    e.SimulatePopulation_tau(40, 10 ** 9, -1, 1)
    check_replay(e, I0, R)


def test_trajectories_on_archived_leaps():
    R = 3
    Sx0, I0 = warm_state("t3small", 9, 60.0)
    e = make_engine("t3small", 9, replicates=R)
    e._susceptible[...] = Sx0
    e._infectious[...] = I0
    e.SimulatePopulation_tau(60, 10 ** 9, -1, 1, leap_block=8)
    assert e._handle.archive_stats()["leaps_archived"] > 0
    check_replay(e, I0, R)


def test_trajectories_large_state_direct():
    """large_9_1_1: 2 MB of infectious counts per replicate, replayed in device scratch slices."""
    from scenarios_large import make_engine as make_large
    R = 2
    e = make_large("large_9_1_1", 3, replicates=R)
    _, I0 = first_infection(e._susceptible, e._infectious)
    e.SimulatePopulation(2500, 10 ** 9, -1, 200)
    ct = e.counters()["time"]
    t0 = e.get_chain_events(0)[0]
    assert len(t0) > 10
    grid = np.unique(np.concatenate([[0.0], t0[[len(t0) // 10, len(t0) // 2]], np.linspace(0, ct.max() * 1.1, 5)]))
    rows = as_rows(e.trajectories(grid))
    for r in range(R):
        np.testing.assert_array_equal(rows[r], replay(e, r, I0, grid))


@pytest.mark.parametrize("name,seed,direct_t,tau_leaps,tau_t", [("s9", 13, 5.0, 0, None), ("t3small", 5, 50.0, 60, 62.0)])
def test_trajectories_equal_curve_marginals(name, seed, direct_t, tau_leaps, tau_t):
    """On replicate r's own reference grid (j * currentTime) / step_num, the rows are the deme and haplotype sums of
    epidemic_curves' infectious and sampled outputs."""
    R, steps = 3, 29
    e, _, _ = run(name, seed, R, direct_t, tau_leaps, tau_t)
    c = e.epidemic_curves(steps, want=("infectious", "sampled"))
    ct = e.counters()["time"]
    for r in range(R):
        grid = (np.arange(steps + 1, dtype=np.float64) * ct[r]) / steps
        np.testing.assert_array_equal(grid, c["time_points"][r])
        got = e.trajectories(grid)
        np.testing.assert_array_equal(got["infectious_deme"][r], c["infectious"][r].sum(axis=2))
        np.testing.assert_array_equal(got["infectious_hap"][r], c["infectious"][r].sum(axis=1))
        np.testing.assert_array_equal(got["sampled_deme"][r], c["sampled"][r].sum(axis=2))
        np.testing.assert_array_equal(got["sampled_hap"][r], c["sampled"][r].sum(axis=1))


def test_trajectories_dev_pointer_holds_the_same_rows():
    R = 3
    e, _, _ = run("s9", 3, R, 4.0)
    grid = np.linspace(0.0, 5.0, 11)
    host = as_rows(e.trajectories(grid))
    ptr = e._handle.trajectories_dev_ptr(grid)

    class _Dev:
        __cuda_array_interface__ = {"shape": host.shape, "typestr": "<i8", "data": (int(ptr), False), "version": 2,
                                    "strides": None}
    np.testing.assert_array_equal(torch.as_tensor(_Dev(), device="cuda").cpu().numpy(), host)


# ---------------------------------------------------------------------------------------------- lineages through time
def ltt_ref(parent, time, grid):
    tp = np.where(parent >= 0, time[np.maximum(parent, 0)], -np.inf)
    return np.array([np.count_nonzero((time >= g) & (tp < g)) for g in grid], np.int64)


def check_ltt(e, R):
    s = e._handle.summaries()
    grid = [-1.0]
    for r in range(R):
        if s[r, 13] > 0:
            _, t = e.get_tree(r)
            grid += list(np.sort(t)[:: max(1, len(t) // 7)]) + [t.min(), t.max(), t.max() + 0.5]
    grid = np.unique(np.asarray(grid, np.float64))
    got = e.lineages_through_time(grid)
    assert got.shape == (R, len(grid)) and got.dtype == np.int64
    for r in range(R):
        if s[r, 13] == 0:
            assert not got[r].any()
            continue
        tree, t = e.get_tree(r)
        np.testing.assert_array_equal(got[r], ltt_ref(tree, t, grid), err_msg="replicate %d" % r)
    assert (s[:, 13] > 0).any()
    return s, got


def test_ltt_direct_genealogy():
    R = 5
    e, _, _ = run("s9", 21, R, 5.0)
    with pytest.raises(VgsimError, match="genealogy"):
        e._handle.lineages_through_time([0.0, 1.0])
    e.GetGenealogy(7)
    s, got = check_ltt(e, R)
    # before the root a fully coalesced tree has the root's one lineage
    full = np.flatnonzero(s[:, 16] == 1)
    assert full.size and (got[full, 0] == 1).all()


def test_ltt_tau_genealogy_from_the_archive():
    R = 4
    Sx0, I0 = warm_state("t3small", 5, 60.0)
    e = make_engine("t3small", 5, replicates=R)
    e._susceptible[...] = Sx0
    e._infectious[...] = I0
    e.SimulatePopulation_tau(60, 10 ** 9, -1, 1, leap_block=8)
    assert e._handle.archive_stats()["leaps_archived"] > 0
    e.GetGenealogy(3)
    check_ltt(e, R)


def test_ltt_forest():
    """A log that starts with many infectious: lineages that reach the start of the log uncoalesced stay roots."""
    R = 6
    e = make_engine("s9", 31, replicates=R)
    e._infectious[0, 0] = 40
    e._susceptible[0, 0] -= 40
    e.SimulatePopulation(300, 10 ** 9, -1, 200)
    e.GetGenealogy(5)
    s, got = check_ltt(e, R)
    assert (s[:, 16] > 1).any()
    r = int(np.flatnonzero(s[:, 16] > 1)[0])
    assert got[r, 0] == s[r, 16]   # the grid starts before the roots (-1.0): every root's lineage counts


def test_ltt_at_the_world_tree_size():
    """Genealogies of 1e5 samples (2e5 nodes, the tree size of BASELINE.json's world configuration)."""
    from vgsim_b200._engine import BirthDeathModel as Eng
    R = 2
    e = Eng(0, 1, 1, 17, False, False, int(1e6), 0.0, replicates=R)
    e.set_transmission_rate(2.0, None)
    e.set_recovery_rate(0.5, None)
    e.set_sampling_rate(1.0, None)
    e.SimulatePopulation(10 ** 7, 100000, -1, 200)
    e.GetGenealogy(11)
    s, _ = check_ltt(e, R)
    assert s[:, 13].max() >= 2e5 - 1


# ---------------------------------------------------------------------------------------------- validation, sharding
def test_grid_errors_from_the_c_abi():
    e, _, _ = run("s9", 11, 2, 3.0)
    h = e._handle
    out = np.zeros(64 * 2 * (h.K + h.H), np.int64)
    for fn in (_capi.lib.vgsim_trajectories, _capi.lib.vgsim_lineages_through_time):
        if fn is _capi.lib.vgsim_lineages_through_time:
            e.GetGenealogy(1)
        for bad, msg in (([1.0, 1.0], "strictly increasing"), ([0.0, 2.0, 1.0], "strictly increasing"),
                         ([0.0, np.nan], "not finite"), ([np.inf], "not finite"), ([], "at least one point")):
            t = np.ascontiguousarray(bad if bad else [0.0], np.float64)
            assert fn(h._h, t.ctypes.data_as(ctypes.c_void_p), len(bad), out.ctypes.data_as(ctypes.c_void_p)) != 0
            assert msg in _capi.lib.vgsim_last_error().decode()
    big = np.arange(40000, dtype=np.float64)
    assert _capi.lib.vgsim_lineages_through_time(h._h, big.ctypes.data_as(ctypes.c_void_p), len(big), None) != 0
    assert "at most 32768" in _capi.lib.vgsim_last_error().decode()
    with pytest.raises(ValueError, match="strictly increasing"):
        e.trajectories([0.0, 0.0])


def test_sharding_does_not_change_trajectories():
    dims, setup = SCENARIOS["t3small"]
    B = np.linspace(1.2, 4.0, 6) * 0.1
    MIG = np.logspace(-4, -1, 4)
    grid = np.append(np.linspace(0.0, 120.0, 25), 1e6)

    def run_rank(rank, world):
        sw = Sweep.grid(dims, setup, [(lambda e, v: e.set_transmission_rate(float(v), None), B),
                                      (lambda e, v: e.set_total_migration_probability(float(v)), MIG)],
                        replicates_per_point=2, seed=5, rank=rank, world=world)
        sw.simulate(1500, 10 ** 9, -1, "direct")
        sw.simulate(12, 10 ** 9, -1, "tau")
        sw.genealogy(seed=np.arange(sw.lo * 2, sw.hi * 2, dtype=np.uint64) + np.uint64(900))
        return sw.trajectories(grid), sw.lineages_through_time(grid)

    parts = {w: [run_rank(g, w) for g in range(w)] for w in (1, 2, 3)}
    whole_t, whole_l = parts[1][0]
    assert whole_l.shape == (len(B) * len(MIG), 2, len(grid))
    assert whole_t["infectious_hap"].shape == (len(B) * len(MIG), 2, len(grid), 4 ** dims[0])
    for w in (2, 3):
        for k in whole_t:
            np.testing.assert_array_equal(np.concatenate([p[0][k] for p in parts[w]], axis=0), whole_t[k])
        np.testing.assert_array_equal(np.concatenate([p[1] for p in parts[w]], axis=0), whole_l)
    assert (whole_l > 1).any() and (whole_t["sampled_deme"] > 0).any() and (whole_t["infectious_deme"] == -1).any()
