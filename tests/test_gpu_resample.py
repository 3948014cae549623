"""Resampling on the device (vgsim_resample): replicate r's whole run -- state, counters, logs, archive, lockdown
records -- becomes the run of replicate source[r]; the seed and the parameter point stay with r.

A clone given its source's seed must then continue exactly like the source (every per-replicate output bit for bit);
with its own seed it is an independent continuation of the same history (the prefix of its log is the source's, the
rest replays to its state, and its law is the oracle's law started from the source's state).
"""
import numpy as np
import pytest

import oracle_pool
from oracle import oracle as O
from scenarios import SCENARIOS
from test_gpu_archive import _same, _snapshot
from test_gpu_curves import check_true_counts, first_infection
from test_gpu_direct import _replay_direct
from test_gpu_direct_large import make_engine as make_any_engine
from test_gpu_tau import _ks_all, _replay_dense_log, make_engine, warm_state
from test_gpu_trajectories import check_replay
from vgsim_b200._capi import COUNTER_NAMES, VgsimError
from vgsim_b200._interface import Simulator
from vgsim_b200.resample import systematic_map
from vgsim_b200.sweep import Sweep

pytestmark = pytest.mark.gpu
SRC6 = np.array([0, 0, 2, 2, 4, 4], np.int32)
BIG = 10 ** 9


def _rows(h, times):
    """Every per-replicate output except the genealogy, one dict per replicate."""
    R = h.R
    c = h.get_counters()
    Sx, I, cd, lock = h.get_state(full=True)
    curves = h.epidemic_curves(12)
    traj = h.trajectories(times)
    out = []
    for r in range(R):
        out.append({"counters": np.array([c[k][r] for k in COUNTER_NAMES]), "time": c["time"][r], "Sx": Sx[r],
                    "I": I[r], "cd": cd[r], "lock": lock[r], "events": h.get_event_log(r), "tau": h.get_tau_log(r),
                    "multi": h.get_multievents(r), "lockdowns": h.get_lockdowns(r),
                    "curves": {k: v[r] for k, v in curves.items()}, "traj": {k: v[r] for k, v in traj.items()}})
    return out


def _genealogy_rows(h, times, seeds):
    h.genealogy(seeds)
    summ = h.summaries()
    ltt = h.lineages_through_time(times)
    return [{"tree": h.get_tree(r), "mut": h.get_mutations(r), "mig": h.get_migrations(r), "summary": summ[r],
             "ltt": ltt[r]} for r in range(h.R)]


def _direct(t):
    return lambda h: h.simulate_direct(10 ** 6, BIG, t, 200)


def _tau(leaps, t=-1.0):
    return lambda h: h.simulate_tau(leaps, BIG, t, 200)


def _blocks(leaps):
    return lambda h: h.simulate_tau_blocks(leaps, BIG, -1.0, 1, leap_block=40)


def _then(*fs):
    def f(h):
        for g in fs:
            g(h)
    return f


# name, seed, warm-up state (oracle direct to t, or None: the scenario's own start), tau variant, phase 1, phase 2
PATHS = {
    "direct_s9": ("s9", 11, None, 0, _direct(3.0), _direct(5.0)),
    "direct_lockdowns": ("example", 1234, None, 0, _direct(45.0), _direct(90.0)),
    "direct_large": ("large_6_2_2", 3, None, 0, lambda h: h.simulate_direct(1500, BIG, -1.0, 200),
                     lambda h: h.simulate_direct(1500, BIG, -1.0, 200)),
    "tau_warp": ("t3small", 5, None, 8, _then(_direct(50.0), _tau(30, 56.0)), _tau(30, 62.0)),
    "tau_team": ("t3small", 5, None, 4, _then(_direct(50.0), _tau(30, 56.0)), _tau(30, 62.0)),
    "blocks_fork_before_archive": ("table3_k10", 7, 60.0, 0, _tau(60), _blocks(90)),
    "blocks_fork_after_archive": ("table3_k10", 7, 60.0, 0, _blocks(90), _blocks(90)),
    "before_first_simulate": ("t3small", 5, 60.0, 0, None, _then(_direct(4.0), _tau(20))),
}


def _forked(path, seed_clones=True):
    """Six replicates through phase 1, forked with SRC6, clones given their sources' seeds, through phase 2."""
    name, seed, warm, variant, phase1, phase2 = PATHS[path]
    R = len(SRC6)
    e = make_any_engine(name, seed, replicates=R)
    if warm is not None:
        Sx0, I0 = warm_state(name, seed, warm)
        e._susceptible[...] = Sx0
        e._infectious[...] = I0
    h = e._sync_params()
    if variant:
        h.set_tau_variant(variant)
    if phase1 is None:  # distinct configured states: the fork must copy them
        Sx, I = h.get_state()
        for r in range(R):
            I[r, r % e.popNum, 0] += 1 + r
            Sx[r, r % e.popNum, np.argmax(Sx[r, r % e.popNum])] -= 1 + r
        h.set_state(Sx, I)
    else:
        phase1(h)
    h.synchronize()
    before = h.get_counters()
    n0 = h.launch_count()
    h.resample(SRC6)
    assert h.launch_count() == n0 + 1
    if seed_clones:
        h.set_seeds(np.uint64(seed) + SRC6.astype(np.uint64))
    phase2(h)
    h.synchronize()
    return e, h, before


@pytest.mark.parametrize("path", list(PATHS))
def test_clone_with_the_source_seed_continues_like_the_source(path):
    e, h, before = _forked(path)
    after = h.get_counters()
    assert (after["events"] > before["events"]).any(), "phase 2 did nothing"
    if path == "direct_lockdowns":
        assert sum(len(h.get_lockdowns(r)[0]) for r in range(h.R)) > 0
    times = np.linspace(0.0, float(after["time"].max()) * 1.1 + 0.5, 17)
    rows = _rows(h, times)
    gs = np.uint64(4242) + SRC6.astype(np.uint64)
    fwd = _genealogy_rows(h, times, None)           # the forward key: the replicates' own (equal) seeds
    _, h2, _ = _forked(path)                         # a twin for the second genealogy (the replay rewinds I, Q9)
    explicit = _genealogy_rows(h2, times, gs)
    assert any(len(t["tree"][0]) > 1 for t in fwd)
    for r in range(h.R):
        s = int(SRC6[r])
        _same(rows[r], rows[s], "replicate %d vs %d" % (r, s))
        _same(fwd[r], fwd[s], "forward-key genealogy %d vs %d" % (r, s))
        _same(explicit[r], explicit[s], "explicit-seed genealogy %d vs %d" % (r, s))


def test_prefix_is_kept_and_clones_diverge():
    R = 6
    e = make_engine("s9", 11, replicates=R)
    Sx0, I0 = first_infection(e._susceptible, e._infectious)
    e.SimulatePopulation(10 ** 6, BIG, 3.0, 200)
    c = e.counters()
    s = int(np.argmax(c["globalInfectious"]))
    assert c["globalInfectious"][s] > 0
    prefix = e.get_chain_events(s)
    e.resample(np.full(R, s))
    assert np.array_equal(e._infectious, e._handle.get_state()[1][s])
    e.SimulatePopulation(10 ** 6, BIG, 5.0, 1)
    c = e.counters()
    Sx_f, I_f = e._handle.get_state()
    tails = set()
    for r in range(R):
        chain = e.get_chain_events(r)
        assert chain.shape[1] > prefix.shape[1]
        np.testing.assert_array_equal(chain[:, :prefix.shape[1]], prefix, err_msg="replicate %d" % r)
        Sx, I = _replay_direct(e, chain, Sx0, I0)
        assert np.array_equal(Sx, Sx_f[r]) and np.array_equal(I, I_f[r])
        tails.add(chain[:, prefix.shape[1]:].tobytes())
    assert len(tails) == R  # every replicate kept its own seed: six different continuations
    check_true_counts(e, R)
    check_replay(e, I0, R)


def test_tau_continuation_of_clones_replays():
    """Clones continued by tau leaps: the dense log after the fork replays from the source's state at the fork."""
    R = 5
    Sx0, I0 = warm_state("t3small", 5, 60.0)
    e = make_engine("t3small", 5, replicates=R)
    e._susceptible[...] = Sx0
    e._infectious[...] = I0
    h = e._sync_params()
    h.simulate_direct(3000, BIG, -1.0, 1)
    c = h.get_counters()
    s = int(np.argmax(c["globalInfectious"]))
    Sx_s, I_s = (x[s] for x in h.get_state())
    h.recycle_log()  # the log starts at the fork: _replay_dense_log replays tau rows only
    h.resample(np.full(R, s, np.int32))
    h.simulate_tau(60, -1, -1.0, 1)
    Sx_f, I_f = h.get_state()
    for r in range(R):
        Sx, I, _, _ = _replay_dense_log(e, h, r, Sx_s, I_s)
        assert np.array_equal(Sx, Sx_f[r]) and np.array_equal(I, I_f[r])
    assert len({I_f[r].tobytes() for r in range(R)}) > 1


def test_fork_into_parameter_points():
    dims, setup = SCENARIOS["t3small"]
    bs = [0.2, 0.45]
    sw = Sweep.grid(dims, setup, [(lambda e, v: e.set_transmission_rate(v, None), bs)], replicates_per_point=3, seed=9)
    sw.simulate(2500, BIG, -1, "direct")
    I = sw.h.get_state()[1]
    s = int(np.argmax(I.sum(axis=(1, 2))))
    sw.resample(np.full(sw.R, s))
    Sx, I, cd, lock = sw.h.get_state(full=True)
    assert I[s].sum() > 0
    for r in range(sw.R):
        assert np.array_equal(I[r], I[s]) and np.array_equal(Sx[r], Sx[s]) and np.array_equal(cd[r], cd[s])
        e = make_engine("t3small", 1)
        e.set_transmission_rate(bs[r // 3], None)
        e._susceptible[...] = Sx[r]
        e._infectious[...] = I[r]
        e.contactDensity[...] = cd[r]
        want = O.OracleModel.from_engine(e).propensities()[0]
        got = sw.h.propensities(r)[0]
        assert np.array_equal(got == 0, want == 0)
        nz = want != 0
        assert (np.abs(got[nz] - want[nz]) / np.abs(want[nz])).max() < 1e-12, r
    # the two points then run apart: faster transmission, more births
    sw.simulate(4000, BIG, -1, "direct")
    b = sw.counters()["bCounter"].reshape(2, 3)
    assert b[1].mean() > b[0].mean()


@pytest.mark.parametrize("method", ["tau", "direct"])
def test_clone_distribution_matches_oracle_from_the_source_state(method):
    name, seed, t0, R = "t3small", 5, 50.0, 1500
    e = make_engine(name, seed, replicates=R)
    h = e._sync_params()
    h.simulate_direct(10 ** 6, BIG, t0, 1)
    c0 = h.get_counters()
    s = int(np.argmax(c0["globalInfectious"]))
    h.resample(np.full(R, s, np.int32))
    Sx_s, I_s = (x[s] for x in h.get_state())
    t_s = float(c0["time"][s])
    keys = ["bCounter", "dCounter", "sCounter", "mCounter", "iCounter", "migPlus", "time", "inf_total", "inf_deme0"]
    if method == "tau":
        dt = 6.0
        h.simulate_tau(100, -1, t_s + dt, 1)  # iterations <= 100: no extinction restart; the time limit binds first
        ora = oracle_pool.run("tau", name, range(1000, 1000 + R), state=(Sx_s, I_s), iterations=50,
                              epidemic_time=dt)  # 50 there == 100 here (quirk Q3, test_tau_distribution_matches_oracle)
        keys.append("leaps")
    else:
        N = 1500
        h.simulate_direct(N, BIG, -1.0, 1)
        ora = oracle_pool.run("direct", name, range(1000, 1000 + R), state=(Sx_s, I_s), iterations=N, sample_size=BIG,
                              attempts=1)
    c = h.get_counters()
    Sx_f, I_f = h.get_state()
    dev = {k: c[k] - c0[k][s] for k in keys if k in c}
    dev["time"] = c["time"] - t_s
    if method == "tau":
        dev["leaps"] = c["leaps"] - c0["leaps"][s]
        ora["leaps"] = ora["events"]
    dev["inf_total"] = I_f.sum(axis=(1, 2))
    dev["inf_deme0"] = I_f[:, 0, :].sum(axis=1)
    bad = _ks_all(dev, ora, keys)
    assert not bad, bad


def _cheap_snapshot(h):
    c = h.get_counters()
    return {"counters": c, "state": h.get_state(full=True), "events": [h.get_event_log(r) for r in range(h.R)],
            "tau": [h.get_tau_log(r) for r in range(h.R)]}


def test_refused_maps_change_nothing():
    R = 6
    e = make_engine("t3small", 5, replicates=R)
    h = e._sync_params()
    h.simulate_direct(10 ** 6, BIG, 40.0, 200)
    h.simulate_tau(10, BIG, -1.0, 1)
    h.synchronize()
    snap = _cheap_snapshot(h)
    n0 = h.launch_count()
    bad = np.arange(R, dtype=np.int32)
    bad[2] = R
    with pytest.raises(VgsimError, match="replicate 2 copies from 6: replicate out of range"):
        h.resample(bad)
    bad[2] = -1
    with pytest.raises(VgsimError, match="replicate 2 copies from -1: replicate out of range"):
        h.resample(bad)
    chain = np.array([0, 0, 1, 3, 4, 5], np.int32)
    with pytest.raises(VgsimError, match="replicate 2 copies from 1, which copies from 0"):
        h.resample(chain)
    assert h.launch_count() == n0
    _same(snap, _cheap_snapshot(h), "after refused maps")
    with pytest.raises(ValueError):
        e.resample(np.zeros(R - 1, np.int64))
    with pytest.raises(ValueError):
        e.resample(np.zeros(R, np.float64))
    # the identity map enqueues nothing
    h.resample(np.arange(R))
    assert h.launch_count() == n0


def test_identity_map_changes_nothing():
    R = 6

    def twin(identity):
        e = make_engine("t3small", 5, replicates=R)
        h = e._sync_params()
        h.simulate_direct(10 ** 6, BIG, 50.0, 200)
        h.simulate_tau(30, BIG, -1.0, 200)
        h.archive_tau_log()
        if identity:
            n0 = h.launch_count()
            h.resample(np.arange(R))
            assert h.launch_count() == n0
        h.simulate_tau(20, BIG, -1.0, 200)
        return _snapshot(e, h, 31)

    _same(twin(False), twin(True), "identity map")


def test_ltt_after_resample_fails_like_after_simulate():
    R = 4
    e = make_engine("s9", 11, replicates=R)
    h = e._sync_params()
    h.simulate_direct(10 ** 6, BIG, 5.0, 200)
    h.genealogy(7)
    grid = np.linspace(0.0, 5.0, 6)
    assert h.lineages_through_time(grid).shape == (R, 6)
    assert h.summaries()[:, 13].max() > 0
    h.resample(np.array([0, 0, 2, 3], np.int32))
    with pytest.raises(VgsimError, match="no genealogy"):
        h.lineages_through_time(grid)
    assert np.all(h.summaries()[:, 13:22] == 0)


def test_simulator_resample_refreshes_the_host_mirror():
    (U, K, S), setup = SCENARIOS["s9"]
    sim = Simulator(U, K, S, seed=3, replicates=4, verbose=False)
    setup(sim.simulation)
    sim.simulate(10 ** 6, BIG, 4.0, "direct")
    I = sim.simulation._handle.get_state()[1]
    s = 1 + int(np.argmax(I[1:].sum(axis=(1, 2))))
    sim.resample(np.full(4, s))
    assert np.array_equal(sim.infectious, I[s])   # the property shows replicate 0, which now holds the run of s
    # after genealogy() the replicates hold the rewound infectious counts (quirk Q9), and that is what is copied
    sim.genealogy(5)
    rewound = sim.simulation._handle.get_state()[1]
    sim.resample(np.full(4, s))
    assert np.array_equal(sim.infectious, rewound[s])
    with pytest.raises(RuntimeError, match="Genealogy was not simulated"):
        sim.get_tree(0)


def test_systematic_map_drives_a_filter_step():
    """A particle-filter step end to end: weights from the trajectories, systematic_map, resample."""
    R = 64
    e = make_engine("t3small", 5, replicates=R)
    e.SimulatePopulation(10 ** 6, BIG, 40.0, 200)
    grid = np.array([20.0, 30.0, 40.0])
    inf = e.trajectories(grid)["infectious_deme"].sum(axis=2)[:, -1]
    w = np.exp(-0.5 * ((inf - np.median(inf)) / (inf.std() + 1.0)) ** 2)
    src = systematic_map(w, 0.37)
    before = e._handle.get_state()[1]
    e.resample(src)
    after = e._handle.get_state()[1]
    for r in range(R):
        assert np.array_equal(after[r], before[src[r]])
    e.SimulatePopulation_tau(20, BIG, 45.0, 200)
    check_true_counts(e, R)
