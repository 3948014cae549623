"""GPU tests of the large-state direct kernel (csrc/direct_large_kernel.cu): model shapes whose direct-method rate
hierarchy does not fit one SM's shared memory, and every shape with vgsim_set_direct_variant bit 0.

The kernel keeps each replicate's rates in 32-ary sum trees in device memory and draws from its own Philox stream, so
it matches the reference (the CPU oracle) in distribution and its rate trees match UpdateAllRates to 1e-12; the
downstream consumers (genealogy replay, curves, exporters) are checked bit for bit on its logs."""
import numpy as np
import pytest

from oracle import oracle as O
import oracle_pool
from vgsim_b200 import Simulator
from vgsim_b200._capi import VgsimError
import scenarios_large
from scenarios_large import LARGE_SCENARIOS
from test_gpu_tau import make_engine as make_small_engine, warm_state as warm_small_state, _ks_all
from test_gpu_direct import _replay_direct
from test_gpu_genealogy import assert_same_genealogy, pcg
from test_gpu_curves import check_true_counts, first_infection, STEPS

pytestmark = pytest.mark.gpu

LARGE = ["large_6_2_2", "large_7_1_2", "large_9_1_1", "large_4_100_3", "large_0_4096_1"]


def make_engine(name, seed=1, replicates=1):
    """A scenario of tests/scenarios_large.py or tests/scenarios.py by name."""
    if name in LARGE_SCENARIOS:
        return scenarios_large.make_engine(name, seed, replicates)
    return make_small_engine(name, seed, replicates)


def warm_state(name, seed, t_end):
    """A mid-epidemic state produced by the oracle's direct method (test_gpu_tau.warm_state for any scenario)."""
    if name not in LARGE_SCENARIOS:
        return warm_small_state(name, seed, t_end)
    om = O.OracleModel.from_engine(make_engine(name, seed))
    om.simulate(10**7, sample_size=10**9, epidemic_time=t_end)
    return om.get_state()


def oracle_direct(name, seeds, N):
    """The oracle's counters and total infectious over `seeds`, run on all host cores (tests/oracle_pool.py's pool)."""
    if name not in LARGE_SCENARIOS:
        return oracle_pool.run("direct", name, seeds, iterations=N, sample_size=N)
    seeds = list(seeds)
    pool = oracle_pool._pool()
    nchunk = max(1, min(len(seeds), 4 * pool._processes))
    out = {}
    for r in pool.map(scenarios_large.oracle_direct, [(name, seeds[i::nchunk], N) for i in range(nchunk)]):
        for k, v in r.items():
            out.setdefault(k, []).extend(v)
    return {k: np.asarray(v) for k, v in out.items()}


def _check_rates(e):
    dev = e.rates()
    ora = O.OracleModel.from_engine(e).rates()
    for k in ("A", "eff", "maxEBM", "ev", "hp", "popRate", "migPop", "totals"):
        a, b = dev[k], ora[k]
        assert np.array_equal(a == 0, b == 0), k
        nz = b != 0
        if nz.any():
            assert (np.abs(a[nz] - b[nz]) / np.abs(b[nz])).max() < 1e-12, k


@pytest.mark.parametrize("name,seed,t_end", [("large_6_2_2", 3, 2.5), ("large_7_1_2", 4, 3.5)])
def test_large_rates_match_oracle(name, seed, t_end):
    Sx, I = warm_state(name, seed, t_end)
    assert (I > 0).sum() > 20
    e = make_engine(name, seed)
    e._susceptible[...] = Sx
    e._infectious[...] = I
    _check_rates(e)


@pytest.mark.parametrize("name,seed,t_end", [("s9", 2020, 4.0), ("example", 1234, 70.0), ("t3small", 5, 60.0),
                                             ("table3_k10", 3, 60.0)])
def test_tree_rates_match_oracle_on_small_shapes(name, seed, t_end):
    Sx, I = warm_state(name, seed, t_end)
    e = make_engine(name, seed)
    e._susceptible[...] = Sx
    e._infectious[...] = I
    e._sync_params().set_direct_variant(1)
    _check_rates(e)


def _run_and_replay(name, R, N, seed=77):
    e = make_engine(name, seed, replicates=R)
    h = e._sync_params()
    h.simulate_direct(N, -1, -1.0, 200)
    assert h.synchronize() == 0
    c = h.get_counters()
    Sx_f, I_f = h.get_state()
    Sx1, I1 = first_infection(e._susceptible, e._infectious)
    for r in range(R):
        chain = h.get_event_log(r)
        assert chain.shape[1] == c["events"][r] <= N
        if chain.shape[1] < N:
            assert c["globalInfectious"][r] == 0 and chain.shape[1] > 100
        assert np.all(np.diff(chain[0]) >= 0)
        Sx, I = _replay_direct(e, chain, Sx1, I1)
        assert np.array_equal(Sx, Sx_f[r]) and np.array_equal(I, I_f[r])
        ty = chain[1].astype(int)
        for code, key in enumerate(["bCounter", "dCounter", "sCounter", "mCounter", "iCounter", "migPlus"]):
            assert (ty == code).sum() == c[key][r], key
        assert c["good_attempt"][r] >= 1 and c["time"][r] == chain[0, -1]
    return e, h, c, I_f


@pytest.mark.parametrize("name", LARGE)
def test_large_log_replays_to_final_state(name):
    e, h, c, I_f = _run_and_replay(name, 8, 4000)
    if e.hapNum >= 4096:  # the descents span the trees: dozens of haplotypes present per replicate
        distinct = [(I_f[r].sum(axis=0) > 0).sum() for r in range(I_f.shape[0])]
        assert np.median(distinct) >= 50, distinct


def _distribution(name, R=1200, N=2500, variant=0):
    e = make_engine(name, 5000, replicates=R)
    h = e._sync_params()
    h.set_direct_variant(variant)
    h.simulate_direct(N, N, -1.0, 200)
    c = h.get_counters()
    Sx_f, I_f = h.get_state()
    keys = ["bCounter", "dCounter", "sCounter", "mCounter", "iCounter", "migPlus", "migNonPlus", "time", "good_attempt",
            "inf_total", "events", "swapLockdown"]
    dev = {k: c[k] for k in keys if k in c}
    dev["inf_total"] = I_f.sum(axis=(1, 2))
    ora = oracle_direct(name, range(1000, 1000 + R), N)
    bad = _ks_all(dev, ora, [k for k in keys if k in dev and k in ora])
    assert not bad, bad
    return c


def test_large_distribution_matches_oracle():
    """(6, 2, 2) with migration, immunity and lockdowns that switch on and off."""
    c = _distribution("large_6_2_2_ld")
    assert c["swapLockdown"].mean() > 0.5 and c["migPlus"].sum() > 0


@pytest.mark.parametrize("name", ["s1", "s2", "s3", "s4", "s5", "s6", "s7", "s8", "s9"])
def test_tree_kernel_distribution_matches_oracle(name):
    _distribution(name, variant=1)


@pytest.mark.parametrize("name,N,variant", [("large_6_2_2_ld", 20000, 0), ("large_4_100_3", 20000, 0), ("s7", 20000, 1)])
def test_large_incremental_totals_equal_fresh_recompute(name, N, variant):
    """totalRate is the deme tree's root, totalMigrationRate kept by increments: after N events both equal a fresh
    recompute from the final state (the bounds of test_incremental_totals_equal_fresh_recompute)."""
    R = 16
    e = make_engine(name, 4242, replicates=R)
    h = e._sync_params()
    h.set_direct_variant(variant)
    h.simulate_direct(N, -1, -1.0, 200)
    s = h.summaries()
    c = h.get_counters()
    checked = 0
    for r in range(R):
        if c["globalInfectious"][r] == 0:
            continue
        fresh = h.rates(r)["totals"]
        assert abs(s[r, 22] - fresh[0]) <= 1e-11 * fresh[0], (r, s[r, 22], fresh[0])
        assert abs(s[r, 23] - fresh[1]) <= 1e-9 * max(fresh[0], fresh[1]), (r, s[r, 23], fresh[1])
        checked += 1
    assert checked >= R // 2


def _logs(name, R, N, seed=31):
    e = make_engine(name, seed, replicates=R)
    h = e._sync_params()
    h.simulate_direct(N, -1, -1.0, 200)
    return [h.get_event_log(r) for r in range(min(R, 16))], h.get_counters()


def test_large_logs_do_not_depend_on_batching():
    """Replicate r's log is a function of its seed alone: the same in a batch of 64, of 16, of 3,000 (more replicates
    than resident warps, so warp slices are reused) and across runs."""
    a, _ = _logs("large_7_1_2", 64, 1500)
    b, _ = _logs("large_7_1_2", 16, 1500)
    c, cnt = _logs("large_7_1_2", 3000, 1500)
    d, _ = _logs("large_7_1_2", 16, 1500)
    assert cnt["events"].min() > 100
    for r in range(16):
        assert np.array_equal(a[r], b[r]) and np.array_equal(b[r], c[r]) and np.array_equal(b[r], d[r]), r


@pytest.mark.parametrize("name", ["large_7_1_2", "large_4_100_3"])
def test_large_curves(name):
    R = 4
    e = make_engine(name, 9, replicates=R)
    Sx0, I0 = first_infection(e._susceptible, e._infectious)
    e.SimulatePopulation(3000, 10 ** 9, -1, 200)
    c = check_true_counts(e, R)
    K, H, S = e.popNum, e.hapNum, e.susNum
    cnt = e.counters()
    for r in (0, R - 1):
        chain = e.get_chain_events(r)
        I_end = c["infectious"][r, -1]
        for p, h in sorted({(0, 0), (K - 1, int(np.argmax(I_end.sum(axis=0)))), (K - 1, H - 1)}):
            want = O.ref_data_infectious(chain, None, I0[p, h], float(cnt["time"][r]), p, h, STEPS)
            Data, Sample, tp, ld = e.get_data_infectious(p, h, STEPS, replicate=r)
            np.testing.assert_array_equal(Data, want[0])
            np.testing.assert_array_equal(Sample, want[1])
        for p, s in sorted({(0, 0), (K - 1, S - 1)}):
            want = O.ref_data_susceptible(chain, None, Sx0[p, s], float(cnt["time"][r]), p, s, STEPS)
            Data, tp, ld = e.get_data_susceptible(p, s, STEPS, replicate=r)
            np.testing.assert_array_equal(Data, want[0])


def test_large_genealogy_bit_exact():
    """An oracle log at (7, 1, 2), loaded into the device and replayed with the oracle's uniform stream."""
    om = O.OracleModel.from_engine(make_engine("large_7_1_2", 2020))
    om.simulate(6000)
    chain = om.events()
    Sx_end, I_end = om.get_state()
    assert om.counters()["sCounter"] >= 2
    e = make_engine("large_7_1_2", 2020, replicates=2)
    h = e._sync_params()
    for r in range(2):
        h.set_event_log(r, chain, I_end)
    u = pcg(13).random(chain.shape[1] * 4 + 16)
    h.genealogy(uniform_stream=[u, u])
    om.genealogy(13)
    for r in range(2):
        assert_same_genealogy(h, r, om)


def test_simulator_end_to_end_at_nine_sites(tmp_path):
    sim = Simulator(number_of_sites=9, seed=12, replicates=2, verbose=False)
    sim.set_transmission_rate(3.0)
    sim.set_recovery_rate(1.0)
    sim.set_sampling_rate(0.3)
    sim.set_mutation_rate(0.05)
    sim.simulate(4000, method='direct')
    sim.genealogy(seed=5)
    tree, times = (np.asarray(x) for x in sim.get_tree())
    n = int(sim.counters()["sCounter"][0])
    assert n >= 2 and len(tree) == 2 * n - 1
    assert (tree < 0).sum() == 1
    child = np.nonzero(tree >= 0)[0]
    assert np.all(times[tree[child]] <= times[child])
    sim.export_newick(file_template="t", file_path=str(tmp_path))
    sim.export_mutations(file_template="t", file_path=str(tmp_path))
    assert any(p.stat().st_size > 0 for p in tmp_path.iterdir())
    data, sample, tp, ld = sim.get_data_infectious(0, 0, 20)
    want = O.ref_data_infectious(sim.get_chain_events(0), None, 1, float(sim.counters()["time"][0]), 0, 0, 20)
    np.testing.assert_array_equal(data, want[0])
    np.testing.assert_array_equal(sample, want[1])


def test_tau_refuses_large_shape_with_a_message():
    e = make_engine("large_7_1_2", 3, replicates=2)
    with pytest.raises(VgsimError, match=r"7 sites = 16384 haplotypes, 1 demes, 2 susceptibility groups.*shared memory"
                                         r".*direct method"):
        e.SimulatePopulation_tau(10, 10 ** 9, -1, 1)
    with pytest.raises(VgsimError, match="direct method"):
        e.propensities()
    e.SimulatePopulation(500, 10 ** 9, -1, 200)
    assert e.counters()["events"].min() > 0
