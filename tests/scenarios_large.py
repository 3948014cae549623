"""Model shapes whose direct-method rate hierarchy exceeds one SM's shared memory (the large-state direct kernel), for
tests/test_gpu_direct_large.py and scripts/bench_direct_large.py.  Same `(dims, setup)` form as tests/scenarios.py.

The oracle workers of tests/oracle_pool.py build engines from tests/scenarios.py by name; `oracle_direct` is the
equivalent worker for these shapes (spawned through the same pool, it imports only numpy, the oracle and the host-side
engine)."""
import os
import sys


def _large(U, K, S, lockdown=False):
    """The mutation rate is high enough that a few thousand events spread the infections over dozens of haplotypes;
    with S = 3, group 2 holds the recovered of 'G...' haplotypes and nobody is susceptible in it (an all-zero sigma
    row)."""
    def setup(e):
        e.set_transmission_rate(3.0, None)
        e.set_recovery_rate(1.0, None)
        e.set_sampling_rate(0.2, None)
        if U > 0:
            e.set_mutation_rate(0.1, None, None)
            e.set_mutation_probabilities([1, 1, 1, 2], None, None)
        if S > 1:
            e.set_susceptibility_type(1, None)
            e.set_susceptibility(0.3, None, 1)
            e.set_immunity_transition(0.05, 1, 0)
        if S > 2 and U > 0:
            e.set_susceptibility_type(2, 'G' + '*' * (U - 1))
            e.set_susceptibility(0.0, None, 2)
            e.set_immunity_transition(0.1, 2, 0)
        if K > 1:
            e.set_total_migration_probability(0.01)
            e.set_sampling_multiplier(2.0, K - 1)
        if lockdown:  # every deme locks down at 300 infectious and reopens below 100
            e.set_npi([0.3, 3e-4, 1e-4], None)
    return setup


LARGE_SCENARIOS = {"large_%d_%d_%d" % d: (d, _large(*d)) for d in
                   ((6, 2, 2), (7, 1, 2), (9, 1, 1), (4, 100, 3), (0, 4096, 1), (6, 1, 3), (7, 2, 2), (4, 10, 3))}
LARGE_SCENARIOS["large_6_2_2_ld"] = ((6, 2, 2), _large(6, 2, 2, lockdown=True))


def make_engine(name, seed=1, replicates=1):
    from vgsim_b200._engine import BirthDeathModel as Eng
    (U, K, S), setup = LARGE_SCENARIOS[name]
    e = Eng(U, K, S, seed, False, False, int(1e6), 0.0, replicates=replicates)
    setup(e)
    return e


def oracle_direct(task):
    """Pool worker: (name, seeds, iterations) -> the oracle's counters and total infectious of each run, as lists."""
    here = os.path.dirname(os.path.abspath(__file__))
    for p in (os.path.dirname(here), here):
        if p not in sys.path:
            sys.path.insert(0, p)
    from oracle import oracle as O
    name, seeds, iterations = task
    out = {}
    for seed in seeds:
        om = O.OracleModel.from_engine(make_engine(name, int(seed)))
        om.simulate(iterations, sample_size=iterations)
        for k, v in om.counters().items():
            out.setdefault(k, []).append(v)
        out.setdefault("inf_total", []).append(int(om.get_state()[1].sum()))
    return out
