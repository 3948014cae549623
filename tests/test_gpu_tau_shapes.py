"""The warp tau kernel has instances with the model shape compiled in ((3, 10, 3) = T3 and (2, 10, 3) = table3_k10):
they must leave exactly what the runtime-shape instance (vgsim_set_tau_variant bit 6) leaves, and the launch tap must
say which instance ran."""
import numpy as np
import pytest

from oracle import oracle as O
from scenarios import SCENARIOS
from vgsim_b200 import _capi
from vgsim_b200._engine import BirthDeathModel as Eng

pytestmark = pytest.mark.gpu

RUNTIME_SHAPE = 64  # variant bit 6


def warm_state(name, seed, t_end):
    (U, K, S), setup = SCENARIOS[name]
    e = Eng(U, K, S, seed, False, False, int(1e6), 0.0)
    setup(e)
    om = O.OracleModel.from_engine(e)
    om.simulate(10**7, sample_size=10**9, epidemic_time=t_end)
    return om.get_state()


def run(name, Sx0, I0, R, leaps, variant, seed0):
    """R replicates from one state, `leaps` leaps each; returns counters, final state, the dense logs of every 61st
    replicate and the fixed-shape tap."""
    (U, K, S), setup = SCENARIOS[name]
    e = Eng(U, K, S, seed0, False, False, int(1e6), 0.0)
    setup(e)
    h = _capi.Handle(U, K, S, R, 1, None)
    try:
        h.set_seeds((np.uint64(seed0) + np.arange(R, dtype=np.uint64)).astype(np.uint64))
        h.upload_params(0, e.param_arrays())
        h.set_state(np.ascontiguousarray(np.broadcast_to(Sx0, (R,) + Sx0.shape)),
                    np.ascontiguousarray(np.broadcast_to(I0, (R,) + I0.shape)))
        h.set_tau_variant(variant)
        h.simulate_tau(leaps, -1, -1.0, 1)
        c = h.get_counters()
        Sx, I = h.get_state()
        logs = [h.get_tau_log(r) for r in range(0, R, 61)]
        return c, Sx, I, logs, h.tau_fixed_shape()
    finally:
        h.close()


def assert_same(a, b):
    ca, cb = a[0], b[0]
    assert set(ca) == set(cb)
    for k in ca:
        assert np.array_equal(ca[k], cb[k]), (k, np.flatnonzero(ca[k] != cb[k])[:10])
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    for (cnt_a, tt_a), (cnt_b, tt_b) in zip(a[3], b[3]):
        assert np.array_equal(cnt_a, cnt_b) and np.array_equal(tt_a, tt_b)


# t3: 4,096 replicates are two visits of the 148 x 14 warps in flight, as in the benchmark's window
@pytest.mark.parametrize("name,seed,t0,R,shape", [("t3", 11, 60.0, 4096, (3, 10, 3)), ("table3_k10", 3, 60.0, 600, (2, 10, 3))])
def test_fixed_shape_kernel_matches_runtime_shape(name, seed, t0, R, shape):
    Sx0, I0 = warm_state(name, seed, t0)
    assert I0.sum() > 0
    fixed = run(name, Sx0, I0, R, 32, 0, 900)
    runtime = run(name, Sx0, I0, R, 32, RUNTIME_SHAPE, 900)
    assert fixed[4] == shape and runtime[4] is None
    assert fixed[0]["leaps"].min() >= 1
    assert_same(fixed, runtime)


def test_other_shapes_run_the_runtime_shape_kernel():
    Sx0, I0 = warm_state("s9", 2020, 4.0)
    assert I0.sum() > 0
    a = run("s9", Sx0, I0, 600, 32, 0, 910)
    b = run("s9", Sx0, I0, 600, 32, RUNTIME_SHAPE, 910)
    assert a[4] is None and b[4] is None
    assert_same(a, b)
