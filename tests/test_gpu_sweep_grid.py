"""Sweep.grid on the device (vgsim_upload_param_grid): every point's blob is the bits vgsim_upload_params writes for the
same point, and a grid sweep runs exactly like the callable sweep over the same point list."""
import numpy as np
import pytest

from scenarios import SCENARIOS
from scenarios_large import LARGE_SCENARIOS
from vgsim_b200 import _capi
from vgsim_b200._engine import BirthDeathModel as Eng
from vgsim_b200.sweep import Sweep

pytestmark = pytest.mark.gpu


def callables(axes):
    """The callable Sweep's point list for `axes`: itertools.product order, every axis's setter in axis order."""
    import itertools

    def mk(vals):
        def f(e):
            for (setter, _), v in zip(axes, vals):
                setter(e, v)
        return f
    return [mk(vals) for vals in itertools.product(*[v for _, v in axes])]


def same_blobs(g, c):
    for pp in range(g.hi - g.lo):
        a, b = g.h.get_params(pp), c.h.get_params(pp)
        assert np.array_equal(a.view(np.int64), b.view(np.int64)), pp


CONFIG4 = [(lambda e, v: e.set_transmission_rate(v, None), list(np.linspace(1.2, 4.0, 32) * 0.1)),
           (lambda e, v: e.set_total_migration_probability(v), list(np.logspace(-4, -1, 32)))]
WORLD = [(lambda e, v: e.set_sampling_multiplier(v, None), [0.5, 1.0, 3.0]),
         (lambda e, v: e.set_npi(list(v), None), [(0.1, 0.01, 0.002), (0.3, 0.02, 0.001)]),
         (lambda e, v: e.set_immunity_transition(v, 1, 0), [1 / 90, 1 / 30, 1 / 365])]
LARGE = [(lambda e, v: e.set_mutation_rate(v, None, None), [0.01, 0.05, 0.1, 0.2]),
         (lambda e, v: e.set_susceptibility(v, None, 1), [0.1, 0.3, 0.6, 0.9])]


@pytest.mark.parametrize("dims,setup,axes", [
    (*SCENARIOS["table3_k10"], CONFIG4),
    (*SCENARIOS["w"], WORLD),
    (*LARGE_SCENARIOS["large_6_2_2"], LARGE),
], ids=["table3_k10", "w", "large_6_2_2"])
def test_blobs_match_the_host_upload(dims, setup, axes):
    g = Sweep.grid(dims, setup, axes)
    c = Sweep(dims, setup, callables(axes))
    same_blobs(g, c)
    _, _, cd_g, _ = g.h.get_state(full=True)
    _, _, cd_c, _ = c.h.get_state(full=True)
    assert np.array_equal(cd_g, cd_c)


def test_simulation_is_the_callable_sweeps():
    dims, setup = SCENARIOS["t3small"]
    axes = [(lambda e, v: e.set_transmission_rate(v, None), [0.15, 0.3, 0.45]),
            (lambda e, v: e.set_contact_density(v, None), [0.7, 1.3]),
            (lambda e, v: e.set_total_migration_probability(v), [1e-3, 3e-2])]
    out = []
    for sw in (Sweep.grid(dims, setup, axes, replicates_per_point=2, seed=21),
               Sweep(dims, setup, callables(axes), replicates_per_point=2, seed=21)):
        sw.simulate(1500, 10 ** 9, -1, "direct")
        r = {"direct": sw.h.get_state(full=True), "counters_direct": sw.counters()}
        sw.simulate(12, 10 ** 9, -1, "tau")
        r["tau"] = sw.h.get_state(full=True)
        r["log"] = [sw.h.get_tau_log(i) for i in range(sw.R)]
        sw.genealogy(seed=np.arange(sw.R, dtype=np.uint64) + np.uint64(500))
        r["counters"] = sw.counters()
        r["summaries"] = sw.summaries()
        out.append(r)
    g, c = out
    for k in ("direct", "tau"):
        assert all(np.array_equal(a, b) for a, b in zip(g[k], c[k]))
    for k in ("counters_direct", "counters"):
        assert all(np.array_equal(g[k][n], c[k][n]) for n in c[k])
    assert all(np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) for a, b in zip(g["log"], c["log"]))
    assert np.array_equal(g["summaries"], c["summaries"])
    assert (g["summaries"][:, :, 10] == 12).any() and (g["summaries"][:, :, 13] > 1).any()


def test_sharding_does_not_change_results():
    dims, setup = SCENARIOS["t3small"]
    axes = [(lambda e, v: e.set_transmission_rate(v, None), list(np.linspace(1.2, 4.0, 5) * 0.1)),
            (lambda e, v: e.set_total_migration_probability(v), list(np.logspace(-4, -1, 4)))]

    def run(rank, world):
        sw = Sweep.grid(dims, setup, axes, replicates_per_point=2, seed=5, rank=rank, world=world)
        sw.simulate(1500, 10 ** 9, -1, "direct")
        sw.simulate(12, 10 ** 9, -1, "tau")
        sw.genealogy(seed=np.arange(sw.lo * 2, sw.hi * 2, dtype=np.uint64) + np.uint64(900))
        return sw.summaries()

    whole = run(0, 1)
    np.testing.assert_array_equal(whole, np.concatenate([run(g, 3) for g in range(3)], axis=0))
    assert whole.shape[:2] == (20, 2)


def test_an_inadmissible_point_fails_the_call():
    dims, setup = SCENARIOS["t3small"]
    # each value is admissible on its own; together the last corner sends more than everyone out of deme 0
    axes = [(lambda e, v: e.set_migration_probability(v, 0, 1), [0.1, 0.6]),
            (lambda e, v: e.set_migration_probability(v, 0, 2), [0.1, 0.6])]
    with pytest.raises(_capi.VgsimError, match=r"parameter grid point 3: .*sum to more than 1"):
        Sweep.grid(dims, setup, axes)
    # straight through the C ABI: the failed call leaves the blob of a point uploaded before untouched
    U, K, S = dims
    e = Eng(U, K, S, 1, False, False, int(1e6), 0.0)
    setup(e)
    h = _capi.Handle(U, K, S, 4, 4, None)
    h.upload_params(0, e.param_arrays())
    before = h.get_params(0)
    mo = sum(e.param_arrays()[k].size for k in _capi.SOURCE_FIELDS[:_capi.SOURCE_FIELDS.index("m")])
    with pytest.raises(_capi.VgsimError, match=r"parameter grid point 1: .*more than 1e-15"):
        # value 1 sends everyone out of deme 0 (0.5 + 0.25 + 0.25 = 1 exactly): nobody stays
        h.upload_param_grid(0, [2], np.array([0, 1, 4]), np.array([mo + 1, mo + 1, mo + 2, mo + 3]),
                            np.array([0.2, 0.5, 0.25, 0.25]), 0, 0, 2)
    assert np.array_equal(h.get_params(0).view(np.int64), before.view(np.int64))


def test_multievents_of_a_susceptibility_type_axis():
    dims, setup = SCENARIOS["t3small"]
    axes = [(lambda e, v: e.set_susceptibility_type(v, 'A*'), [0, 1, 2]),
            (lambda e, v: e.set_transmission_rate(v, None), [0.3, 0.5])]
    out = []
    for sw in (Sweep.grid(dims, setup, axes, seed=8), Sweep(dims, setup, callables(axes), seed=8)):
        sw.simulate(2000, 10 ** 9, -1, "direct")
        sw.simulate(6, 10 ** 9, -1, "tau")
        out.append([sw.h.get_multievents(r) for r in range(sw.R)])
    for a, b in zip(*out):
        assert all(np.array_equal(a[k], b[k]) for k in b)
    # the death records of haplotype 'AA' carry its susceptibility type, the grid's axis 0
    death = [m["nhap"][(m["type"] == 1) & (m["hap"] == 0)] for m in out[0]]
    assert all((d == r // 2).all() for r, d in enumerate(death)) and sum(d.size for d in death) > 0
