"""Error paths of the C ABI on a device: replicate indices outside [0, R) are rejected by every entry point that takes
one (the count functions return -1), the Python getters raise instead of returning empty arrays, and a rejected
genealogy call frees what it allocated."""
import ctypes

import numpy as np
import pytest

from vgsim_b200 import _capi
from test_gpu_tau import make_engine

pytestmark = pytest.mark.gpu

lib = _capi.lib
N = None  # NULL pointer argument

# every entry point that takes a replicate index, called with NULL outputs and zero lengths
INDEXED = {
    "vgsim_propensities": lambda h, r: lib.vgsim_propensities(h, r, N, N, N, N),
    "vgsim_rates": lambda h, r: lib.vgsim_rates(h, r, N, N, N, N, N, N, N, N),
    "vgsim_get_event_log": lambda h, r: lib.vgsim_get_event_log(h, r, N, 0),
    "vgsim_get_multievents": lambda h, r: lib.vgsim_get_multievents(h, r, 0, N, N, N, N, N, N, N),
    "vgsim_get_tau_log": lambda h, r: lib.vgsim_get_tau_log(h, r, 0, N, N),
    "vgsim_set_event_log": lambda h, r: lib.vgsim_set_event_log(h, r, N, 0, N),
    "vgsim_get_lockdowns": lambda h, r: lib.vgsim_get_lockdowns(h, r, N, N, N),
    "vgsim_get_tree": lambda h, r: lib.vgsim_get_tree(h, r, N, N, N),
    "vgsim_get_mutations": lambda h, r: lib.vgsim_get_mutations(h, r, N, N, N, N, N),
    "vgsim_get_migrations": lambda h, r: lib.vgsim_get_migrations(h, r, N, N, N, N),
}
COUNTS = ("vgsim_num_lockdowns", "vgsim_tree_size", "vgsim_num_mutations", "vgsim_num_migrations")


@pytest.fixture(scope="module")
def handle():
    e = make_engine("s9", 42, replicates=8)
    e.SimulatePopulation(20000, 20000, -1, 200)
    e.GetGenealogy(None)
    h = e._handle
    assert any(lib.vgsim_tree_size(h._h, r) > 0 for r in range(h.R))
    return h


@pytest.mark.parametrize("where", ["negative", "R"])
def test_c_entry_points_reject_replicate_out_of_range(handle, where):
    r = -1 if where == "negative" else handle.R

    def other_error():  # a different message first, so that each check sees the message of its own call
        assert lib.vgsim_set_tau_variant(handle._h, -1) != 0

    for name, call in INDEXED.items():
        other_error()
        assert call(handle._h, r) != 0, name
        assert lib.vgsim_last_error().decode() == "replicate out of range", name
    for name in COUNTS:
        other_error()
        assert getattr(lib, name)(handle._h, r) == -1, name
        assert lib.vgsim_last_error().decode() == "replicate out of range", name
    for name in COUNTS:  # in range they count
        assert getattr(lib, name)(handle._h, 0) >= 0, name


@pytest.mark.parametrize("getter", ["get_tree", "get_mutations", "get_migrations", "get_lockdowns"])
def test_python_getters_raise_on_replicate_out_of_range(handle, getter):
    for r in (-1, handle.R):
        with pytest.raises(_capi.VgsimError, match="replicate out of range"):
            getattr(handle, getter)(r)


def test_rejected_genealogy_frees_its_scratch():
    """uniform_stream without stream_offsets is rejected; 20 such calls at 4,096 T3 replicates leave free memory as the
    first one left it (each call used to keep a R*K*H*8-byte copy of the infectious counts, 21 MB here)."""
    import torch
    e = make_engine("t3", 11, replicates=4096)
    e.SimulatePopulation(200, 10**9, -1, 1)
    h = e._handle
    u = np.zeros(4096, np.float64)
    free = []
    for _ in range(20):
        rc = lib.vgsim_genealogy(h._h, N, u.ctypes.data_as(ctypes.c_void_p), N, 0)
        assert rc != 0
        assert "stream_offsets" in lib.vgsim_last_error().decode()
        torch.cuda.synchronize()
        free.append(torch.cuda.mem_get_info()[0])
    assert free[-1] == free[0], [(f - free[0]) / 2**20 for f in free]
