"""Host side of the trajectories / lineages-through-time rows (no GPU): the time-grid rules, and the all-gather of
[n, T, X] int64 rows over ranks with gloo (the rows a sweep gathers besides its summaries)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from vgsim_b200 import _shard
from vgsim_b200._capi import time_grid


def test_valid_grid_is_float64_and_contiguous():
    t = time_grid([0, 1.5, 2, 1e9])
    assert t.dtype == np.float64 and t.flags.c_contiguous and t.tolist() == [0.0, 1.5, 2.0, 1e9]
    assert time_grid(np.arange(10.0)[::2]).flags.c_contiguous
    assert time_grid([-3.0]).tolist() == [-3.0]


@pytest.mark.parametrize("bad,msg", [([], "at least one point"), ([1.0, 1.0], "strictly increasing"),
                                     ([0.0, 2.0, 1.0], "strictly increasing"), ([0.0, np.nan, 2.0], "not finite"),
                                     ([0.0, np.inf], "not finite"), ([-np.inf, 0.0], "not finite"),
                                     ([[0.0, 1.0]], "one-dimensional")])
def test_invalid_grids_are_refused(bad, msg):
    with pytest.raises(ValueError, match=msg):
        time_grid(bad)


T, X = 7, 5


def _rows(ids):
    # row of global replicate g: a function of g only, -1 where "not simulated", as trajectories rows are
    ids = np.asarray(list(ids), np.int64)
    a = ids[:, None, None] * 1000 + np.arange(T)[None, :, None] * 10 + np.arange(X)[None, None, :]
    a[:, T - 1 - (ids % 3)] = -1
    return a


def _worker(rank, world, port, total, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        lo, hi = _shard.replicate_range(rank, world, total)
        out = _shard.gather_summaries(torch.from_numpy(_rows(range(lo, hi))), world)
        q.put((rank, out.dtype == torch.int64, out.numpy()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("total", [10, 11])
def test_gather_trajectory_rows_world2_gloo(total):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    world = 2
    procs = [ctx.Process(target=_worker, args=(r, world, port, total, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = {r: (is64, a) for r, is64, a in (q.get(timeout=120) for _ in range(world))}
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    want = _rows(range(total))
    for r in range(world):
        assert got[r][0] and np.array_equal(got[r][1], want)
