#!/usr/bin/env python
"""Set-up time of a parameter sweep through both constructors: `Sweep(points=...)` (one host-derived upload and one
stream synchronisation per point) and `Sweep.grid` (axes resolved on the host, points built on the device).

Workloads:
  - configs[4]: one rank's share of the 256 x 256 R0 x total-migration grid on the table-3 model with K = 10 (world 8:
    8,192 points, one replicate each), exactly what scripts/run_sweep.py sets up;
  - world: a 64 x 64 grid of the same axes on the K = 100 world model (4,096 points on one rank).
Each timing is a host clock around the constructor that ends in a device synchronise; the two paths alternate, `runs`
times each.  Prints one JSON record with the median and range of each, the card's name and power limit read in the
same run, and whether the two paths left bit-identical blobs.

    python scripts/bench_sweep_setup.py [runs]
"""
import gc
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from scenarios import SCENARIOS  # noqa: E402
from vgsim_b200 import _shard  # noqa: E402
from vgsim_b200.sweep import Sweep  # noqa: E402

runs = int(sys.argv[1]) if len(sys.argv) > 1 else 3
if not torch.cuda.is_available():
    sys.exit("bench_sweep_setup.py needs a CUDA device")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip().split(", ")
    return {"gpu": q[0], "power_limit": q[1] if len(q) > 1 else None}


def axes(n0, n1):
    B = np.linspace(1.2, 4.0, n0) * (0.099 + 0.001)
    MIG = np.logspace(-4, -1, n1)
    return [(lambda e, v: e.set_transmission_rate(float(v), None), list(B)),
            (lambda e, v: e.set_total_migration_probability(float(v)), list(MIG))]


def points(ax):
    def mk(b, m):
        def f(e):
            ax[0][0](e, b)
            ax[1][0](e, m)
        return f
    return [mk(b, m) for b in ax[0][1] for m in ax[1][1]]


def timed(make):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sw = make()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, sw


def measure(name, n0, n1, world):
    dims, setup = SCENARIOS[name]
    ax = axes(n0, n1)
    pts = points(ax)
    t = {"callable": [], "grid": []}
    makers = {"callable": lambda: Sweep(dims, setup, pts, 1, seed=31337, rank=0, world=world, device=0),
              "grid": lambda: Sweep.grid(dims, setup, ax, 1, seed=31337, rank=0, world=world, device=0)}
    same = None
    timed(makers["grid"])  # warm-up: module load, first allocations
    for _ in range(runs):
        kept = {}
        for path in ("callable", "grid"):
            s, sw = timed(makers[path])
            t[path].append(s)
            kept[path] = sw
        if same is None:
            a, b = kept["callable"], kept["grid"]
            same = all(np.array_equal(a.h.get_params(pp).view(np.int64), b.h.get_params(pp).view(np.int64))
                       for pp in range(a.hi - a.lo))
        for sw in kept.values():
            sw.h.close()
        del kept
        gc.collect()
    lo, hi = _shard.replicate_range(0, world, len(pts))
    return {"model": name, "dims": list(dims), "grid": [n0, n1], "world": world, "points_on_rank": hi - lo,
            "blobs_identical": bool(same),
            **{path: {"median_s": float(np.median(v)), "min_s": float(min(v)), "max_s": float(max(v)), "runs": v}
               for path, v in t.items()}}


rec = card()
rec["configs4_rank0_of_8"] = measure("table3_k10", 256, 256, 8)
rec["world_k100"] = measure("w", 64, 64, 1)
print(json.dumps(rec))
