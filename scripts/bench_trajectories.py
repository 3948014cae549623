#!/usr/bin/env python
"""Trajectories (vgsim_trajectories) against the epidemic curves (vgsim_epidemic_curves) on the same event logs, and
lineages through time (vgsim_lineages_through_time) after a sweep rank's genealogy.

1. T3 shape (3 sites x 10 demes x 3 groups), 4,096 replicates: the direct method to the first window, tau leaps in
   recycled blocks to each later window, as bench.py takes them there.  From each window's state one batch of `leaps`
   dense tau leaps is the log both passes read.  The two kernels alternate on that log: trajectories on one grid of
   T = 101 points over [0, max currentTime], curves with infectious + sampled and step_num = 100 (101 points per
   replicate).  Each reads the log once (16 B per row, 4 Pp B per dense leap row; 14 GB at 32 leaps, far above the
   126 MB of L2): log bytes over kernel time, against the 7.7 TB/s of the B200's HBM3e.
2. The configs[4] rank of scripts/run_sweep.py: 8,192 points of the table-3 K = 10 model, direct 20,000 events, 64 tau
   leaps, genealogy; then lineages through time on T = 101 points, checked against the definition on a few trees.

Kernel times are the handle's CUDA event pair (vgsim_last_kernel_ms).  Prints one JSON record, with the card's name and
power limit read in the same run.

    python scripts/bench_trajectories.py [--replicates 4096] [--leaps 32] [--windows 60,120] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from scenarios import SCENARIOS  # noqa: E402
from vgsim_b200._engine import BirthDeathModel as Eng  # noqa: E402
from vgsim_b200.sweep import Sweep  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        name, power, clock = [x.strip() for x in q.stdout.strip().split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as ex:  # the name alone, from the runtime
        return {"name": torch.cuda.get_device_name(), "power_limit": "unknown (%s)" % ex}


def t3_windows(args):
    (U, K, S), setup = SCENARIOS["t3"]
    R, L = args.replicates, args.leaps
    e = Eng(U, K, S, 2024, False, False, int(1e6), 0.0, replicates=R, device=0)
    setup(e)
    h = e._sync_params()
    Pp = (h.P + 7) & ~7
    windows = [float(x) for x in args.windows.split(",")]
    h.simulate_direct(250000, -1, windows[0], 200)
    out = []
    for wt in windows:
        for _ in range(400):   # tau in recycled blocks up to the window (no-op for the direct method's window)
            c = h.get_counters()
            if bool(np.all((c["time"] >= np.float32(wt)) | (c["globalInfectious"] == 0))):
                break
            h.recycle_log()
            h.simulate_tau(L, -1, wt, 1)
        Sx, I = h.get_state()
        # the log both passes read: `leaps` dense leaps from the window's state
        h.reset()
        h.set_seeds(np.arange(R, dtype=np.uint64) + np.uint64(int(wt) * 7919))
        h.set_state(Sx, I)
        h.simulate_tau(L, -1, -1.0, 1)
        c = h.get_counters()
        ct = c["time"]
        log_bytes = float(c["events"].sum()) * 16 + float(c["leaps"].sum()) * 4 * Pp
        grid = np.linspace(0.0, float(ct.max()), 101)
        rec = {"window_t": wt, "replicates": R, "leaps_per_replicate": L, "log_bytes": log_bytes,
               "max_current_time": float(ct.max()), "trajectories_ms": [], "curves_ms": []}
        for _ in range(args.reps):   # alternate, the first pair warms both kernels up
            h.trajectories_dev_ptr(grid)
            rec["trajectories_ms"].append(h.last_kernel_ms())
            h.epidemic_curves(100, want=("infectious", "sampled"))
            rec["curves_ms"].append(h.last_kernel_ms())
        # check: at the last grid point (= the largest currentTime) the rows hold the final state
        tr = h.trajectories(grid)
        _, I_end = h.get_state()
        last = ct == ct.max()
        assert np.array_equal(tr["infectious_deme"][last, -1], I_end[last].sum(axis=2))
        assert np.array_equal(tr["infectious_hap"][last, -1], I_end[last].sum(axis=1))
        for k in ("trajectories", "curves"):
            t = sorted(rec.pop(k + "_ms")[1:])
            rec[k] = {"kernel_ms_median": t[len(t) // 2], "kernel_ms_min": t[0], "kernel_ms_max": t[-1],
                      "log_GBps": log_bytes / (t[len(t) // 2] * 1e-3) / 1e9,
                      "share_of_hbm_peak": log_bytes / (t[len(t) // 2] * 1e-3) / HBM_BYTES_PER_S}
        rec["trajectories"]["bytes_written"] = R * 101 * 2 * (K + 4 ** U) * 8
        rec["curves"]["bytes_written"] = R * 101 * 2 * K * 4 ** U * 8
        out.append(rec)
    return out


def ltt_sweep_rank(args):
    dims, setup = SCENARIOS["table3_k10"]
    B = np.linspace(1.2, 4.0, 256)[:32] * 0.1       # rows 0..31 of scripts/run_sweep.py's R0 grid: rank 0 of 8
    MIG = np.logspace(-4, -1, 256)
    sw = Sweep.grid(dims, setup, [(lambda e, v: e.set_transmission_rate(float(v), None), B),
                                  (lambda e, v: e.set_total_migration_probability(float(v)), MIG)], 1, seed=31337,
                    device=0)
    sw.simulate(20000, 10 ** 9, -1, "direct")
    sw.simulate(64, 10 ** 9, -1, "tau")
    sw.genealogy()
    s = sw.h.summaries()
    grid = np.linspace(0.0, float(s[:, 12].max()), 101)
    ms = []
    for _ in range(args.reps):
        sw.h.lineages_through_time_dev_ptr(grid)
        ms.append(sw.h.last_kernel_ms())
    got = sw.h.lineages_through_time(grid)
    checked = 0
    for r in np.flatnonzero(s[:, 13] > 0)[:: max(1, int((s[:, 13] > 0).sum()) // 8)]:
        parent, _, t = sw.h.get_tree(int(r))
        tp = np.where(parent >= 0, t[np.maximum(parent, 0)], -np.inf)
        assert np.array_equal(got[r], [np.count_nonzero((t >= g) & (tp < g)) for g in grid]), r
        checked += 1
    assert not got[s[:, 13] == 0].any()
    nodes = float(s[:, 13].sum())
    t = sorted(ms[1:])
    return {"replicates": sw.R, "tree_nodes_total": nodes, "largest_tree": float(s[:, 13].max()), "grid_points": 101,
            "kernel_ms_median": t[len(t) // 2], "kernel_ms_min": t[0], "nodes_per_s": nodes / (t[len(t) // 2] * 1e-3),
            "trees_checked_against_definition": checked}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--replicates", type=int, default=4096)
    ap.add_argument("--leaps", type=int, default=32)
    ap.add_argument("--windows", default="60,120")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    torch.cuda.init()
    rec = {"card": card(), "t3": t3_windows(args), "ltt_configs4_rank": ltt_sweep_rank(args)}
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
