"""Times the large-state direct kernel (csrc/direct_large_kernel.cu) on shapes whose rate hierarchy does not fit one
SM's shared memory, and prints one JSON line per shape.

Per shape: a warm-up call, then --runs timed calls, each on a fresh engine with the same seeds, each
`vgsim_simulate_direct(iterations)` from the first infection; kernel ms from vgsim_last_kernel_ms (CUDA events around
the launch), events from the counters.  The card name and power limit are read in the same run.  On (4, 10, 3), a shape
the shared-memory kernel holds, the two kernels are timed alternately (vgsim_set_direct_variant bit 0) for the record:
the selection never moves a fitting shape.  --oracle also times the CPU oracle (the reference's algorithm, one core) at
the same shapes for context.

    python scripts/bench_direct_large.py [--replicates 4096] [--iterations 2000] [--runs 3] [--oracle]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

from scenarios_large import LARGE_SCENARIOS, make_engine  # noqa: E402

SHAPES = ["large_6_1_3", "large_7_2_2", "large_9_1_1", "large_4_100_3"]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = (x.strip() for x in out.split(","))
        return name, power
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        return None, None


def time_calls(name, R, iterations, variant, runs):
    """runs timed calls, each on a fresh engine (same seeds) after one untimed call that loads the module"""
    ms, ev = [], []
    for i in range(runs + 1):
        e = make_engine(name, 1, R)
        h = e._sync_params()
        h.set_direct_variant(variant)
        h.simulate_direct(iterations, -1, -1.0, 200)
        if i:
            ms.append(h.last_kernel_ms())
            ev.append(int(h.get_counters()["events"].sum()))
        h.close()
    return ms, ev


def replicates_that_fit(name, want):
    """R such that the per-replicate state (I, its Restart copy, eff and the event log) takes at most a third of the card."""
    import torch
    (U, K, S), _ = LARGE_SCENARIOS[name]
    free, _ = torch.cuda.mem_get_info()
    per = 8 * (2 * K * 4 ** U + K * K) + 16 * 4096
    return int(max(1, min(want, free // 3 // per)))


def oracle_rate(name, iterations, seeds=3):
    from oracle import oracle as O
    n, t0 = 0, time.perf_counter()
    for s in range(seeds):
        om = O.OracleModel.from_engine(make_engine(name, 100 + s))
        om.simulate(iterations)
        n += int(om.counters()["events"])
    return n / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--replicates", type=int, default=4096)
    ap.add_argument("--iterations", type=int, default=2000)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--oracle", action="store_true")
    a = ap.parse_args()
    name_gpu, power = card()
    for name in SHAPES + ["large_4_10_3"]:
        R = replicates_that_fit(name, a.replicates)
        rec = {"shape": LARGE_SCENARIOS[name][0], "scenario": name, "replicates": R, "iterations": a.iterations,
               "gpu": name_gpu, "power_limit": power}
        if name == "large_4_10_3":  # a shape the shared-memory kernel holds: both kernels, alternating
            res = {0: ([], []), 1: ([], [])}
            for _ in range(a.runs):
                for v in (0, 1):
                    ms, ev = time_calls(name, R, a.iterations, v, 1)
                    res[v][0].extend(ms)
                    res[v][1].extend(ev)
            for v, key in ((0, "shared_kernel"), (1, "large_kernel")):
                ms, ev = res[v]
                rec[key] = {"kernel_ms_median": float(np.median(ms)), "kernel_ms_min": min(ms), "kernel_ms_max": max(ms),
                            "events": int(np.median(ev)), "events_per_s": float(np.median(ev) / (np.median(ms) / 1e3))}
        else:
            ms, ev = time_calls(name, R, a.iterations, 0, a.runs)
            rec.update({"kernel_ms_median": float(np.median(ms)), "kernel_ms_min": min(ms), "kernel_ms_max": max(ms),
                        "events": int(np.median(ev)), "events_per_s": float(np.median(ev) / (np.median(ms) / 1e3))})
        if a.oracle:
            rec["oracle_events_per_s_one_core"] = oracle_rate(name, a.iterations)
        print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
