#!/usr/bin/env python
"""Device resampling (vgsim_resample) at the two extremes of its work: many small runs and a few large ones.

1. T3 shape (3 sites x 10 demes x 3 groups), 4,096 replicates: the direct method to t = 60, then one call of 32 dense
   tau leaps (the 32 dense rows of a replicate are 3.4 MB, 13.8 GB over the batch).  A systematic map over fixed-seed
   random weights decides which replicates are overwritten.  Re-applying the same map copies the same bytes, so the
   kernel is timed with CUDA events over `--reps` launches of it.  For scale, in the same run: the same segment sizes
   copied with one cudaMemcpyAsync per (replicate, array), issued from the host between two buffers laid out like the
   moved runs, and the 32-leap tau step that built the batch.
2. The world shape (K = 100 demes, 1.97 MB per dense leap): 32 replicates, the direct method to t = 40, then 101 dense
   tau leaps (about 200 MB per replicate): few destinations, so the copy has to be split into chunks to fill the GPU.

Algorithmic bytes: one read and one write of every used byte of every copied run, over kernel time, against the
7.7 TB/s of the B200's HBM3e.  Prints one JSON record, with the card's name and power limit read in the same run.

    python scripts/bench_resample.py [--replicates 4096] [--leaps 32] [--reps 10] [--world-replicates 32]
"""
import argparse
import ctypes
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
from vgsim_b200.resample import systematic_map  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        name, power, clock = [x.strip() for x in q.stdout.strip().split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as ex:  # the name alone, from the runtime
        return {"name": torch.cuda.get_device_name(), "power_limit": "unknown (%s)" % ex}


def segments(h, src):
    """Used bytes of every (destination, array) copy the map asks for, in the order of csrc/resample_kernel.cu (after
    plain tau calls: no archived leaps, so every leap still has its dense row)."""
    K, H, S = h.K, h.H, h.S
    Pp = (h.P + 7) & ~7
    c = h.get_counters()
    fixed = [K * H * 8, K * S * 8, K * H * 8, K * S * 8, K * 8, K * 4, K * K * 8, K * 8, K * 8,
             8, 16, 96, 4, 4, 8, 8, 4, 4]
    out = []
    for r in np.flatnonzero(src != np.arange(len(src))):
        s = int(src[r])
        ev, lp = int(c["events"][s]), int(c["leaps"][s])
        nloc = len(h.get_lockdowns(s)[0])
        out += fixed + [ev * 8, ev * 8, lp * 16, lp * Pp * 4, 4, 0, nloc * 4, nloc * 8]
    return [n for n in out if n > 0]


def time_resample(h, src, reps):
    h.resample(src)  # warm-up: module load, the map buffer
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        h.resample(src)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def _cudart():
    for name in ("libcudart.so.12", "libcudart.so"):  # torch has loaded the runtime it was built with
        try:
            return ctypes.CDLL(name)
        except OSError:
            pass
    return ctypes.CDLL("/usr/local/cuda/lib64/libcudart.so")


def time_memcpy_per_segment(sizes, reps):
    """One cudaMemcpyAsync per segment between two device buffers holding the segments back to back (16-byte aligned
    starts), issued from the host on the default stream; CUDA events around the whole pass."""
    rt = _cudart()
    rt.cudaMemcpyAsync.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p]
    rt.cudaMemcpyAsync.restype = ctypes.c_int
    sz = np.asarray(sizes, np.int64)
    off = np.concatenate([[0], np.cumsum((sz + 15) // 16 * 16)])
    src = torch.empty(int(off[-1]), dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    ps, pd = src.data_ptr(), dst.data_ptr()
    calls = [(pd + int(o), ps + int(o), int(n)) for o, n in zip(off[:-1], sz)]
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def one_pass():
        for d, s, n in calls:
            if rt.cudaMemcpyAsync(d, s, n, 3, stream) != 0:
                raise RuntimeError("cudaMemcpyAsync failed")
    one_pass()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        one_pass()
    b.record()
    b.synchronize()
    ms = a.elapsed_time(b) / reps
    del src, dst
    torch.cuda.empty_cache()
    return ms, len(calls)


def record(h, src, reps, memcpy=False):
    sizes = segments(h, src)
    moved = int(np.sum(sizes))
    ms = time_resample(h, src, reps)
    out = {"replicates": h.R, "overwritten": int((src != np.arange(h.R)).sum()), "copies": len(sizes),
           "bytes_copied": moved, "algorithmic_bytes": 2 * moved, "resample_ms": ms,
           "resample_GBps": 2 * moved / (ms * 1e-3) / 1e9,
           "fraction_of_hbm_peak": 2 * moved / (ms * 1e-3) / HBM_BYTES_PER_S}
    if memcpy:
        mms, n = time_memcpy_per_segment(sizes, max(2, reps // 5))
        out.update({"memcpy_per_segment_ms": mms, "memcpy_calls": n,
                    "memcpy_per_segment_GBps": 2 * moved / (mms * 1e-3) / 1e9})
    return out


def run(scenario, R, seed, t_direct, leaps, reps, memcpy):
    (U, K, S), setup = SCENARIOS[scenario]
    e = Eng(U, K, S, seed, False, False, int(1e6), 0.0, replicates=R, device=0)
    setup(e)
    h = e._sync_params()
    h.simulate_direct(250000, -1, t_direct, 200)
    h.simulate_tau(leaps, -1, -1.0, 1)
    tau_ms = h.last_kernel_ms()
    c = h.get_counters()
    w = np.random.default_rng(12345).random(R)
    src = systematic_map(w, 0.5)
    out = {"shape": "%s: %d sites x %d demes x %d groups, P = %d" % (scenario, U, K, S, h.P),
           "direct_to_t": t_direct, "tau_leaps": leaps, "leaps_taken_mean": float(c["leaps"].mean()),
           "dense_row_bytes": ((h.P + 7) & ~7) * 4, "tau_step_ms": tau_ms}
    out.update(record(h, src, reps, memcpy))
    # the map is a copy of the batch: every destination now holds its source's run
    Sx, I = h.get_state()
    assert all(np.array_equal(I[r], I[src[r]]) for r in range(R))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--replicates", type=int, default=4096)
    ap.add_argument("--leaps", type=int, default=32)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--world-replicates", type=int, default=32)
    ap.add_argument("--world-leaps", type=int, default=101)
    args = ap.parse_args()
    torch.cuda.init()
    res = {"card": card(), "hbm_peak_Bps": HBM_BYTES_PER_S}
    res["t3"] = run("t3", args.replicates, 2024, 60.0, args.leaps, args.reps, True)
    torch.cuda.empty_cache()
    res["world"] = run("w", args.world_replicates, 4242, 40.0, args.world_leaps, args.reps, False)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
