"""Replicate sharding over the GPUs of one node (SURVEY.md §8e).

Every replicate / parameter-sweep point is an independent Markov chain (the reference runs one chain per
process), so the path shards by replicate with NO data-path collective: rank g owns a contiguous range of
global replicate ids, each replicate's Philox key is derived from its GLOBAL id (so results do not depend on
the GPU count), and the only exchange is one all-gather of the fixed-size per-replicate summary vectors
(`VGSIM_NSUMMARY` fp64 each) at the end — NCCL over NVLink on GPUs, gloo in the CPU tests.
"""
import numpy as np


def replicate_range(rank, world, total):
    """[lo, hi) of global replicate ids owned by `rank` when `total` replicates are split over `world` ranks
    (contiguous, sizes differ by at most one, earlier ranks take the remainder)."""
    if not (0 <= rank < world):
        raise ValueError("rank out of range")
    base, rem = divmod(int(total), int(world))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def replicate_seeds(seed0, lo, hi, batch=0):
    """Philox keys of global replicates [lo, hi) for batch `batch`: seed0 + id in the low 32 bits' range, the
    batch index in the high word — a pure function of the GLOBAL id, never of the rank layout."""
    ids = np.arange(lo, hi, dtype=np.uint64)
    return (np.uint64(seed0) + ids + (np.uint64(batch) << np.uint64(32))).astype(np.uint64)


def sweep_point(replicate_id, n_inner):
    """(outer, inner) grid coordinates of a parameter-sweep replicate (BASELINE config 5: R0 x migration grid)."""
    return divmod(int(replicate_id), int(n_inner))


def gather_summaries(local, world, group=None):
    """All-gather per-replicate rows: `local` is a [n_local, ...] torch tensor of any trailing shape and dtype (CUDA for
    nccl, CPU for gloo), e.g. the summaries [n_local, NSUMMARY] float64, trajectories [n_local, T, 2K + 2H] int64 or
    lineages through time [n_local, T] int64.  Returns [sum n_local, ...] in global replicate order.  Ranks may own
    different numbers of replicates (remainder ranks), so rows are padded to the maximum and trimmed after the
    gather."""
    import torch
    import torch.distributed as dist
    if world == 1:
        return local.clone()
    n = torch.tensor([local.shape[0]], dtype=torch.int64, device=local.device)
    counts = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(counts, n, group=group)
    counts = [int(c.item()) for c in counts]
    nmax = max(counts)
    padded = torch.zeros((nmax,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    padded[: local.shape[0]] = local
    out = torch.empty((world * nmax,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, padded, group=group)
    out = out.view((world, nmax) + tuple(local.shape[1:]))
    return torch.cat([out[g, : counts[g]] for g in range(world)], dim=0)
