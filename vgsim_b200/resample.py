"""Resampling maps for `Simulator.resample` / `BirthDeathModel.resample` / `Sweep.resample`.

A map gives every replicate slot r the replicate whose run it continues, source[r].  The device gather needs a map in
which a replicate that is copied from keeps its own run (source[source[r]] == source[r]); `systematic_map` builds such
maps from particle weights.
"""
import numpy as np


def systematic_map(weights, u):
    """Systematic resampling of R replicates by non-negative `weights` with the offset `u` in [0, 1).

    Replicate i gets floor or ceil of R * w_i / sum(w) offspring: the number of points (u + k) / R, k = 0..R-1, that fall
    in its interval of the cumulative normalised weights.  Every replicate with at least one offspring keeps its own slot;
    its extra copies fill the slots of replicates without offspring, in ascending slot order.  Returns int32[R]."""
    w = np.asarray(weights, dtype=np.float64)
    if w.ndim != 1 or w.size == 0:
        raise ValueError("weights must be a non-empty one-dimensional array")
    if not np.all(np.isfinite(w)) or np.any(w < 0):
        raise ValueError("weights must be finite and non-negative")
    total = w.sum()
    if not total > 0:
        raise ValueError("weights must not all be zero")
    u = float(u)
    if not 0.0 <= u < 1.0:
        raise ValueError("u must be in [0, 1)")
    R = w.size
    edges = np.cumsum(w) / total * R
    edges[-1] = R  # the last interval ends at R exactly, whatever the rounding of the sum
    # offspring of i: points u + k in [edges[i-1], edges[i])
    upto = np.minimum(np.ceil(edges - u), R).astype(np.int64)  # points u + k < edges[i]
    counts = np.diff(np.concatenate(([0], upto)))
    source = np.arange(R, dtype=np.int32)
    extra = np.repeat(np.arange(R), np.maximum(counts - 1, 0))
    dead = np.flatnonzero(counts == 0)
    source[dead] = extra  # as many extra copies as slots without offspring: the counts sum to R
    return source
