"""ctypes binding of libvgsim_b200.so (include/vgsim_b200.h).

The library is the product: it is loaded at import time and a missing/unbuildable library is a hard
error (no CPU fallback).  Creating a handle needs a CUDA device; everything host-side (parameter
validation in ``_engine.py``) works without one.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# VGSIM_B200_LIB: A/B debugging of two builds of this same library (never a different implementation)
LIB_PATH = os.environ.get("VGSIM_B200_LIB") or os.path.join(_HERE, "libvgsim_b200.so")

NCOUNTERS = 12
NSUMMARY = 24
COUNTER_NAMES = ("bCounter", "dCounter", "sCounter", "mCounter", "iCounter", "migPlus", "migNonPlus",
                 "swapLockdown", "good_attempt", "events", "leaps", "globalInfectious")

c_void_p, c_int, c_int64, c_uint64, c_float, c_char_p = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                                         ctypes.c_uint64, ctypes.c_float, ctypes.c_char_p)
# the source arrays of vgsim_upload_params in argument order (keys of BirthDeathModel.param_arrays); a parameter grid's
# patch indices address their concatenation
SOURCE_FIELDS = ("b", "d", "s", "mRate", "hapMutType", "sigma", "suscType", "T", "m", "cd", "cdBefore", "cdAfter",
                 "startLD", "endLD", "sm", "sizes")


def blob_len(sites, K, S):
    """Doubles in one parameter point's device blob (the Dims layout of csrc/common.cuh)."""
    H, Um = 4 ** sites, max(sites, 1)
    n = 3 * H + 3 * H * sites + H + S * H + S * S + S + K * K + 7 * K + H + 4 * H * Um + 1 + K
    return (n + 1) & ~1


def _load():
    from . import build as _build
    if not os.path.exists(LIB_PATH):
        # in-tree build (nvcc cross-compiles sm_100a without a GPU); raises if nvcc is unavailable
        _build.build()
    lib = ctypes.CDLL(LIB_PATH)
    if not hasattr(lib, "vgsim_resample") and LIB_PATH == _build.LIB and _build.have_nvcc():
        # a library built from older sources (it lacks the newest entry point): rebuild once and load the new file
        del lib
        _build.build(force=True)
        lib = ctypes.CDLL(LIB_PATH)
    P = c_void_p
    sig = {
        "vgsim_last_error": (c_char_p, []),
        "vgsim_version": (c_int, []),
        "vgsim_create": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_void_p)]),
        "vgsim_destroy": (c_int, [P]),
        "vgsim_set_stream": (c_int, [P, P]),
        "vgsim_set_seeds": (c_int, [P, P]),
        "vgsim_upload_params": (c_int, [P, c_int] + [P] * 17),
        "vgsim_upload_param_grid": (c_int, [P, c_int, c_int, P, P, P, P, c_int64, c_int, c_int]),
        "vgsim_get_params": (c_int, [P, c_int, P]),
        "vgsim_set_replicate_params": (c_int, [P, P]),
        "vgsim_set_state": (c_int, [P, P, P]),
        "vgsim_get_state": (c_int, [P, P, P, P, P]),
        "vgsim_set_state_dev": (c_int, [P, P, P]),
        "vgsim_state_dev": (c_int, [P, ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p)]),
        "vgsim_reset": (c_int, [P]),
        "vgsim_set_async": (c_int, [P, c_int]),
        "vgsim_wait": (c_int, [P]),
        "vgsim_recycle_log": (c_int, [P]),
        "vgsim_archive_tau_log": (c_int, [P]),
        "vgsim_archive_stats": (c_int, [P, ctypes.POINTER(c_int64), ctypes.POINTER(c_int64), ctypes.POINTER(c_int64)]),
        "vgsim_simulate_direct": (c_int, [P, c_int64, c_int64, c_float, c_int64]),
        "vgsim_simulate_tau": (c_int, [P, c_int64, c_int64, c_float, c_int64]),
        "vgsim_simulate_tau_blocks": (c_int, [P, c_int64, c_int64, c_float, c_int64, c_int64]),
        "vgsim_synchronize": (c_int, [P]),
        "vgsim_prop_num": (c_int64, [P]),
        "vgsim_propensities": (c_int, [P, c_int, P, P, P, P]),
        "vgsim_rates": (c_int, [P, c_int] + [P] * 8),
        "vgsim_get_counters": (c_int, [P, P, P]),
        "vgsim_get_event_log": (c_int, [P, c_int, P, c_int64]),
        "vgsim_get_multievents": (c_int, [P, c_int, c_int64] + [P] * 7),
        "vgsim_get_tau_log": (c_int, [P, c_int, c_int64, P, P]),
        "vgsim_set_event_log": (c_int, [P, c_int, P, c_int64, P]),
        "vgsim_num_lockdowns": (c_int64, [P, c_int]),
        "vgsim_get_lockdowns": (c_int, [P, c_int, P, P, P]),
        "vgsim_genealogy": (c_int, [P, P, P, P, c_int]),
        "vgsim_tree_size": (c_int64, [P, c_int]),
        "vgsim_get_tree": (c_int, [P, c_int, P, P, P]),
        "vgsim_num_mutations": (c_int64, [P, c_int]),
        "vgsim_get_mutations": (c_int, [P, c_int, P, P, P, P, P]),
        "vgsim_num_migrations": (c_int64, [P, c_int]),
        "vgsim_get_migrations": (c_int, [P, c_int, P, P, P, P]),
        "vgsim_epidemic_curves": (c_int, [P, c_int, c_int, c_int, P, P, P, P, P, P]),
        "vgsim_summaries": (c_int, [P, P]),
        "vgsim_summaries_dev": (c_int, [P, ctypes.POINTER(c_void_p)]),
        "vgsim_trajectories": (c_int, [P, P, c_int64, P]),
        "vgsim_trajectories_dev": (c_int, [P, P, c_int64, ctypes.POINTER(c_void_p)]),
        "vgsim_lineages_through_time": (c_int, [P, P, c_int64, P]),
        "vgsim_lineages_through_time_dev": (c_int, [P, P, c_int64, ctypes.POINTER(c_void_p)]),
        "vgsim_resample": (c_int, [P, P]),
        "vgsim_launch_count": (c_int64, [P]),
        "vgsim_set_tau_variant": (c_int, [P, c_int]),
        "vgsim_set_direct_variant": (c_int, [P, c_int]),
        "vgsim_tau_fixed_shape": (c_int, [P]),
        "vgsim_debug_tau_phases": (c_int, [P, P, c_int]),
        "vgsim_debug_tau_cta_end": (c_int, [P, P, c_int]),
        "vgsim_last_kernel_ms": (c_int, [P, ctypes.POINTER(c_float)]),
        "vgsim_last_kernel_id": (c_int64, [P]),
        "vgsim_kernel_ms": (c_int, [P, c_int64, ctypes.POINTER(c_float)]),
        "vgsim_counters_dev": (c_int, [P, ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p)]),
        "vgsim_test_poisson": (c_int, [P, c_int64, c_uint64, P]),
        "vgsim_test_hypergeometric": (c_int, [P, P, P, c_int64, P, c_int64, P, P]),
        "vgsim_test_choose": (c_int, [P, c_int, P, c_int, c_int, c_int, P, P, P, P]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError here = the library does not export the declared ABI
        fn.restype = res
        fn.argtypes = args
    return lib, tuple(sig)


lib, EXPORTS = _load()


class VgsimError(RuntimeError):
    pass


def _ck(rc):
    if rc != 0:
        raise VgsimError(lib.vgsim_last_error().decode())


def _count(n):
    """Result of an int64 count function: -1 is an error (e.g. a replicate out of range)."""
    if n < 0:
        raise VgsimError(lib.vgsim_last_error().decode())
    return int(n)


def _p(a):
    return None if a is None else a.ctypes.data_as(c_void_p)


def _arr(a, dtype):
    return None if a is None else np.ascontiguousarray(a, dtype=dtype)


def time_grid(times):
    """`times` as the contiguous float64 grid vgsim_trajectories / vgsim_lineages_through_time take: one dimension, at
    least one point, finite and strictly increasing values (ValueError otherwise; the C ABI checks the same rules)."""
    t = np.ascontiguousarray(times, dtype=np.float64)
    if t.ndim != 1:
        raise ValueError("time grid must be one-dimensional (got shape %s)" % (t.shape,))
    if t.size == 0:
        raise ValueError("time grid needs at least one point")
    bad = np.flatnonzero(~np.isfinite(t))
    if bad.size:
        raise ValueError("time grid: point %d (%r) is not finite" % (bad[0], t[bad[0]]))
    bad = np.flatnonzero(np.diff(t) <= 0)
    if bad.size:
        raise ValueError("time grid must be strictly increasing (point %d, %r, is not after point %d, %r)"
                         % (bad[0] + 1, t[bad[0] + 1], bad[0], t[bad[0]]))
    return t


class Handle:
    """RAII wrapper of a vgsim_handle (R replicates of one model shape on one CUDA device)."""

    def __init__(self, sites, K, S, replicates=1, param_points=1, device=None):
        self.sites, self.K, self.S, self.R, self.n_pp = sites, K, S, replicates, param_points
        self.H = 4 ** sites
        self._h = c_void_p()
        _ck(lib.vgsim_create(sites, K, S, replicates, param_points, -1 if device is None else int(device),
                             ctypes.byref(self._h)))
        self.P = int(lib.vgsim_prop_num(self._h))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib.vgsim_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- setup
    def set_stream(self, cuda_stream_ptr):
        _ck(lib.vgsim_set_stream(self._h, c_void_p(cuda_stream_ptr)))

    def set_seeds(self, seeds):
        seeds = _arr(seeds, np.uint64)
        assert seeds.shape == (self.R,)
        _ck(lib.vgsim_set_seeds(self._h, _p(seeds)))

    def upload_params(self, pp, a, reset_contact_density=True, cd_mask=None):
        f, i = np.float64, np.int64
        arrs = [_arr(a.get(k), f) for k in ("b", "d", "s", "mRate", "hapMutType", "sigma")]
        arrs.append(_arr(a.get("suscType"), i))
        arrs += [_arr(a.get(k), f) for k in ("T", "m", "cd", "cdBefore", "cdAfter", "startLD", "endLD", "sm")]
        arrs.append(_arr(a.get("sizes"), i))
        if cd_mask is None:
            cd_mask = np.full(self.K, 1 if reset_contact_density else 0, dtype=np.int32)
        arrs.append(_arr(cd_mask, np.int32))
        _ck(lib.vgsim_upload_params(self._h, pp, *[_p(x) for x in arrs]))

    def upload_param_grid(self, base_pp, axis_len, patch_off, patch_idx, patch_val, first_point, dst_pp0, n_points):
        """Points [dst_pp0, dst_pp0 + n_points) = points first_point.. of the row-major product of the axes, built on the
        device from point base_pp and one patch per axis value (include/vgsim_b200.h: vgsim_upload_param_grid)."""
        axis_len = _arr(axis_len, np.int32)
        off, idx, val = _arr(patch_off, np.int64), _arr(patch_idx, np.int64), _arr(patch_val, np.float64)
        assert off.shape == (int(axis_len.sum()) + 1,) and idx.shape == val.shape == (int(off[-1]),)
        _ck(lib.vgsim_upload_param_grid(self._h, int(base_pp), len(axis_len), _p(axis_len), _p(off), _p(idx), _p(val),
                                        int(first_point), int(dst_pp0), int(n_points)))

    def get_params(self, pp):
        """The device blob of parameter point pp (float64[blob_len])."""
        out = np.zeros(blob_len(self.sites, self.K, self.S), np.float64)
        _ck(lib.vgsim_get_params(self._h, int(pp), _p(out)))
        return out

    def set_replicate_params(self, mapping):
        m = _arr(mapping, np.int32)
        _ck(lib.vgsim_set_replicate_params(self._h, _p(m)))

    def set_state(self, Sx, I):
        Sx, I = _arr(Sx, np.int64), _arr(I, np.int64)
        assert Sx is None or Sx.shape == (self.R, self.K, self.S)
        assert I is None or I.shape == (self.R, self.K, self.H)
        _ck(lib.vgsim_set_state(self._h, _p(Sx), _p(I)))

    def set_state_dev(self, dSx_ptr, dI_ptr):
        _ck(lib.vgsim_set_state_dev(self._h, c_void_p(dSx_ptr), c_void_p(dI_ptr)))

    def state_dev_ptrs(self):
        a, b = c_void_p(), c_void_p()
        _ck(lib.vgsim_state_dev(self._h, ctypes.byref(a), ctypes.byref(b)))
        return a.value, b.value

    def reset(self):
        _ck(lib.vgsim_reset(self._h))

    def set_async(self, on=True):
        """Host-buffer copies only enqueue (buffers must be pinned and stay valid until wait())."""
        _ck(lib.vgsim_set_async(self._h, 1 if on else 0))

    def wait(self):
        _ck(lib.vgsim_wait(self._h))

    def archive_tau_log(self):
        """Dense tau rows -> sparse archive (non-zero counts only); frees the dense capacity for the next leap block."""
        _ck(lib.vgsim_archive_tau_log(self._h))

    def archive_stats(self):
        a, b, c = c_int64(), c_int64(), c_int64()
        _ck(lib.vgsim_archive_stats(self._h, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)))
        return {"entries_total": a.value, "entries_max": b.value, "leaps_archived": c.value}

    def recycle_log(self):
        _ck(lib.vgsim_recycle_log(self._h))

    def get_state(self, full=False, out=None):
        """out=(Sx, I): caller-owned (e.g. pinned) int64 buffers of the right shape to fill instead."""
        if out is not None:
            Sx, I = out
            assert Sx.shape == (self.R, self.K, self.S) and I.shape == (self.R, self.K, self.H)
            assert Sx.dtype == np.int64 and I.dtype == np.int64 and Sx.flags.c_contiguous and I.flags.c_contiguous
            _ck(lib.vgsim_get_state(self._h, _p(Sx), _p(I), None, None))
            return Sx, I
        Sx = np.empty((self.R, self.K, self.S), np.int64)
        I = np.empty((self.R, self.K, self.H), np.int64)
        cd = np.empty((self.R, self.K), np.float64)
        lock = np.empty((self.R, self.K), np.int64)
        _ck(lib.vgsim_get_state(self._h, _p(Sx), _p(I), _p(cd), _p(lock)))
        return (Sx, I, cd, lock) if full else (Sx, I)

    def resample(self, source):
        """Replicate r's whole run becomes the run replicate source[r] had before the call (include/vgsim_b200.h:
        vgsim_resample); seeds and parameter points stay with the slot.  A replicate that is copied from must keep its
        own run (source[source[r]] == source[r])."""
        s = np.asarray(source)
        if s.shape != (self.R,) or not np.issubdtype(s.dtype, np.integer):
            raise ValueError("resample: source must be an integer array of length %d (got %s of shape %s)"
                             % (self.R, s.dtype, s.shape))
        bad = np.flatnonzero((s < -2 ** 31) | (s >= 2 ** 31))
        if bad.size:
            raise ValueError("resample: replicate %d copies from %d: replicate out of range" % (bad[0], s[bad[0]]))
        s = np.ascontiguousarray(s, dtype=np.int32)
        _ck(lib.vgsim_resample(self._h, _p(s)))

    # ---- hot path
    def simulate_direct(self, iterations, sample_size=-1, time=-1.0, attempts=200, sync=True):
        _ck(lib.vgsim_simulate_direct(self._h, iterations, sample_size, time, attempts))
        if sync:
            self.synchronize()

    def simulate_tau(self, iterations, sample_size=-1, time=-1.0, attempts=200, sync=True):
        _ck(lib.vgsim_simulate_tau(self._h, iterations, sample_size, time, attempts))
        if sync:
            self.synchronize()

    def simulate_tau_blocks(self, iterations, sample_size=-1, time=-1.0, attempts=200, leap_block=128, sync=True):
        """simulate_tau in blocks of `leap_block` leaps, finished blocks moved to the sparse archive."""
        _ck(lib.vgsim_simulate_tau_blocks(self._h, iterations, sample_size, time, attempts, leap_block))
        if sync:
            self.synchronize()

    # bit 16 (ERR_CLAMPED): a MULTITYPE BIRTH record drew more coalescences than its cell has lineage pairs left.  The
    # reference walks off the end of a vector there (src/_BirthDeath.pyx:885-915: `lbs -= 2` per coalescence with no
    # bound); the device clamps, the tree stays valid -- reported as a warning, everything else raises.
    NONFATAL_FLAGS = 16

    def synchronize(self, strict=True):
        rc = lib.vgsim_synchronize(self._h)
        if rc != 0 and strict:
            msg = lib.vgsim_last_error().decode()
            if rc & ~self.NONFATAL_FLAGS:
                raise VgsimError(msg)
            import warnings
            warnings.warn(msg, RuntimeWarning, stacklevel=2)
        return rc

    def genealogy(self, seed=None, uniform_stream=None, raw_words=False, sync=True):
        seeds = None
        if seed is not None:
            seeds = (np.uint64(seed) + np.arange(self.R, dtype=np.uint64)) if np.isscalar(seed) else _arr(seed, np.uint64)
            seeds = _arr(seeds, np.uint64)
        us = offs = None
        if uniform_stream is not None:
            if isinstance(uniform_stream, np.ndarray) and uniform_stream.ndim == 1:
                uniform_stream = [uniform_stream]
            assert len(uniform_stream) == self.R
            dt = np.uint64 if raw_words else np.float64
            parts = [np.ascontiguousarray(u, dtype=dt) for u in uniform_stream]
            offs = np.zeros(self.R + 1, np.int64)
            offs[1:] = np.cumsum([len(x) for x in parts])
            us = np.concatenate(parts) if offs[-1] else np.zeros(1, dt)
        _ck(lib.vgsim_genealogy(self._h, _p(seeds), _p(us), _p(offs), 1 if raw_words else 0))
        if sync:
            self.synchronize()

    # ---- taps and outputs
    def propensities(self, replicate=0):
        out = np.empty(self.P, np.float64)
        dI = np.empty((self.K, self.H), np.float64)
        dS = np.empty((self.K, self.S), np.float64)
        tau = np.zeros(1, np.float64)
        _ck(lib.vgsim_propensities(self._h, replicate, _p(out), _p(dI), _p(dS), _p(tau)))
        return out, dI, dS, float(tau[0])

    def rates(self, replicate=0):
        K, H = self.K, self.H
        r = dict(A=np.empty(K), eff=np.empty((K, K)), maxEBM=np.empty(K), ev=np.empty((K, H, 4)), hp=np.empty((K, H)),
                 popRate=np.empty(K), migPop=np.empty(K), totals=np.empty(2))
        _ck(lib.vgsim_rates(self._h, replicate, *[_p(r[k]) for k in ("A", "eff", "maxEBM", "ev", "hp", "popRate",
                                                                     "migPop", "totals")]))
        return r

    def get_counters(self, out=None):
        if out is not None:
            c, t = out
            assert c.shape == (self.R, NCOUNTERS) and c.dtype == np.int64 and t.shape == (self.R,)
            _ck(lib.vgsim_get_counters(self._h, _p(c), _p(t)))
            return c, t
        c = np.empty((self.R, NCOUNTERS), np.int64)
        t = np.empty(self.R, np.float64)
        _ck(lib.vgsim_get_counters(self._h, _p(c), _p(t)))
        d = {name: c[:, i].copy() for i, name in enumerate(COUNTER_NAMES)}
        d["time"] = t
        return d

    def get_event_log(self, replicate=0):
        n = int(self.get_counters()["events"][replicate])
        out = np.zeros((6, n), np.float64)
        _ck(lib.vgsim_get_event_log(self._h, replicate, _p(out), n))
        return out

    def epidemic_curves(self, step_num, rep_first=0, rep_count=None,
                        want=("infectious", "susceptible", "removed", "sampled")):
        """One pass over the logs of replicates [rep_first, rep_first + rep_count): dict of int64 arrays
        infectious [n, T+1, K, H], susceptible [n, T+1, K, S], removed / sampled [n, T+1, K, H] (those named in
        `want`), time_points [n, T+1] and last_point [n]."""
        n = self.R - rep_first if rep_count is None else int(rep_count)
        T1 = int(step_num) + 1
        shapes = {"infectious": (n, T1, self.K, self.H), "susceptible": (n, T1, self.K, self.S),
                  "removed": (n, T1, self.K, self.H), "sampled": (n, T1, self.K, self.H)}
        out = {k: np.zeros(shapes[k], np.int64) for k in shapes if k in want}
        out["time_points"] = np.zeros((n, T1), np.float64)
        out["last_point"] = np.zeros(n, np.int32)
        _ck(lib.vgsim_epidemic_curves(self._h, int(rep_first), n, int(step_num), _p(out.get("infectious")),
                                      _p(out.get("susceptible")), _p(out.get("removed")), _p(out.get("sampled")),
                                      _p(out["time_points"]), _p(out["last_point"])))
        return out

    def get_tau_log(self, replicate=0):
        L = int(self.get_counters()["leaps"][replicate])
        counts = np.zeros((L, self.P), np.int32)
        tt = np.zeros((L, 2), np.float64)
        _ck(lib.vgsim_get_tau_log(self._h, replicate, L, _p(counts), _p(tt)))
        return counts, tt

    def get_multievents(self, replicate=0):
        L = int(self.get_counters()["leaps"][replicate])
        n = L * self.P
        i = np.int64
        num, typ, hap, pop, nhap, npop = (np.zeros(n, i) for _ in range(6))
        t = np.zeros(n, np.float64)
        _ck(lib.vgsim_get_multievents(self._h, replicate, n, _p(num), _p(t), _p(typ), _p(hap), _p(pop), _p(nhap), _p(npop)))
        return dict(num=num, time=t, type=typ, hap=hap, pop=pop, nhap=nhap, npop=npop)

    def set_event_log(self, replicate, chain6xN, I_end):
        chain = _arr(chain6xN, np.float64)
        I_end = _arr(I_end, np.int64)
        _ck(lib.vgsim_set_event_log(self._h, replicate, _p(chain), chain.shape[1], _p(I_end)))

    def get_lockdowns(self, replicate=0):
        n = _count(lib.vgsim_num_lockdowns(self._h, replicate))
        st, pop, t = np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n, np.float64)
        _ck(lib.vgsim_get_lockdowns(self._h, replicate, _p(st), _p(pop), _p(t)))
        return st, pop, t

    def get_tree(self, replicate=0):
        n = _count(lib.vgsim_tree_size(self._h, replicate))
        parent, pop, t = np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n, np.float64)
        if n:
            _ck(lib.vgsim_get_tree(self._h, replicate, _p(parent), _p(pop), _p(t)))
        return parent, pop, t

    def get_mutations(self, replicate=0):
        n = _count(lib.vgsim_num_mutations(self._h, replicate))
        node, AS, DS, site = (np.zeros(n, np.int64) for _ in range(4))
        t = np.zeros(n, np.float64)
        if n:
            _ck(lib.vgsim_get_mutations(self._h, replicate, _p(node), _p(AS), _p(DS), _p(site), _p(t)))
        return node, AS, DS, site, t

    def get_migrations(self, replicate=0):
        n = _count(lib.vgsim_num_migrations(self._h, replicate))
        node, oldp, newp = (np.zeros(n, np.int64) for _ in range(3))
        t = np.zeros(n, np.float64)
        if n:
            _ck(lib.vgsim_get_migrations(self._h, replicate, _p(node), _p(t), _p(oldp), _p(newp)))
        return node, t, oldp, newp

    def summaries(self):
        out = np.zeros((self.R, NSUMMARY), np.float64)
        _ck(lib.vgsim_summaries(self._h, _p(out)))
        return out

    def summaries_dev_ptr(self):
        p = c_void_p()
        _ck(lib.vgsim_summaries_dev(self._h, ctypes.byref(p)))
        return p.value

    def trajectories(self, times):
        """Every replicate's epidemic on the shared grid `times` (include/vgsim_b200.h: vgsim_trajectories): dict of int64
        arrays infectious_deme [R, T, K], infectious_hap [R, T, H], sampled_deme [R, T, K], sampled_hap [R, T, H] (state
        after every log row with time <= times[j]; samplings cumulative since the log start).  Rows of points after a
        replicate's current time are -1."""
        t = time_grid(times)
        K, H = self.K, self.H
        out = np.empty((self.R, t.size, 2 * (K + H)), np.int64)
        _ck(lib.vgsim_trajectories(self._h, _p(t), t.size, _p(out)))
        return {"infectious_deme": out[..., :K].copy(), "infectious_hap": out[..., K:K + H].copy(),
                "sampled_deme": out[..., K + H:2 * K + H].copy(), "sampled_hap": out[..., 2 * K + H:].copy()}

    def trajectories_dev_ptr(self, times):
        """Device pointer of the rows of `trajectories(times)`, int64 [R, T, 2K + 2H] in the order infectious per deme,
        per haplotype, sampled per deme, per haplotype (owned by the handle, valid until the next call)."""
        t = time_grid(times)
        p = c_void_p()
        _ck(lib.vgsim_trajectories_dev(self._h, _p(t), t.size, ctypes.byref(p)))
        return p.value

    def lineages_through_time(self, times):
        """Lineages of every replicate's genealogy alive at each grid time, int64 [R, T] (zeros for a replicate without
        a tree; include/vgsim_b200.h: vgsim_lineages_through_time)."""
        t = time_grid(times)
        out = np.empty((self.R, t.size), np.int64)
        _ck(lib.vgsim_lineages_through_time(self._h, _p(t), t.size, _p(out)))
        return out

    def lineages_through_time_dev_ptr(self, times):
        """Device pointer of the rows of `lineages_through_time(times)`, int64 [R, T] (owned by the handle)."""
        t = time_grid(times)
        p = c_void_p()
        _ck(lib.vgsim_lineages_through_time_dev(self._h, _p(t), t.size, ctypes.byref(p)))
        return p.value

    def last_kernel_ms(self):
        ms = c_float()
        _ck(lib.vgsim_last_kernel_ms(self._h, ctypes.byref(ms)))
        return float(ms.value)

    def kernel_ms_async(self):
        """Returns a callable that reads the device time of the launch just enqueued (blocking only when called)."""
        kid = int(lib.vgsim_last_kernel_id(self._h))

        def read():
            ms = c_float()
            _ck(lib.vgsim_kernel_ms(self._h, kid, ctypes.byref(ms)))
            return float(ms.value)
        return read

    def counters_dev_ptrs(self):
        a, b = c_void_p(), c_void_p()
        _ck(lib.vgsim_counters_dev(self._h, ctypes.byref(a), ctypes.byref(b)))
        return a.value, b.value

    def launch_count(self):
        return int(lib.vgsim_launch_count(self._h))

    def tau_phase_cycles(self, reset=True):
        """Critical-path cycles per leap phase accumulated by the tau kernel when variant bit 1 is set."""
        out = np.zeros(16, np.uint64)
        _ck(lib.vgsim_debug_tau_phases(self._h, _p(out), 1 if reset else 0))
        return out

    def tau_cta_end(self, reset=True):
        out = np.zeros(1024, np.uint64)
        _ck(lib.vgsim_debug_tau_cta_end(self._h, _p(out), 1 if reset else 0))
        return out.reshape(512, 2)

    def set_tau_variant(self, variant):
        """0 = small mutation / out-migration groups drawn as one Poisson total + multinomial split (product path),
        1 = every channel drawn separately like the reference (parity tap)."""
        _ck(lib.vgsim_set_tau_variant(self._h, int(variant)))

    def tau_fixed_shape(self):
        """(U, K, S) compiled into the warp kernel instance the last tau launch ran, None when it read the shape at
        run time (variant bit 6 forces that instance)."""
        v = int(lib.vgsim_tau_fixed_shape(self._h))
        return (v >> 16, (v >> 8) & 0xff, v & 0xff) if v else None

    def set_direct_variant(self, variant):
        """0 = the shared-memory direct kernel wherever a replicate's rates fit one SM's shared memory, the large-state
        kernel elsewhere; bit 0 = the large-state kernel on every shape (parity tap)."""
        _ck(lib.vgsim_set_direct_variant(self._h, int(variant)))


def test_poisson(lam, seed=1):
    lam = np.ascontiguousarray(lam, np.float64)
    out = np.zeros(lam.shape, np.int64)
    _ck(lib.vgsim_test_poisson(_p(lam), lam.size, seed, _p(out)))
    return out


def test_hypergeometric(good, bad, sample, raw_words):
    good, bad, sample = (np.ascontiguousarray(x, np.int64) for x in (good, bad, sample))
    raw = np.ascontiguousarray(raw_words, np.uint64)
    out = np.zeros(good.shape, np.int64)
    used = np.zeros(1, np.int64)
    _ck(lib.vgsim_test_hypergeometric(_p(good), _p(bad), _p(sample), good.size, _p(raw), raw.size, _p(out), _p(used)))
    return out, int(used[0])


def test_choose(w, x, skip=-1, small=False):
    """Device cumulative search (choose.cuh) over weights w for every target in x: (index, before, weight, residual)."""
    w = np.ascontiguousarray(w, np.float64)
    x = np.ascontiguousarray(x, np.float64)
    idx = np.zeros(x.shape, np.int64)
    before, wsel, resid = (np.zeros(x.shape, np.float64) for _ in range(3))
    _ck(lib.vgsim_test_choose(_p(w), w.size, _p(x), x.size, int(skip), 1 if small else 0, _p(idx), _p(before), _p(wsel),
                              _p(resid)))
    return idx, before, wsel, resid
