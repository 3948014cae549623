"""systematic_map (vgsim_b200/resample.py): systematic resampling maps that vgsim_resample accepts."""
import numpy as np
import pytest

from vgsim_b200.resample import systematic_map


def _weights(rng, R):
    w = rng.random(R) * (rng.random(R) < 0.6)
    w[rng.integers(R)] += 0.1  # never all zero
    return w


def test_rule_and_offspring_counts():
    rng = np.random.default_rng(1)
    for _ in range(500):
        R = int(rng.integers(1, 200))
        w = _weights(rng, R)
        src = systematic_map(w, rng.random())
        assert src.shape == (R,) and src.dtype == np.int32
        assert np.all((src >= 0) & (src < R))
        assert np.array_equal(src[src], src)  # a replicate that is copied from keeps its own run
        n = np.bincount(src, minlength=R)
        e = R * w / w.sum()
        assert np.all((n == np.floor(e)) | (n == np.ceil(e))), (w, n)


def test_survivors_keep_their_slots_and_copies_fill_the_dead_in_order():
    rng = np.random.default_rng(2)
    for _ in range(200):
        R = int(rng.integers(2, 100))
        src = systematic_map(_weights(rng, R), rng.random())
        n = np.bincount(src, minlength=R)
        alive = np.flatnonzero(n > 0)
        assert np.array_equal(src[alive], alive)
        dead = np.flatnonzero(n == 0)
        assert np.array_equal(src[dead], np.repeat(alive, n[alive] - 1))
    np.testing.assert_array_equal(systematic_map([0, 1, 0, 3], 0.5), [3, 1, 3, 3])


def test_deterministic_in_u():
    rng = np.random.default_rng(3)
    w = _weights(rng, 64)
    for u in (0.0, 0.25, 0.999):
        np.testing.assert_array_equal(systematic_map(w, u), systematic_map(w.copy(), u))
    maps = {systematic_map(w, u).tobytes() for u in np.linspace(0.0, 0.99, 23)}
    assert len(maps) > 1


def test_equal_weights_give_the_identity():
    for R in (1, 7, 64, 1000):
        for u in (0.0, 0.5, 0.9999):
            np.testing.assert_array_equal(systematic_map(np.full(R, 2.5), u), np.arange(R))


@pytest.mark.parametrize("w", [[0.0, 0.0, 0.0], [1.0, -0.5, 2.0], [1.0, np.nan], [np.inf, 1.0], []])
def test_bad_weights_raise(w):
    with pytest.raises(ValueError):
        systematic_map(w, 0.5)


@pytest.mark.parametrize("u", [-0.1, 1.0, 1.5])
def test_u_outside_the_unit_interval_raises(u):
    with pytest.raises(ValueError):
        systematic_map([1.0, 2.0], u)
