"""CPU: the prioritized-replay restatement of test_prioritized_replay_gpu.py against brute force, and the C-ABI's checks
that run before any launch."""
import ctypes as C

import numpy as np
import pytest

from test_prioritized_replay_gpu import build_tree, descend, restated_draws


@pytest.mark.parametrize("L,zeros", [(1, 0.0), (8, 0.0), (4096, 0.3), (1 << 16, 0.9)])
def test_descent_equals_searchsorted_where_unambiguous(L, zeros):
    """The descent picks leaf i with cumsum[i-1] <= u < cumsum[i] (searchsorted on a float64 cumsum) wherever u is not
    within rounding of a boundary, and never an empty leaf: even u at or beyond the total lands on a nonzero leaf."""
    rng = np.random.default_rng(L)
    leaves = np.exp(rng.uniform(0, np.log(1e6), L)) * (rng.random(L) >= zeros)
    leaves[rng.integers(L)] = 1.0  # at least one nonzero leaf
    tree = build_tree(leaves)
    assert tree[1] > 0
    u = np.concatenate([rng.random(20000) * tree[1], [0.0, tree[1], np.nextafter(tree[1], np.inf)]])
    got = descend(tree, u) - L
    assert (leaves[got] > 0).all()
    cs = np.cumsum(leaves)
    want = np.minimum(np.searchsorted(cs, u, side="right"), L - 1)
    # a boundary is ambiguous when u lies within the two sums' rounding (log2 L additions of relative 2^-53 each)
    slack = (np.log2(L) + 2) * 2.0 ** -52 * tree[1]
    lo = np.searchsorted(cs, u - slack, side="right")
    hi = np.searchsorted(cs, u + slack, side="right")
    clear = (lo == hi) & (u < tree[1] - slack)
    assert clear.mean() > 0.99
    assert np.array_equal(got[clear], want[clear])


def test_restated_tree_is_pairwise_and_draws_are_stratified():
    leaves = np.array([0.0, 3.0, 0.0, 1.0, 4.0, 0.0, 0.0, 0.0])
    tree = build_tree(leaves)
    assert tree[1] == 8.0 and list(tree[2:4]) == [4.0, 4.0] and list(tree[4:8]) == [3.0, 1.0, 4.0, 0.0]
    slots, w = restated_draws(tree, 3, 0, 8, 1.0, 5)
    # strata [k, k+1) of a total of 8: slot 1 holds [0, 3), slot 3 [3, 4), slot 4 [4, 8)
    assert list(slots) == [1, 1, 1, 3, 4, 4, 4, 4]
    assert np.allclose(w, np.where(slots == 3, 1.0, np.where(slots == 1, 1 / 3, 1 / 4)))
    slots, w = restated_draws(np.zeros(16), 3, 0, 5, 0.4, 0)
    assert not slots.any() and not w.any()


def test_bad_sizes_are_refused_before_any_launch():
    """Capacity beyond 2^26, an L that does not fit the capacity and n beyond the capacity fail on the host (the fake
    pointers are never dereferenced)."""
    from gym_uav_collision_avoidance_b200 import _capi, build

    build.build()
    lib = _capi.load()
    fake = C.c_void_p(256)
    assert lib.uavca_per_sync(fake, 1 << 27, fake, fake, (1 << 26) + 1, None) == -1
    assert "2^26" in _capi.last_error()
    assert lib.uavca_per_sync(fake, 1024, fake, fake, 1025, None) == -1 and "L = 2048" in _capi.last_error()
    assert lib.uavca_per_update(fake, 1024, 1000, fake, fake, fake, 1001, None) == -1
    assert lib.uavca_per_sample(fake, fake, fake, fake, fake, 1000, 10, 2, fake, fake, 1024, 8, float("nan"), 0, 0,
                                fake, fake, fake, fake, fake, fake, fake, None) == -1
    assert "beta" in _capi.last_error()
