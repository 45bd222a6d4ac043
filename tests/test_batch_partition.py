"""b200m_batch_partition, the split of a batch's pairs over a group's devices (pure host code): contiguous ranges in pair
order that cover every pair, with the least possible largest range cost."""
import itertools

import numpy as np
import pytest

from lidar_global_registration_b200 import build as b200_build
from lidar_global_registration_b200 import matcher as M


@pytest.fixture(scope="module", autouse=True)
def _lib():
    b200_build.build()
    M.load_library()


def _check_ranges(first, n_pairs, n_parts):
    assert first.shape == (n_parts + 1,)
    assert first[0] == 0 and first[-1] == n_pairs
    assert np.all(np.diff(first) >= 0)
    # unused parts are empty ranges at the end
    used = np.flatnonzero(np.diff(first) > 0)
    if used.size:
        assert np.all(np.diff(first)[used[-1] + 1:] == 0)


def _largest(cost, first):
    return max((sum(cost[a:b]) for a, b in zip(first[:-1], first[1:])), default=0.0)


def _brute_force(cost, n_parts):
    n = len(cost)
    best = sum(cost)
    for k in range(1, min(n_parts, n) + 1):
        for cuts in itertools.combinations(range(1, n), k - 1):
            b = (0,) + cuts + (n,)
            best = min(best, max(sum(cost[x:y]) for x, y in zip(b[:-1], b[1:])))
    return best


@pytest.mark.parametrize("seed", range(40))
def test_optimum_equals_brute_force(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 10))
    parts = int(rng.integers(1, 6))
    if seed % 2:   # integer costs: every sum is exact
        cost = [float(x) for x in rng.integers(0, 20, n)]
    else:
        cost = [float(x) for x in rng.exponential(1e9, n) * (rng.random(n) > 0.2)]
    first = M.batch_partition(cost, parts)
    _check_ranges(first, n, parts)
    got, want = _largest(cost, first), _brute_force(cost, parts)
    if seed % 2:
        assert got == want
    else:
        assert got == pytest.approx(want, rel=1e-12, abs=0)


def test_edge_cases():
    # empty batch
    assert M.batch_partition([], 4).tolist() == [0, 0, 0, 0, 0]
    # fewer pairs than parts: one pair per range, the rest empty at the end
    assert M.batch_partition([3.0, 1.0, 2.0], 8).tolist() == [0, 1, 2, 3, 3, 3, 3, 3, 3]
    # zero-cost pairs go with their neighbours and never raise the bound
    first = M.batch_partition([0.0, 5.0, 0.0, 0.0, 5.0, 0.0], 2)
    _check_ranges(first, 6, 2)
    assert _largest([0.0, 5.0, 0.0, 0.0, 5.0, 0.0], first) == 5.0
    first = M.batch_partition([0.0] * 5, 3)
    _check_ranges(first, 5, 3)
    assert np.all(np.diff(first) > 0)   # enough pairs: every part gets one
    # one dominant pair gets a range of its own
    cost = [1.0] * 10 + [1000.0] + [1.0] * 10
    first = M.batch_partition(cost, 3)
    _check_ranges(first, 21, 3)
    assert _largest(cost, first) == 1000.0
    assert [10, 11] in [[int(a), int(b)] for a, b in zip(first[:-1], first[1:])]
    # one part: everything
    assert M.batch_partition([1.0, 2.0, 3.0], 1).tolist() == [0, 3]
    # equal pairs spread evenly
    first = M.batch_partition([1.0] * 64, 8)
    assert np.all(np.diff(first) == 8)


@pytest.mark.parametrize("cost,parts", [([1.0, float("nan")], 2), ([1.0, -1.0], 2), ([float("inf")], 2), ([1.0], 0)])
def test_bad_arguments(cost, parts):
    with pytest.raises(M.B200MatchError):
        M.batch_partition(cost, parts)


def test_large_batch_is_fast_and_optimal_bound():
    rng = np.random.default_rng(7)
    cost = rng.integers(1, 1000, 5000).astype(np.float64)
    for parts in (2, 3, 8, 64):
        first = M.batch_partition(cost, parts)
        _check_ranges(first, len(cost), parts)
        got = _largest(cost.tolist(), first)
        # the least bound is feasible and one less is not (integer costs: the optimum is an integer)
        assert got >= cost.sum() / parts and got >= cost.max()

        def feasible(bound):
            n, acc = 1, 0.0
            for c in cost:
                if acc + c > bound:
                    n, acc = n + 1, c
                else:
                    acc += c
            return n <= parts

        assert feasible(got) and not feasible(got - 1)
