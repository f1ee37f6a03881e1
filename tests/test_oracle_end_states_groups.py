"""The group reference (tests/group_reference.py) against brute force and hand-built cases: stable members, minimax ties,
NaN distances, singletons and the cyclic gather."""
import numpy as np
import pytest

import group_reference as GR


def brute_minimax(dist):
    k = len(dist)
    best = None
    for p in range(k):
        r = 0.0 if k == 1 else -np.inf
        for q in range(k):
            if q == p:
                continue
            d = dist[min(p, q)][max(p, q)]
            d = np.inf if np.isnan(d) else d
            r = max(r, d)
        if best is None or r < best[1]:
            best = (p, r)
    return best


def test_members_are_a_stable_sort_by_label():
    rng = np.random.default_rng(1)
    for _ in range(20):
        k = int(rng.integers(1, 12))
        labels = np.concatenate([np.arange(k), rng.integers(0, k, int(rng.integers(0, 60)))])
        rng.shuffle(labels)
        ids = rng.permutation(1000)[:len(labels)]
        offsets, mem = GR.members(labels, k, ids)
        assert offsets[0] == 0 and offsets[-1] == len(labels)
        for c in range(k):
            want = [ids[p] for p in range(len(labels)) if labels[p] == c]
            assert mem[offsets[c]:offsets[c + 1]].tolist() == want
    with pytest.raises(ValueError):
        GR.members([0, 3], 3)


def test_minimax_against_brute_force():
    rng = np.random.default_rng(2)
    for _ in range(200):
        k = int(rng.integers(1, 9))
        d = rng.integers(0, 4, (k, k)).astype(np.float64)  # small integers: many ties
        d[rng.random((k, k)) < 0.1] = np.nan
        d[rng.random((k, k)) < 0.05] = np.inf
        i, r = GR.minimax(d)
        bi, br = brute_minimax(d)
        assert (i, r) == (bi, br)


def test_ties_go_to_the_smallest_position():
    assert GR.minimax([[0.0, 2.5], [9.0, 0.0]]) == (0, 2.5)  # a pair: both r are d(0, 1); the lower entry is ignored
    d = np.array([[0, 1, 1], [0, 0, 1], [0, 0, 0]], dtype=np.float64)
    assert GR.minimax(d) == (0, 1.0)
    # the middle member is closest to both ends: r = 1 against 2
    d = np.array([[0, 1, 2], [0, 0, 1], [0, 0, 0]], dtype=np.float64)
    assert GR.minimax(d) == (1, 1.0)


def test_nan_is_infinite_and_singletons_have_radius_zero():
    assert GR.minimax([[np.nan]]) == (0, 0.0)
    nan = np.full((3, 3), np.nan)
    assert GR.minimax(nan) == (0, np.inf)
    d = np.array([[0, np.nan, 1], [0, 0, 2], [0, 0, 0]], dtype=np.float64)
    # r(0) = inf (NaN to 1), r(1) = inf, r(2) = max(1, 2) = 2
    assert GR.minimax(d) == (2, 2.0)


def test_groups_with_a_given_matrix():
    labels = np.array([2, 0, 2, 1, 0, 2])
    cfg = np.array([0.0, 10.0, 1.0, 5.0, 11.5, 3.0])

    def matrix_of(c, pos):
        x = cfg[pos]
        return np.abs(x[:, None] - x[None, :])

    offsets, mem, reps, radius, sizes = GR.groups(labels, 3, matrix_of, ids=np.arange(6) + 100)
    assert offsets.tolist() == [0, 2, 3, 6]
    assert mem.tolist() == [101, 104, 103, 100, 102, 105]
    assert sizes.tolist() == [2, 1, 3]
    assert reps.tolist() == [101, 103, 102] and radius.tolist() == [1.5, 0.0, 2.0]


def test_cyclic_gather():
    offsets = np.array([0, 3, 4, 6], dtype=np.uint32)
    mem = np.array([7, 8, 9, 4, 5, 6], dtype=np.uint32)
    # per_group below, equal to and above the group sizes; selected repeated and out of order
    assert GR.gather(offsets, mem, [2, 0, 2], 2).tolist() == [5, 6, 7, 8, 5, 6]
    assert GR.gather(offsets, mem, [0, 1], 3).tolist() == [7, 8, 9, 4, 4, 4]
    assert GR.gather(offsets, mem, [2, 0], 5).tolist() == [5, 6, 5, 6, 5, 7, 8, 9, 7, 8]
    assert GR.gather(offsets, mem, [], 4).tolist() == []
