"""The nearest-configuration reference (tests/nearest_reference.py) against brute force and hand-built cases: ties,
duplicates, NaN, k > m and m = 0."""
import numpy as np
import pytest

import nearest_reference as NR


def brute_nearest(dist, k):
    """Repeatedly take the smallest (d, i) not yet taken, comparing keys one by one."""
    m, n_queries = dist.shape
    ids, out = [], []
    for j in range(n_queries):
        taken = set()
        row_ids, row_d = [], []
        for _ in range(k):
            best = None
            for i in range(m):
                if i in taken:
                    continue
                d = float(dist[i, j])
                d = np.inf if np.isnan(d) else d
                if best is None or (d, i) < best:
                    best = (d, i)
            if best is None:
                row_ids.append(0xFFFFFFFF)
                row_d.append(np.inf)
            else:
                taken.add(best[1])
                row_ids.append(best[1])
                row_d.append(best[0])
        ids.append(row_ids)
        out.append(row_d)
    return np.array(ids, dtype=np.uint32).reshape(n_queries, k), np.array(out, dtype=np.float64).reshape(n_queries, k)


def test_against_brute_force():
    rng = np.random.default_rng(1)
    for _ in range(200):
        m, n_queries, k = int(rng.integers(0, 12)), int(rng.integers(1, 5)), int(rng.integers(1, 15))
        d = rng.integers(0, 4, (m, n_queries)).astype(np.float64)  # small integers: many ties
        d[rng.random((m, n_queries)) < 0.1] = np.nan
        d[rng.random((m, n_queries)) < 0.05] = np.inf
        ids, out = NR.nearest(d, k)
        want_ids, want_out = brute_nearest(d, k)
        assert np.array_equal(ids, want_ids)
        assert out.tobytes() == want_out.tobytes()


def test_ties_go_to_the_smallest_index():
    d = np.array([[2.0], [1.0], [2.0], [1.0], [0.5]])
    ids, out = NR.nearest(d, 4)
    assert ids.tolist() == [[4, 1, 3, 0]]
    assert out.tolist() == [[0.5, 1.0, 1.0, 2.0]]


def test_duplicate_candidates_are_all_ranked():
    d = np.array([[3.0, 0.0], [3.0, 0.0], [3.0, 0.0]])
    ids, out = NR.nearest(d, 2)
    assert ids.tolist() == [[0, 1], [0, 1]]
    assert out.tolist() == [[3.0, 3.0], [0.0, 0.0]]


def test_nan_counts_as_inf_and_inf_is_ranked_by_index():
    d = np.array([[np.nan], [np.inf], [7.0], [np.nan]])
    ids, out = NR.nearest(d, 4)
    assert ids.tolist() == [[2, 0, 1, 3]]
    assert out[0, 0] == 7.0 and np.all(np.isinf(out[0, 1:]))
    assert not np.any(np.isnan(out))


def test_k_above_m_pads():
    d = np.array([[1.0, 2.0], [0.5, np.nan]])
    ids, out = NR.nearest(d, 5)
    assert ids.tolist() == [[1, 0] + [0xFFFFFFFF] * 3, [0, 1] + [0xFFFFFFFF] * 3]
    assert out[0].tolist() == [0.5, 1.0] + [np.inf] * 3
    assert out[1].tolist() == [2.0] + [np.inf] * 4


def test_no_candidates_is_all_padding():
    ids, out = NR.nearest(np.zeros((0, 3)), 7)
    assert ids.shape == (3, 7) and np.all(ids == 0xFFFFFFFF)
    assert np.all(out == np.inf)


def test_matrix_must_be_two_dimensional():
    with pytest.raises(ValueError):
        NR.nearest(np.zeros(4), 1)
