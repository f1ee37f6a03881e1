"""The clustering reference (tests/cluster_reference.py) against independent implementations: scipy's complete linkage +
fcluster(t, "distance") on tie-free matrices, connected components of D <= t for single linkage, and hand-built cases
that pin the tie rule, the label order and the +inf / NaN / separate_contact behaviour."""
import numpy as np
import pytest
from scipy.cluster.hierarchy import fcluster, linkage
from scipy.sparse.csgraph import connected_components

import cluster_reference as CR


def _random_matrix(rng, n):
    return rng.random((n, n)) * 10.0  # only the upper triangle is read; continuous: no ties


@pytest.mark.parametrize("n", [2, 7, 40, 150])
def test_complete_linkage_equals_scipy(n):
    rng = np.random.default_rng(n)
    d = _random_matrix(rng, n)
    z = linkage(d[np.triu_indices(n, 1)], method="complete")
    heights = z[:, 2]
    for t in list(np.quantile(heights, [0.0, 0.2, 0.5, 0.9])) + [heights[n // 3], heights[-1], -1.0, np.inf]:
        got, k = CR.cluster_segment(d, CR.LINKAGE_COMPLETE, t)
        want = CR.canonical(fcluster(z, t, criterion="distance")) if t >= 0 else np.arange(n, dtype=np.uint32)
        assert np.array_equal(got, want), t
        assert k == len(np.unique(want))


@pytest.mark.parametrize("n", [2, 9, 60, 200])
def test_single_linkage_equals_connected_components(n):
    rng = np.random.default_rng(100 + n)
    d = _random_matrix(rng, n)
    iu = np.triu_indices(n, 1)
    for t in list(np.quantile(d[iu], [0.0, 0.01, 0.05, 0.3])) + [d[0, n - 1]]:
        adj = np.zeros((n, n), bool)
        adj[iu] = d[iu] <= t
        _, comp = connected_components(adj, directed=False)
        got, k = CR.cluster_segment(d, CR.LINKAGE_SINGLE, t)
        assert np.array_equal(got, CR.canonical(comp)) and k == len(np.unique(comp)), t
        # and scipy's single linkage
        z = linkage(d[iu], method="single")
        assert np.array_equal(got, CR.canonical(fcluster(z, t, criterion="distance")))


def _upper(n, entries, fill=5.0):
    d = np.full((n, n), fill)
    for (p, q), v in entries.items():
        d[p, q] = v
    return d


def test_tie_rule_and_label_order():
    # d01 = d12 = 1 < d02 = 2: the tie (1, 0, 1) < (1, 1, 2) merges {0, 1} first; complete linkage then keeps 2 apart
    d = _upper(3, {(0, 1): 1.0, (1, 2): 1.0, (0, 2): 2.0})
    assert CR.cluster_segment(d, CR.LINKAGE_COMPLETE, 1.0)[0].tolist() == [0, 0, 1]
    assert CR.cluster_segment(d, CR.LINKAGE_SINGLE, 1.0)[0].tolist() == [0, 0, 0]
    # d02 = d12 = 1 < d01 = 2: (1, 0, 2) wins, 1 stays alone
    d = _upper(3, {(0, 2): 1.0, (1, 2): 1.0, (0, 1): 2.0})
    assert CR.cluster_segment(d, CR.LINKAGE_COMPLETE, 1.0)[0].tolist() == [0, 1, 0]
    # labels follow the smallest position of each cluster
    d = _upper(5, {(1, 3): 0.5, (0, 4): 0.25})
    assert CR.cluster_segment(d, CR.LINKAGE_COMPLETE, 1.0)[0].tolist() == [0, 1, 2, 1, 0]
    # the threshold is inclusive
    assert CR.cluster_segment(d, CR.LINKAGE_SINGLE, 0.5)[1] == 3 and CR.cluster_segment(d, CR.LINKAGE_SINGLE, np.nextafter(0.5, 0))[1] == 4
    # equal linkages everywhere: chained by the tie rule, complete linkage grows the cluster of 0 one position at a time
    d = np.ones((4, 4))
    assert CR.cluster_segment(d, CR.LINKAGE_COMPLETE, 1.0)[0].tolist() == [0, 0, 0, 0]


def test_infinite_nan_and_separate_contact():
    d = _upper(4, {(0, 1): np.nan, (0, 2): 1.0, (1, 2): 1.0, (2, 3): np.inf, (0, 3): 1.0, (1, 3): 1.0})
    # NaN is +inf: it never merges, and under complete linkage it keeps 0 and 1 apart
    got, k = CR.cluster_segment(d, CR.LINKAGE_COMPLETE, np.inf)
    assert got.tolist() == [0, 1, 0, 1] and k == 2
    got, k = CR.cluster_segment(d, CR.LINKAGE_SINGLE, np.inf)
    assert got.tolist() == [0, 0, 0, 0] and k == 1
    # separate_contact: pairs whose contact flags differ are +inf
    d = np.zeros((4, 4))
    contact = np.array([True, False, True, False])
    got, k = CR.cluster_segment(d, CR.LINKAGE_SINGLE, 1.0, contact, separate_contact=True)
    assert got.tolist() == [0, 1, 0, 1] and k == 2
    assert CR.cluster_segment(d, CR.LINKAGE_SINGLE, 1.0, contact, separate_contact=False)[1] == 1


def test_threshold_below_every_distance_gives_singletons():
    rng = np.random.default_rng(3)
    d = _random_matrix(rng, 30) + 1.0
    for lk in (CR.LINKAGE_SINGLE, CR.LINKAGE_COMPLETE):
        got, k = CR.cluster_segment(d, lk, 0.5)
        assert got.tolist() == list(range(30)) and k == 30


def test_segments_number_clusters_globally():
    rng = np.random.default_rng(4)
    mats = [_random_matrix(rng, n) for n in (0, 1, 5, 12)]
    labels, counts = CR.cluster_segments(mats, CR.LINKAGE_COMPLETE, 3.0)
    assert counts[0] == 0 and counts[1] == 1 and len(labels) == 18
    base = 0
    for s, n in enumerate((0, 1, 5, 12)):
        lo = sum((0, 1, 5, 12)[:s])
        seg = labels[lo:lo + n]
        assert np.array_equal(seg - base, CR.canonical(seg))
        base += int(counts[s])
    with pytest.raises(ValueError):
        CR.cluster_segment(mats[2], CR.LINKAGE_SINGLE, np.nan)
    with pytest.raises(ValueError):
        CR.cluster_segment(mats[2], 2, 1.0)
