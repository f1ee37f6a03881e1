"""Reference side of the nearest-configuration tests (include/fksgpu.h, fks_nearest_configurations): the definition applied
literally to a distance matrix it is given, so the GPU tests can feed it the GPU's own pairwise matrix.

- dist[i][j] is the distance from candidate i to query j; NaN counts as +inf;
- query j's answer is the first k candidates of a stable sort by (d, i), in that order, with their d;
- when m < k the remaining slots hold id 0xFFFFFFFF and +inf."""
import numpy as np

PAD_ID = np.uint32(0xFFFFFFFF)


def nearest(dist, k):
    """(ids [n_queries][k] uint32, distances [n_queries][k] float64) from an m x n_queries matrix."""
    dist = np.asarray(dist, dtype=np.float64)
    if dist.ndim != 2:
        raise ValueError("dist must be m x n_queries")
    m, n_queries = dist.shape
    ids = np.full((n_queries, k), PAD_ID, dtype=np.uint32)
    out = np.full((n_queries, k), np.inf, dtype=np.float64)
    take = min(k, m)
    for j in range(n_queries):
        d = dist[:, j].copy()
        d[np.isnan(d)] = np.inf
        order = np.argsort(d, kind="stable")[:take]  # stable: equal d keep increasing i
        ids[j, :take] = order
        out[j, :take] = d[order]
    return ids, out
