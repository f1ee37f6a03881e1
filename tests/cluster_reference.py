"""Reference side of the clustering tests (include/fksgpu.h, fks_end_states_cluster): flat agglomerative clustering under a
distance cutoff, applied literally.  It takes distance matrices rather than records, so the GPU tests can feed it the GPU's
own pairwise matrix, and it lives beside the other parity helpers, so the oracle is unchanged.

Per segment: start from singletons; a cluster is named by its smallest position (its representative); the linkage of two
clusters is the min (single) or max (complete) of the distances of their members; while some pair has a finite linkage
<= the threshold, merge the pair with the smallest (linkage, smaller rep, larger rep).  Every merge scans all active pairs."""
import numpy as np

LINKAGE_SINGLE, LINKAGE_COMPLETE = 0, 1


def segment_distances(dist, contact=None, separate_contact=False):
    """The clustering's view of a segment's matrix: entries [p][q], p < q, with NaN -> +inf and, with separate_contact,
    +inf between records whose contact flags differ; mirrored into a symmetric matrix with +inf on the diagonal."""
    dist = np.asarray(dist, dtype=np.float64)
    n = dist.shape[0]
    iu = np.triu_indices(n, 1)
    vals = dist[iu].copy()
    vals[np.isnan(vals)] = np.inf
    if separate_contact and contact is not None:
        contact = np.asarray(contact, dtype=bool)
        vals[contact[iu[0]] != contact[iu[1]]] = np.inf
    w = np.full((n, n), np.inf)
    w[iu] = vals
    w.T[iu] = vals
    return w


def cluster_segment(dist, linkage, max_cluster_distance, contact=None, separate_contact=False):
    """Segment-local labels (0 .. k-1 in increasing order of representative) and k."""
    if np.isnan(max_cluster_distance):
        raise ValueError("max_cluster_distance is NaN")
    if linkage not in (LINKAGE_SINGLE, LINKAGE_COMPLETE):
        raise ValueError("unknown linkage")
    n = np.asarray(dist).shape[0]
    if n == 0:
        return np.zeros(0, np.uint32), 0
    w = segment_distances(dist, contact, separate_contact)
    op = np.minimum if linkage == LINKAGE_SINGLE else np.maximum
    rep = np.arange(n)
    while True:
        # w is symmetric with +inf off the active clusters: the first minimum in row-major order is at (a, b) with a < b,
        # a the smallest representative of any pair at that linkage and b its smallest partner -- the smallest key
        k = int(np.argmin(w))
        a, b = divmod(k, n)
        lab = w[a, b]
        if not (lab < np.inf and lab <= max_cluster_distance):
            break
        row = op(w[a], w[b])
        row[a] = row[b] = np.inf
        w[a, :] = row
        w[:, a] = row
        w[b, :] = np.inf
        w[:, b] = np.inf
        rep[rep == b] = a
    reps = np.unique(rep)
    return np.searchsorted(reps, rep).astype(np.uint32), len(reps)


def cluster_segments(dists, linkage, max_cluster_distance, contacts=None, separate_contact=False):
    """Global labels and per-segment counts of a call whose segment s has the matrix dists[s] (contact flags contacts[s])."""
    labels, counts, base = [], [], 0
    for s, d in enumerate(dists):
        lab, k = cluster_segment(d, linkage, max_cluster_distance, None if contacts is None else contacts[s], separate_contact)
        labels.append(lab + base)
        counts.append(k)
        base += k
    return (np.concatenate(labels).astype(np.uint32) if labels else np.zeros(0, np.uint32)), np.array(counts, dtype=np.uint64)


def canonical(labels):
    """Relabel a flat clustering by first occurrence (0, 1, ... in order of each cluster's smallest position)."""
    _, first, inv = np.unique(np.asarray(labels), return_index=True, return_inverse=True)
    rank = np.empty(len(first), dtype=np.int64)
    rank[np.argsort(first)] = np.arange(len(first))
    return rank[inv].astype(np.uint32)
