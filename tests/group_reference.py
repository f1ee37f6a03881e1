"""Reference side of the group tests (include/fksgpu.h, fks_end_states_groups and fks_end_states_gather_starts): the
definitions applied literally.  The minimax search takes a distance matrix rather than records, so the GPU tests can feed
it the GPU's own pairwise matrix, and it lives beside the other parity helpers, so the oracle is unchanged.

- members: the positions of each label in increasing order (a stable sort by label), as record ids;
- representative: the member p with the smallest r(p) = max over the other members q of d(min(p,q), max(p,q)), d the
  matrix entry [min][max] with NaN as +inf; ties to the smallest position; a singleton's r is 0.0;
- gather: slot s, j < per_group takes member j mod k of group selected[s]."""
import numpy as np


def members(labels, n_clusters, ids=None):
    """(offsets [n_clusters + 1], members [m]) of positions with labels[p]; ids maps positions to record ids."""
    labels = np.asarray(labels, dtype=np.int64)
    if labels.size and (labels.min() < 0 or labels.max() >= n_clusters):
        raise ValueError("a label is not below n_clusters")
    order = np.argsort(labels, kind="stable")
    sizes = np.bincount(labels, minlength=n_clusters)
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint32)
    rec = order if ids is None else np.asarray(ids)[order]
    return offsets, rec.astype(np.uint32)


def minimax(dist):
    """(member index, r) of the minimax member of a group whose k x k matrix (members in position order) is dist."""
    dist = np.asarray(dist, dtype=np.float64)
    k = dist.shape[0]
    if k == 0:
        raise ValueError("a group without members")
    if k == 1:
        return 0, 0.0
    iu = np.triu_indices(k, 1)
    vals = dist[iu].copy()
    vals[np.isnan(vals)] = np.inf
    w = np.full((k, k), -np.inf)  # the diagonal takes no part in the maximum
    w[iu] = vals
    w.T[iu] = vals
    r = w.max(axis=1)
    i = int(np.argmin(r))  # the first of the smallest: the smallest position
    return i, float(r[i])


def groups(labels, n_clusters, matrix_of, ids=None):
    """offsets, members, representatives, radius, sizes; matrix_of(c, member_positions) returns group c's matrix."""
    offsets, mem = members(labels, n_clusters, ids)
    order = np.argsort(np.asarray(labels, dtype=np.int64), kind="stable")
    reps = np.zeros(n_clusters, np.uint32)
    radius = np.zeros(n_clusters, np.float64)
    for c in range(n_clusters):
        a, b = int(offsets[c]), int(offsets[c + 1])
        i, r = minimax(matrix_of(c, order[a:b]))
        reps[c] = mem[a + i]
        radius[c] = r
    return offsets, mem, reps, radius, np.diff(offsets).astype(np.uint64)


def gather(offsets, members_, selected, per_group):
    """Record ids of the n_selected * per_group starts: slot s, j takes member j mod k of group selected[s]."""
    out = []
    for g in selected:
        a, b = int(offsets[g]), int(offsets[g + 1])
        out.append(np.asarray(members_[a:b])[np.arange(per_group) % (b - a)])
    return np.concatenate(out).astype(np.uint32) if out else np.zeros(0, np.uint32)
