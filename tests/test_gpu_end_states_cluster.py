"""fks_end_states_cluster on the device against the clustering reference (tests/cluster_reference.py), which is fed the
matrices fks_end_states_pairwise_distance returns for the same ids.  Single and complete linkage use only min / max over
distances, so on the same distance bits the partition is unique: labels and counts must match exactly.  Thresholds are
taken as entries of those matrices (np.quantile with method="lower"), so a distance that differs by one ulp from the
pairwise kernel's shows up."""
import numpy as np
import pytest
import torch

from fast_kinematic_simulator_b200 import capi, workloads as W
from scipy.cluster.hierarchy import fcluster, linkage

import cluster_reference as CR
import device_records as DR

pytestmark = pytest.mark.gpu

SMALL_MAX = 160  # segments up to this many positions are clustered in shared memory (fks_consumers.cu)
MAX_SEGMENT = 8192


class Segments:
    """Ids of the records of every segment, their GPU distance matrices and contact flags."""

    def __init__(self, sim, dr, rec, segments):
        self.sim, self.dr = sim, dr
        self.segments = [np.asarray(s, dtype=np.uint32) for s in segments]
        self.offsets = np.concatenate([[0], np.cumsum([len(s) for s in self.segments])]).astype(np.uint64)
        self.ids = np.concatenate(self.segments) if self.segments else np.zeros(0, np.uint32)
        self.d_order = DR.u32(self.ids) if len(self.ids) else None
        self.mats = [DR.gpu_matrix(sim, dr, s) for s in self.segments]
        contact = (rec["flags"] & capi.FLAG_DID_CONTACT) != 0
        self.contacts = [contact[s] for s in self.segments]

    def entries(self, q):
        """entries of the matrices (upper triangles, finite) at quantiles q: thresholds equal to distances"""
        v = np.concatenate([m[np.triu_indices(len(m), 1)] for m in self.mats])
        v = v[np.isfinite(v)]
        return [float(x) for x in np.quantile(v, q, method="lower")]

    def run(self, lk, t, separate=False, stream=None):
        labels = torch.full((max(len(self.ids), 1),), -1, dtype=torch.int32, device="cuda")
        counts = self.sim.end_states_cluster(self.dr, self.offsets, labels, t, lk, self.d_order, separate,
                                             stream=stream if stream is not None else DR.stream())
        return labels[:len(self.ids)].cpu().numpy().view(np.uint32), counts

    def check(self, lk, t, separate=False):
        got, counts = self.run(lk, t, separate)
        want, want_counts = CR.cluster_segments(self.mats, lk, t, self.contacts, separate)
        assert np.array_equal(counts, want_counts), (lk, t, separate)
        assert np.array_equal(got, want), (lk, t, separate, int(np.sum(got != want)))
        return counts


def _chunks(ids, sizes):
    out, i, k = [], 0, 0
    while i < len(ids):
        out.append(ids[i:i + sizes[k % len(sizes)]])
        i += sizes[k % len(sizes)]
        k += 1
    return out


@pytest.mark.parametrize("name,n", [("arm_table", 700), ("se2_arena", 800), ("se3_narrow_passage", 800)])
def test_workload_end_states_match_the_reference(name, n):
    _, sim, dr, rec = DR.simulated(name, n)
    order = torch.empty(n, dtype=torch.int32, device="cuda")
    n_free, _ = sim.end_states_partition(dr, n, order, stream=DR.stream())
    order = order.cpu().numpy().view(np.uint32)
    # the planner's split: parts of the partition, cut into segments on both sides of the shared-memory limit
    parts = _chunks(order[:n_free], [40, SMALL_MAX, 250]) + _chunks(order[n_free:], [SMALL_MAX + 1, 90])
    split = Segments(sim, dr, rec, parts)
    # mixed contact flags in one segment: records in their natural order
    mixed = Segments(sim, dr, rec, _chunks(np.arange(n, dtype=np.uint32), [100, 300]))
    for lk in (CR.LINKAGE_SINGLE, CR.LINKAGE_COMPLETE):
        for t in split.entries([0.01, 0.1, 0.4]):
            split.check(lk, t)
        for t in mixed.entries([0.02, 0.3]):
            mixed.check(lk, t, separate=False)
            mixed.check(lk, t, separate=True)
    sim.close()


def test_segment_sizes_across_the_shared_memory_limit():
    _, sim, dr, rec = DR.simulated("se2_arena", 2100)
    sizes = [0, 1, 2, 31, 33, SMALL_MAX - 1, SMALL_MAX, SMALL_MAX + 1, 1500]
    segs = Segments(sim, dr, rec, np.split(np.arange(sum(sizes), dtype=np.uint32), np.cumsum(sizes)[:-1]))
    for lk in (CR.LINKAGE_SINGLE, CR.LINKAGE_COMPLETE):
        for t in segs.entries([0.05, 0.5]):
            counts = segs.check(lk, t)
            assert counts[0] == 0 and counts[1] == 1
    sim.close()


def test_one_segment_of_8192_against_scipy():
    n = MAX_SEGMENT
    rng = np.random.default_rng(8192)
    cfg = np.stack([rng.uniform(0, 10, n), rng.uniform(0, 10, n), rng.uniform(-3, 3, n)], axis=1)
    sim, dr, rec = DR.synthetic_se2(cfg, np.zeros(n, bool))
    mat = DR.gpu_matrix(sim, dr, np.arange(n, dtype=np.uint32))
    cond = mat[np.triu_indices(n, 1)]
    del mat
    assert np.all(np.isfinite(cond)) and len(np.unique(cond)) == len(cond)  # tie-free: scipy's order is then ours
    offsets = np.array([0, n], dtype=np.uint64)
    labels = torch.empty(n, dtype=torch.int32, device="cuda")
    for lk, method in ((CR.LINKAGE_COMPLETE, "complete"), (CR.LINKAGE_SINGLE, "single")):
        z = linkage(cond, method=method)
        for t in (z[n // 2, 2], z[n - n // 50, 2], float(np.quantile(z[:, 2], 0.9))):
            counts = sim.end_states_cluster(dr, offsets, labels, t, lk, stream=DR.stream())
            want = CR.canonical(fcluster(z, t, criterion="distance"))
            assert np.array_equal(labels.cpu().numpy().view(np.uint32), want), (method, t)
            assert counts.tolist() == [len(np.unique(want))]
    sim.close()


def test_ties_nan_and_contact_flags_on_synthetic_records():
    rng = np.random.default_rng(11)
    n = 600
    # SE(2) configurations on a small integer grid: most distances tie with many others
    cfg = np.stack([rng.integers(0, 3, n), rng.integers(0, 3, n), rng.integers(-1, 2, n) * (np.pi / 2)], axis=1).astype(np.float64)
    cfg[rng.random(n) < 0.05] = np.nan  # NaN configurations: their distances are NaN, clustered as +inf
    sim, dr, rec = DR.synthetic_se2(cfg, rng.random(n) < 0.4)
    segs = Segments(sim, dr, rec, _chunks(np.arange(n, dtype=np.uint32), [100, 400, 37, 63]))
    values = np.unique(np.concatenate([m[np.isfinite(m)] for m in segs.mats]))
    for lk in (CR.LINKAGE_SINGLE, CR.LINKAGE_COMPLETE):
        for t in (values[0], values[1], values[len(values) // 3], values[-1], np.inf):
            for separate in (False, True):
                segs.check(lk, t, separate)
    sim.close()


def test_all_legs_of_a_sequence_in_one_call():
    w = W.make("se2_arena", n_particles=300)
    n, m_legs = 300, 3
    sim = w.make_simulator()
    stride = sim.config_stride
    there = np.broadcast_to(w.targets.reshape(-1, stride), (n, stride))
    legs = np.stack([there, w.starts.reshape(n, stride), there])  # out, back, out again
    dr = torch.empty(m_legs * n * sim.result_stride, dtype=torch.uint8, device="cuda")
    sim.forward_simulate_sequence_device(torch.from_numpy(w.starts).cuda(), torch.from_numpy(np.ascontiguousarray(legs)).cuda(), n, n,
                                         m_legs, dr, stream=DR.stream())
    segments = []
    for k in range(m_legs):
        order = torch.empty(n, dtype=torch.int32, device="cuda")
        n_free, _ = sim.end_states_partition(dr[k * n * sim.result_stride:], n, order, stream=DR.stream())
        ids = order.cpu().numpy().view(np.uint32) + np.uint32(k * n)  # leg-major records from the base pointer
        segments += [ids[:n_free], ids[n_free:]]
    rec = dr.cpu().numpy().view(sim.dtype)
    segs = Segments(sim, dr, rec, segments)
    for lk in (CR.LINKAGE_SINGLE, CR.LINKAGE_COMPLETE):
        for t in segs.entries([0.05, 0.3]):
            counts = segs.check(lk, t)
            assert len(counts) == 2 * m_legs
    sim.close()


def test_repeated_calls_and_a_side_stream_agree():
    rng = np.random.default_rng(5)
    n = 64 * 20 + 700
    cfg = np.stack([rng.uniform(0, 4, n), rng.uniform(0, 4, n), rng.uniform(-3, 3, n)], axis=1)
    sim, dr, rec = DR.synthetic_se2(cfg, rng.random(n) < 0.5)
    segs = Segments(sim, dr, rec, _chunks(np.arange(n, dtype=np.uint32), [64] * 20 + [700]))
    t = segs.entries([0.1])[0]
    first = segs.run(capi.LINKAGE_COMPLETE, t, True)
    side = torch.cuda.Stream()
    for _ in range(3):
        again = segs.run(capi.LINKAGE_COMPLETE, t, True)
        assert np.array_equal(again[0], first[0]) and np.array_equal(again[1], first[1])
    with torch.cuda.stream(side):
        on_side = segs.run(capi.LINKAGE_COMPLETE, t, True, stream=side.cuda_stream)
    assert np.array_equal(on_side[0], first[0]) and np.array_equal(on_side[1], first[1])
    sim.close()


def test_invalid_arguments_and_empty_calls():
    rng = np.random.default_rng(6)
    sim, dr, rec = DR.synthetic_se2(rng.uniform(0, 1, (MAX_SEGMENT + 1, 3)), np.zeros(MAX_SEGMENT + 1, bool))
    labels = torch.empty(MAX_SEGMENT + 1, dtype=torch.int32, device="cuda")
    ok = np.array([0, 10], dtype=np.uint64)

    def refused(offsets=ok, t=1.0, lk=capi.LINKAGE_SINGLE, d_results=dr, d_labels=labels):
        with pytest.raises(capi.FksError) as e:
            sim.end_states_cluster(d_results, offsets, d_labels, t, lk)
        assert e.value.code == capi.ERR_INVALID_ARGUMENT

    refused(t=float("nan"))
    refused(lk=2)
    refused(lk=-1)
    refused(d_labels=None)
    refused(d_results=None)
    refused(offsets=np.array([1, 10], dtype=np.uint64))
    refused(offsets=np.array([0, 10, 5], dtype=np.uint64))
    refused(offsets=np.array([0, MAX_SEGMENT + 1], dtype=np.uint64))
    refused(offsets=np.arange(0, 2 ** 32 + 1, MAX_SEGMENT, dtype=np.uint64))  # m = 2^32 in segments of the maximum
    # nothing to cluster: no launch, counts are zero
    before = sim.launch_count
    assert sim.end_states_cluster(None, np.zeros(3, np.uint64), None, 1.0).tolist() == [0, 0]
    assert sim.end_states_cluster(None, np.zeros(1, np.uint64), None, 1.0).tolist() == []
    assert sim.launch_count == before
    # one call launches the same kernels whatever the number of segments
    sim.end_states_cluster(dr, np.array([0, 5], dtype=np.uint64), labels, 1.0)
    one = sim.launch_count - before
    sim.end_states_cluster(dr, np.arange(0, 1001, 5, dtype=np.uint64), labels, 1.0)
    assert sim.launch_count - before == 2 * one
    sim.close()
