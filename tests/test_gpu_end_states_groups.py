"""fks_end_states_groups and fks_end_states_gather_starts on the device against the group reference
(tests/group_reference.py), fed the matrices fks_end_states_pairwise_distance returns for the same ids.  Offsets, members,
representatives, radius bits and host sizes must match exactly; so must the gathered starts and targets.  The last tests run
one planner edge on the device and the same edge through the host, and require byte-identical records of the next batch."""
import numpy as np
import pytest
import torch

from fast_kinematic_simulator_b200 import capi, workloads as W

import cluster_reference as CR
import group_reference as GR

pytestmark = pytest.mark.gpu

SMALL_MAX = 256  # groups up to this many members are searched by one CTA (fks_device_types.h)
MAX_GROUP = 8192


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _u32(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint32).view(np.int32)).cuda()


def _host_u32(t):
    return t.cpu().numpy().view(np.uint32)


def _simulated(name, n):
    w = W.make(name, n_particles=n)
    sim = w.make_simulator()
    dr = torch.empty(n * sim.result_stride, dtype=torch.uint8, device="cuda")
    sim.forward_simulate_device(torch.from_numpy(w.starts).cuda(), torch.from_numpy(w.targets).cuda(), n, w.targets.shape[0], dr, True,
                                capi.NOISE_PHILOX, stream=_stream())
    torch.cuda.synchronize()
    return w, sim, dr


def _synthetic_se2(cfg):
    sim = W.make("se2_arena", n_particles=4).make_simulator()
    rec = np.zeros(len(cfg), dtype=sim.dtype)
    rec["cfg"] = cfg
    return sim, torch.from_numpy(rec.view(np.uint8).copy()).cuda()


def _gpu_matrix(sim, dr, ids):
    m = len(ids)
    out = torch.empty(m, m, dtype=torch.float64, device="cuda")
    sim.end_states_pairwise_distance(dr, m, out, _u32(ids), stream=_stream())
    torch.cuda.synchronize()
    return out.cpu().numpy()


def run_groups(sim, dr, labels, n_clusters, ids=None, stream=None):
    m = len(labels)
    off = torch.full((n_clusters + 1,), -1, dtype=torch.int32, device="cuda")
    mem = torch.full((max(m, 1),), -1, dtype=torch.int32, device="cuda")
    reps = torch.full((max(n_clusters, 1),), -1, dtype=torch.int32, device="cuda")
    radius = torch.full((max(n_clusters, 1),), -1.0, dtype=torch.float64, device="cuda")
    sizes = sim.end_states_groups(dr, m, _u32(labels), n_clusters, off, mem, reps, radius, None if ids is None else _u32(ids),
                                  stream=stream if stream is not None else _stream())
    return (_host_u32(off), _host_u32(mem)[:m], _host_u32(reps)[:n_clusters], radius.cpu().numpy()[:n_clusters], sizes), (off, mem)


def check_groups(sim, dr, labels, n_clusters, ids=None, matrix_of=None):
    """GPU groups against the reference; matrix_of(c, positions) defaults to the GPU pairwise matrix of the group's records."""
    labels = np.asarray(labels, dtype=np.uint32)
    ids_np = np.arange(len(labels), dtype=np.uint32) if ids is None else np.asarray(ids, dtype=np.uint32)
    if matrix_of is None:
        def matrix_of(c, pos):
            return _gpu_matrix(sim, dr, ids_np[pos])
    got, dev = run_groups(sim, dr, labels, n_clusters, ids)
    want = GR.groups(labels, n_clusters, matrix_of, ids_np)
    off, mem, reps, radius, sizes = got
    assert np.array_equal(off, want[0])
    assert np.array_equal(mem, want[1])
    assert np.array_equal(reps, want[2]), int(np.sum(reps != want[2]))
    assert np.array_equal(radius.view(np.uint64), want[3].view(np.uint64))
    assert sizes.dtype == np.uint64 and np.array_equal(sizes, want[4])
    return got, dev


def segment_matrices(sim, dr, ids, offsets):
    """matrix_of for groups that stay inside segments: the submatrix of the segment's GPU pairwise matrix (an entry depends
    only on its two records, so the bits are those of a matrix over the group alone)."""
    seg_of = np.repeat(np.arange(len(offsets) - 1), np.diff(offsets).astype(np.int64))
    mats = [_gpu_matrix(sim, dr, ids[offsets[s]:offsets[s + 1]]) if offsets[s + 1] > offsets[s] else None for s in range(len(offsets) - 1)]

    def matrix_of(c, pos):
        s = seg_of[pos[0]]
        assert np.all(seg_of[pos] == s)
        local = pos - int(offsets[s])
        return mats[s][np.ix_(local, local)]

    return mats, matrix_of


def _cluster(sim, dr, ids, offsets, lk, t):
    labels = torch.empty(max(len(ids), 1), dtype=torch.int32, device="cuda")
    counts = sim.end_states_cluster(dr, np.asarray(offsets, np.uint64), labels, t, lk, _u32(ids), stream=_stream())
    return _host_u32(labels)[:len(ids)], int(counts.sum())


def _entries(mats, q):
    v = np.concatenate([m[np.triu_indices(len(m), 1)] for m in mats if m is not None])
    v = v[np.isfinite(v)]
    return [float(x) for x in np.quantile(v, q, method="lower")]


@pytest.mark.parametrize("name,n", [("se2_arena", 2000), ("se3_narrow_passage", 1500), ("arm_table", 1200)])
def test_workload_end_states_through_partition_and_cluster(name, n):
    _, sim, dr = _simulated(name, n)
    order = torch.empty(n, dtype=torch.int32, device="cuda")
    n_free, _ = sim.end_states_partition(dr, n, order, stream=_stream())
    ids = _host_u32(order)
    offsets = np.array([0, n_free, n], dtype=np.int64)
    mats, matrix_of = segment_matrices(sim, dr, ids, offsets)
    largest = 0
    for lk in (CR.LINKAGE_SINGLE, CR.LINKAGE_COMPLETE):
        for t in _entries(mats, [0.02, 0.2, 0.6]):
            labels, k = _cluster(sim, dr, ids, offsets, lk, t)
            got, _ = check_groups(sim, dr, labels, k, ids, matrix_of)
            largest = max(largest, int(got[4].max()))
    assert largest > SMALL_MAX  # both kernels of the search ran
    sim.close()


def test_all_legs_of_a_sequence_in_one_call():
    w = W.make("se2_arena", n_particles=400)
    n, m_legs = 400, 3
    sim = w.make_simulator()
    stride = sim.config_stride
    there = np.broadcast_to(w.targets.reshape(-1, stride), (n, stride))
    legs = np.stack([there, w.starts.reshape(n, stride), there])
    dr = torch.empty(m_legs * n * sim.result_stride, dtype=torch.uint8, device="cuda")
    sim.forward_simulate_sequence_device(torch.from_numpy(w.starts).cuda(), torch.from_numpy(np.ascontiguousarray(legs)).cuda(), n, n,
                                         m_legs, dr, stream=_stream())
    ids, offsets = [], [0]
    for k in range(m_legs):
        order = torch.empty(n, dtype=torch.int32, device="cuda")
        n_free, _ = sim.end_states_partition(dr[k * n * sim.result_stride:], n, order, stream=_stream())
        leg = _host_u32(order) + np.uint32(k * n)
        ids.append(leg)
        offsets += [offsets[-1] + n_free, offsets[-1] + n]
    ids = np.concatenate(ids)
    offsets = np.array(offsets, dtype=np.int64)
    mats, matrix_of = segment_matrices(sim, dr, ids, offsets)
    for t in _entries(mats, [0.05, 0.4]):
        labels, k = _cluster(sim, dr, ids, offsets, CR.LINKAGE_COMPLETE, t)
        check_groups(sim, dr, labels, k, ids, matrix_of)
    sim.close()


def test_ties_and_nan_configurations():
    rng = np.random.default_rng(21)
    n, k = 1500, 60
    # SE(2) configurations on a small integer grid: most distances tie; some NaN; group 0 all NaN (every r = +inf)
    cfg = np.stack([rng.integers(0, 3, n), rng.integers(0, 3, n), rng.integers(-1, 2, n) * (np.pi / 2)], axis=1).astype(np.float64)
    cfg[rng.random(n) < 0.05] = np.nan
    labels = rng.integers(1, k, n).astype(np.uint32)
    labels[rng.permutation(n)[:700]] = np.uint32(k - 1)  # one group across the small / large boundary
    labels[:k] = np.arange(k)
    labels[k:k + 5] = 0
    rng.shuffle(labels)
    nan_rows = np.flatnonzero(labels == 0)
    cfg[nan_rows] = np.nan
    sim, dr = _synthetic_se2(cfg)
    got, _ = check_groups(sim, dr, labels, k)
    assert got[3][0] == np.inf and got[2][0] == nan_rows[0]
    assert got[4].max() > SMALL_MAX
    # a permuted order of positions: ids are record ids
    ids = rng.permutation(n).astype(np.uint32)
    check_groups(sim, dr, labels, k, ids)
    sim.close()


def test_group_sizes_across_the_kernel_boundary_up_to_8192():
    sizes = [1, 2, 3, 31, SMALL_MAX - 1, SMALL_MAX, SMALL_MAX + 1, 1000, MAX_GROUP]
    n = sum(sizes)
    rng = np.random.default_rng(8192)
    cfg = np.stack([rng.uniform(0, 10, n), rng.uniform(0, 10, n), rng.uniform(-3, 3, n)], axis=1)
    sim, dr = _synthetic_se2(cfg)
    labels = np.repeat(np.arange(len(sizes)), sizes).astype(np.uint32)
    rng.shuffle(labels)
    ids = rng.permutation(n).astype(np.uint32)
    got, _ = check_groups(sim, dr, labels, len(sizes), ids)
    assert got[4].tolist() == sizes and got[3][0] == 0.0
    sim.close()


def test_repeated_calls_and_a_side_stream_agree():
    rng = np.random.default_rng(5)
    n, k = 6000, 700
    cfg = np.stack([rng.uniform(0, 4, n), rng.uniform(0, 4, n), rng.uniform(-3, 3, n)], axis=1)
    sim, dr = _synthetic_se2(cfg)
    labels = np.concatenate([np.arange(k), rng.integers(0, k, n - k - 600), np.full(600, 3)]).astype(np.uint32)
    rng.shuffle(labels)
    first, _ = run_groups(sim, dr, labels, k)
    for _ in range(3):
        again, _ = run_groups(sim, dr, labels, k)
        for a, b in zip(first, again):
            assert a.tobytes() == b.tobytes()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        on_side, _ = run_groups(sim, dr, labels, k, stream=side.cuda_stream)
    for a, b in zip(first, on_side):
        assert a.tobytes() == b.tobytes()
    sim.close()


def _gather(sim, dr, dev, n_clusters, selected, per_group, group_targets=None, stream=None):
    off, mem = dev
    stride = sim.config_stride
    n_out = len(selected) * per_group
    starts = torch.full((max(n_out, 1), stride), -7.0, dtype=torch.float64, device="cuda")
    targets = None if group_targets is None else torch.full((max(n_out, 1), stride), -7.0, dtype=torch.float64, device="cuda")
    gt = None if group_targets is None else torch.from_numpy(np.ascontiguousarray(group_targets, dtype=np.float64)).cuda()
    sim.end_states_gather_starts(dr, off, mem, n_clusters, selected, per_group, starts, gt, targets,
                                 stream=stream if stream is not None else _stream())
    torch.cuda.synchronize()
    return starts.cpu().numpy()[:n_out], None if targets is None else targets.cpu().numpy()[:n_out]


def test_gather_is_the_cyclic_fill():
    rng = np.random.default_rng(9)
    n, k = 3000, 40
    cfg = np.stack([rng.uniform(0, 4, n), rng.uniform(0, 4, n), rng.uniform(-3, 3, n)], axis=1)
    sim, dr = _synthetic_se2(cfg)
    labels = np.concatenate([np.arange(k), rng.integers(0, k, n - k)]).astype(np.uint32)
    rng.shuffle(labels)
    ids = rng.permutation(n).astype(np.uint32)
    got, dev = run_groups(sim, dr, labels, k, ids)
    off, mem, sizes = got[0], got[1], got[4]
    want_off, want_mem = GR.members(labels, k, ids)
    assert np.array_equal(off, want_off) and np.array_equal(mem, want_mem)
    small = int(np.argmin(sizes))
    for selected in ([small], [5, 5, 0, 39, small, 5], list(range(k))[::-1]):
        for per_group in (1, int(sizes[small]), int(sizes.max()) + 17):
            g_targets = rng.uniform(-1, 1, (len(selected), 3))
            starts, targets = _gather(sim, dr, dev, k, selected, per_group, g_targets)
            want = GR.gather(off, mem, selected, per_group)
            assert starts.tobytes() == np.ascontiguousarray(cfg[want]).tobytes()
            assert targets.tobytes() == np.repeat(g_targets, per_group, axis=0).tobytes()
            starts_only, none = _gather(sim, dr, dev, k, selected, per_group)
            assert none is None and starts_only.tobytes() == starts.tobytes()
    sim.close()


def _one_edge(name, n, per_group, q):
    """One planner edge on the device and through the host; returns the second batch's records of both."""
    w, sim, dr = _simulated(name, n)
    stride = sim.config_stride
    # device edge: partition, cluster, groups, gather, simulate
    order = torch.empty(n, dtype=torch.int32, device="cuda")
    n_free, _ = sim.end_states_partition(dr, n, order, stream=_stream())
    offsets = np.array([0, n_free, n], dtype=np.uint64)
    mat = _gpu_matrix(sim, dr, _host_u32(order))
    vals = mat[np.triu_indices(n, 1)]
    t = float(np.quantile(vals[np.isfinite(vals)], q, method="lower"))
    labels = torch.empty(n, dtype=torch.int32, device="cuda")
    counts = sim.end_states_cluster(dr, offsets, labels, t, capi.LINKAGE_COMPLETE, order, stream=_stream())
    k = int(counts.sum())
    off = torch.empty(k + 1, dtype=torch.int32, device="cuda")
    mem = torch.empty(n, dtype=torch.int32, device="cuda")
    reps = torch.empty(k, dtype=torch.int32, device="cuda")
    radius = torch.empty(k, dtype=torch.float64, device="cuda")
    sizes = sim.end_states_groups(dr, n, labels, k, off, mem, reps, radius, order, stream=_stream())
    by_size = np.argsort(-sizes.astype(np.int64), kind="stable")
    selected = np.concatenate([by_size[:4], by_size[-2:], by_size[:2]])  # the largest and the smallest groups, two repeats
    g_targets = np.where(np.arange(len(selected))[:, None] % 2 == 0, w.targets.reshape(-1, stride)[:1], w.starts.reshape(-1, stride)[:1])
    n2 = len(selected) * per_group
    starts = torch.empty(n2, stride, dtype=torch.float64, device="cuda")
    targets = torch.empty(n2, stride, dtype=torch.float64, device="cuda")
    sim.end_states_gather_starts(dr, off, mem, k, selected, per_group, starts, torch.from_numpy(np.ascontiguousarray(g_targets)).cuda(),
                                 targets, stream=_stream())
    dr2 = torch.empty(n2 * sim.result_stride, dtype=torch.uint8, device="cuda")
    sim.forward_simulate_device(starts, targets, n2, n2, dr2, True, capi.NOISE_PHILOX, first_particle_id=n, stream=_stream())
    torch.cuda.synchronize()
    device_records = dr2.cpu().numpy().tobytes()
    # host edge: download the records and the labels, group and gather in numpy, simulate from host buffers
    rec = dr.cpu().numpy().view(sim.dtype)
    h_off, h_mem = GR.members(_host_u32(labels), k, _host_u32(order))
    assert np.array_equal(h_off.astype(np.uint64)[1:] - h_off[:-1], sizes)
    h_ids = GR.gather(h_off, h_mem, selected, per_group)
    h_starts = np.ascontiguousarray(rec["cfg"][h_ids])
    h_targets = np.ascontiguousarray(np.repeat(g_targets, per_group, axis=0))
    out = sim.forward_simulate_robots(h_starts, h_targets, True, capi.NOISE_PHILOX, first_particle_id=n)
    host_records = np.ascontiguousarray(out.records).tobytes()
    sim.close()
    return device_records, host_records, sizes[selected]


@pytest.mark.parametrize("name,n,q", [("se2_arena", 600, 0.2), ("arm_table", 512, 0.3)])
def test_one_planner_edge_on_the_device_equals_the_host_edge(name, n, q):
    for per_group in (3, 64):
        device_records, host_records, chosen = _one_edge(name, n, per_group, q)
        assert chosen.min() < 64 and chosen.max() > 3  # per_group above some chosen groups' sizes and below others
        assert len(device_records) == len(host_records) and device_records == host_records


def test_invalid_arguments_and_empty_calls():
    rng = np.random.default_rng(6)
    n = 12000
    sim, dr = _synthetic_se2(rng.uniform(0, 1, (n, 3)))
    off = torch.empty(n + 1, dtype=torch.int32, device="cuda")
    mem = torch.empty(n, dtype=torch.int32, device="cuda")
    reps = torch.empty(n, dtype=torch.int32, device="cuda")
    radius = torch.empty(n, dtype=torch.float64, device="cuda")

    def refused(labels, k, m=None, **kw):
        args = dict(d_results=dr, m=len(labels) if m is None else m, d_labels=_u32(labels) if len(labels) else None, n_clusters=k,
                    d_group_offsets=off, d_members=mem, d_representatives=reps, d_radius=radius)
        args.update(kw)
        with pytest.raises(capi.FksError) as e:
            sim.end_states_groups(**args)
        assert e.value.code == capi.ERR_INVALID_ARGUMENT

    refused([0, 1, 2], 2)  # a label >= n_clusters, found on the device
    refused([0, 2, 2], 3)  # cluster 1 has no member
    refused(np.zeros(MAX_GROUP + 1, np.uint32), 1)  # more than 8192 members
    refused([0, 1], 3)  # n_clusters > m
    refused([0, 0], 0)
    refused([], 1, m=2 ** 32)
    for name in ("d_results", "d_labels", "d_group_offsets", "d_members", "d_representatives", "d_radius"):
        refused([0, 1], 2, **{name: None})
    # after refusals the workspace is clean: a valid call works
    check_groups(sim, dr, [1, 0, 1], 2)
    # nothing to group: no launch
    before = sim.launch_count
    assert sim.end_states_groups(None, 0, None, 0, None, None, None, None).tolist() == []
    assert sim.launch_count == before
    # the same launches for 1 group or 10 000
    sim.end_states_groups(dr, 5, _u32(np.zeros(5)), 1, off, mem, reps, radius)
    one = sim.launch_count - before
    sim.end_states_groups(dr, n, _u32(np.arange(n) % 10000), 10000, off, mem, reps, radius)
    assert sim.launch_count - before == 2 * one

    labels = np.arange(n) % 10
    _, dev = run_groups(sim, dr, labels, 10)
    d_off, d_mem = dev
    starts = torch.empty(100, 3, dtype=torch.float64, device="cuda")
    targets = torch.empty(100, 3, dtype=torch.float64, device="cuda")
    gt = torch.zeros(10, 3, dtype=torch.float64, device="cuda")

    def refused_gather(selected=(0, 1), per_group=2, n_clusters=10, **kw):
        args = dict(d_results=dr, d_group_offsets=d_off, d_members=d_mem, d_starts=starts)
        args.update(kw)
        with pytest.raises(capi.FksError) as e:
            sim.end_states_gather_starts(args["d_results"], args["d_group_offsets"], args["d_members"], n_clusters, selected, per_group,
                                         args["d_starts"], kw.get("d_group_targets"), kw.get("d_targets"))
        assert e.value.code == capi.ERR_INVALID_ARGUMENT

    refused_gather(per_group=0)
    refused_gather(per_group=0, selected=())
    refused_gather(selected=(0, 10))
    refused_gather(selected=(1,) * 2, per_group=2 ** 31)  # 2^32 starts
    refused_gather(selected=(-1,))
    for name in ("d_results", "d_group_offsets", "d_members", "d_starts"):
        refused_gather(**{name: None})
    refused_gather(d_targets=targets)
    refused_gather(d_group_targets=gt)
    before = sim.launch_count
    sim.end_states_gather_starts(None, None, None, 10, [], 4, None)
    assert sim.launch_count == before
    sim.end_states_gather_starts(dr, d_off, d_mem, 10, [3], 4, starts, gt, targets)
    assert sim.launch_count == before + 1
    sim.close()
