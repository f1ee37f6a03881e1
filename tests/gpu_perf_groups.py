"""Developer aid (not a test): fks_end_states_groups and a whole planner edge on the device against the host round trip
they replace.  Prints the card, then
1. per group shape (2048 groups x 64 members, 8 x 1024, 1 x 8192; synthetic SE(2) end states, labels shuffled over the
   positions): the median device time of the groups call over warmed repeats (CUDA events; the call returns after its
   stream finished), and the host path's time: labels and records downloaded, members by a stable sort in numpy, and per
   group its pairwise matrix downloaded and searched for the minimax member (host clock, one pass).  Both must agree.
2. one arm_table planner edge (simulate -> partition -> cluster -> groups -> gather -> simulate), device-resident, against
   the same edge with the host round trip (labels, order and records downloaded, groups and starts made in numpy, the next
   batch simulated from host buffers); host clock around each edge, edges alternating, median of the repeats.  Both must
   give byte-identical second-batch records."""
import subprocess
import sys
import time

sys.path.insert(0, ".")
sys.path.insert(0, "tests")
import numpy as np
import torch

from fast_kinematic_simulator_b200 import capi, workloads as W

import group_reference as GR


def _u32(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint32).view(np.int32)).cuda()


def groups_shape(n_groups, size, reps):
    n = n_groups * size
    rng = np.random.default_rng(n_groups * 7919 + size)
    sim = W.make("se2_arena", n_particles=4).make_simulator()
    rec = np.zeros(n, dtype=sim.dtype)
    rec["cfg"] = np.stack([rng.uniform(0, 4, n), rng.uniform(0, 4, n), rng.uniform(-np.pi, np.pi, n)], axis=1)
    dr = torch.from_numpy(rec.view(np.uint8).copy()).cuda()
    labels = np.repeat(np.arange(n_groups), size).astype(np.uint32)
    rng.shuffle(labels)
    d_labels = _u32(labels)
    off = torch.empty(n_groups + 1, dtype=torch.int32, device="cuda")
    mem = torch.empty(n, dtype=torch.int32, device="cuda")
    rep = torch.empty(n_groups, dtype=torch.int32, device="cuda")
    rad = torch.empty(n_groups, dtype=torch.float64, device="cuda")
    sim.end_states_groups(dr, n, d_labels, n_groups, off, mem, rep, rad)  # warm-up
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        sim.end_states_groups(dr, n, d_labels, n_groups, off, mem, rep, rad)
        b.record()
    torch.cuda.synchronize()
    gpu_ms = float(np.median([a.elapsed_time(b) for a, b in ev]))

    mat = torch.empty(size * size, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    h_labels = d_labels.cpu().numpy().view(np.uint32)
    dr.cpu()  # the records, as a host caller would need them for the next batch's starts
    h_off, h_mem = GR.members(h_labels, n_groups)
    h_rep = np.zeros(n_groups, np.uint32)
    h_rad = np.zeros(n_groups)
    d_mem = _u32(h_mem)
    for c in range(n_groups):
        a, k = int(h_off[c]), int(h_off[c + 1] - h_off[c])
        sim.end_states_pairwise_distance(dr, k, mat, d_mem[a:a + k])
        i, r = GR.minimax(mat[:k * k].cpu().numpy().reshape(k, k))
        h_rep[c], h_rad[c] = h_mem[a + i], r
    host_ms = (time.perf_counter() - t0) * 1e3
    same = (np.array_equal(off.cpu().numpy().view(np.uint32), h_off) and np.array_equal(mem.cpu().numpy().view(np.uint32), h_mem)
            and np.array_equal(rep.cpu().numpy().view(np.uint32), h_rep) and rad.cpu().numpy().tobytes() == h_rad.tobytes())
    print("%5d groups x %5d members  fks_end_states_groups %9.3f ms   labels + records D2H, numpy, pairwise + D2H per group %9.1f ms"
          "   same: %s" % (n_groups, size, gpu_ms, host_ms, same), flush=True)
    assert same
    sim.close()


def edge(n, per_group, n_selected, reps):
    """n <= 8192: the cluster call takes parts of at most 8 192 positions"""
    w = W.make("arm_table", n_particles=n)
    sim = w.make_simulator()
    stride = sim.config_stride
    d_starts0, d_target0 = torch.from_numpy(w.starts).cuda(), torch.from_numpy(w.targets).cuda()
    dr = torch.empty(n * sim.result_stride, dtype=torch.uint8, device="cuda")
    order = torch.empty(n, dtype=torch.int32, device="cuda")
    labels = torch.empty(n, dtype=torch.int32, device="cuda")
    mem = torch.empty(n, dtype=torch.int32, device="cuda")
    n2 = n_selected * per_group
    starts = torch.empty(n2, stride, dtype=torch.float64, device="cuda")
    targets = torch.empty(n2, stride, dtype=torch.float64, device="cuda")
    dr2 = torch.empty(n2 * sim.result_stride, dtype=torch.uint8, device="cuda")
    # the cutoff: a fixed quantile of the distances among the first batch's first 2 048 records
    sim.forward_simulate_device(d_starts0, d_target0, n, 1, dr, True, capi.NOISE_PHILOX)
    s = min(n, 2048)
    m = torch.empty(s, s, dtype=torch.float64, device="cuda")
    sim.end_states_pairwise_distance(dr, s, m)
    v = m.cpu().numpy()[np.triu_indices(s, 1)]
    t = float(np.quantile(v[np.isfinite(v)], 0.05, method="lower"))
    mat = torch.empty(n * n, dtype=torch.float64, device="cuda")  # the host path's per-group matrices

    def first_half():
        sim.forward_simulate_device(d_starts0, d_target0, n, 1, dr, True, capi.NOISE_PHILOX)
        n_free, _ = sim.end_states_partition(dr, n, order)
        k = int(sim.end_states_cluster(dr, np.array([0, n_free, n], np.uint64), labels, t, capi.LINKAGE_COMPLETE, order).sum())
        return k

    def choose(sizes):
        sel = np.resize(np.argsort(-sizes.astype(np.int64), kind="stable"), n_selected)  # the largest groups
        g_targets = np.repeat(w.targets.reshape(1, stride), len(sel), axis=0)
        return sel, g_targets

    def device_edge():
        k = first_half()
        off = torch.empty(k + 1, dtype=torch.int32, device="cuda")
        rep = torch.empty(k, dtype=torch.int32, device="cuda")
        rad = torch.empty(k, dtype=torch.float64, device="cuda")
        sizes = sim.end_states_groups(dr, n, labels, k, off, mem, rep, rad, order)
        sel, g_targets = choose(sizes)
        sim.end_states_gather_starts(dr, off, mem, k, sel, per_group, starts, torch.from_numpy(g_targets).cuda(), targets)
        sim.forward_simulate_device(starts, targets, n2, n2, dr2, True, capi.NOISE_PHILOX, first_particle_id=n)
        torch.cuda.synchronize()
        return k

    def host_edge():
        k = first_half()
        rec = dr.cpu().numpy().view(sim.dtype)
        h_off, h_mem = GR.members(labels.cpu().numpy().view(np.uint32), k, order.cpu().numpy().view(np.uint32))
        d_mem = _u32(h_mem)
        for c in range(k):  # representatives, as the device call gives them: each group's pairwise matrix on the host
            a, kc = int(h_off[c]), int(h_off[c + 1] - h_off[c])
            sim.end_states_pairwise_distance(dr, kc, mat, d_mem[a:a + kc])
            GR.minimax(mat[:kc * kc].cpu().numpy().reshape(kc, kc))
        sel, g_targets = choose(np.diff(h_off).astype(np.uint64))
        ids = GR.gather(h_off, h_mem, sel, per_group)
        out = sim.forward_simulate_robots(np.ascontiguousarray(rec["cfg"][ids]), np.repeat(g_targets, per_group, axis=0), True,
                                          capi.NOISE_PHILOX, first_particle_id=n)
        return k, out.records

    device_edge()  # warm-up
    host_edge()
    dev_ms, host_ms = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        k = device_edge()
        dev_ms.append((time.perf_counter() - t0) * 1e3)
        t0 = time.perf_counter()
        _, host_rec = host_edge()
        host_ms.append((time.perf_counter() - t0) * 1e3)
    same = dr2.cpu().numpy().tobytes() == np.ascontiguousarray(host_rec).tobytes()
    print("arm_table edge: %5d particles, %4d groups, %d x %d next starts  device-resident %8.1f ms   host round trip %8.1f ms"
          "   same records: %s" % (n, k, n_selected, per_group, float(np.median(dev_ms)), float(np.median(host_ms)), same), flush=True)
    assert same
    sim.close()


if __name__ == "__main__":
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    print("device:", torch.cuda.get_device_name(0), "|", q.stdout.strip().splitlines()[0] if q.stdout.strip() else "nvidia-smi unavailable")
    groups_shape(2048, 64, reps=20)
    groups_shape(8, 1024, reps=10)
    groups_shape(1, 8192, reps=5)
    edge(2368, 256, 8, reps=5)
    edge(4096, 512, 16, reps=3)
