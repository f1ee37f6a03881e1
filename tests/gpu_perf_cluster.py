"""Developer aid (not a test): fks_end_states_cluster on three segment shapes -- 2048 segments x 64 positions (many planner
edges), 64 x 1024 and 1 x 8192 -- against what a caller can do without it: fks_end_states_pairwise_distance per segment, the
matrix copied to the host, scipy linkage + fcluster there.  Records are synthetic SE(2) end states (uniform in a 4 x 4 box,
any heading), the threshold the 10 % quantile of a segment's distances.  Prints the card, then per workload and linkage the
median device time of the call over warmed repeats (CUDA events; the call returns after its stream finished) and the host
path's time, and checks that both give the same partition (the distances are tie-free)."""
import subprocess
import sys
import time

sys.path.insert(0, ".")
sys.path.insert(0, "tests")
import numpy as np
import torch
from scipy.cluster.hierarchy import fcluster, linkage

from fast_kinematic_simulator_b200 import capi, workloads as W

import cluster_reference as CR


def run(n_seg, seg_len, reps):
    n = n_seg * seg_len
    rng = np.random.default_rng(n_seg * 7919 + seg_len)
    sim = W.make("se2_arena", n_particles=4).make_simulator()
    rec = np.zeros(n, dtype=sim.dtype)
    rec["cfg"] = np.stack([rng.uniform(0, 4, n), rng.uniform(0, 4, n), rng.uniform(-np.pi, np.pi, n)], axis=1)
    dr = torch.from_numpy(rec.view(np.uint8).copy()).cuda()
    offsets = np.arange(0, n + 1, seg_len, dtype=np.uint64)
    labels = torch.empty(n, dtype=torch.int32, device="cuda")
    mat = torch.empty(seg_len, seg_len, dtype=torch.float64, device="cuda")
    ids = torch.arange(n, dtype=torch.int32, device="cuda")
    sim.end_states_pairwise_distance(dr, seg_len, mat, ids[:seg_len])
    d0 = mat.cpu().numpy()
    t = float(np.quantile(d0[np.triu_indices(seg_len, 1)], 0.1, method="lower"))
    for lk, method in ((capi.LINKAGE_SINGLE, "single"), (capi.LINKAGE_COMPLETE, "complete")):
        sim.end_states_cluster(dr, offsets, labels, t, lk)  # warm-up
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a, b in ev:
            a.record()
            counts = sim.end_states_cluster(dr, offsets, labels, t, lk)
            b.record()
        torch.cuda.synchronize()
        gpu_ms = float(np.median([a.elapsed_time(b) for a, b in ev]))
        got = labels.cpu().numpy().view(np.uint32)

        # the alternative: pairwise matrix per segment, device -> host, scipy on the host
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        want, base = [], 0
        for s in range(n_seg):
            sim.end_states_pairwise_distance(dr, seg_len, mat, ids[s * seg_len:(s + 1) * seg_len])
            d = mat.cpu().numpy()
            z = linkage(d[np.triu_indices(seg_len, 1)], method=method)
            lab = CR.canonical(fcluster(z, t, criterion="distance"))
            want.append(lab + base)
            base += int(lab.max()) + 1
        host_ms = (time.perf_counter() - t0) * 1e3
        same = np.array_equal(got, np.concatenate(want)) and int(counts.sum()) == base
        print("%5d x %5d  %-8s  t=%.4f  clusters %7d  fks_end_states_cluster %10.3f ms   pairwise + D2H + scipy %10.1f ms   same partition: %s"
              % (n_seg, seg_len, method, t, int(counts.sum()), gpu_ms, host_ms, same), flush=True)
        assert same
    sim.close()


if __name__ == "__main__":
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    print("device:", torch.cuda.get_device_name(0), "|", q.stdout.strip().splitlines()[0] if q.stdout.strip() else "nvidia-smi unavailable")
    run(2048, 64, reps=20)
    run(64, 1024, reps=10)
    run(1, 8192, reps=3)
