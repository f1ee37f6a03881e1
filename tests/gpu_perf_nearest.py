"""Developer aid (not a test): fks_nearest_configurations against the path a caller has without it -- the pairwise
distances of candidate chunks together with the queries (fks_end_states_pairwise_distance takes at most 65 535 records
and computes the whole matrix), the candidate x query block downloaded, then numpy.argpartition and a sort of the k kept.
Prints the card and its power limit, then per robot (synthetic SE(2) configurations, random arm_table joint values) and
shape (queries x candidates: 1 x 2^20, 64 x 65 536, 4 096 x 65 536), k = 64:
- the device time of the call: the median over warmed repeats of CUDA events around it (the candidates stay in L2 between
  repeats: 2^20 SE(2) configurations are 25 MB);
- the existing path's time: host clock from the first pairwise launch to the sorted host answer, one warmed pass;
- whether both gave the same ids and distance bits (random configurations: no ties at the k-th place).
Usage: python tests/gpu_perf_nearest.py [--reps R] [--out FILE.json]"""
import argparse
import json
import subprocess
import sys
import time

sys.path.insert(0, ".")
import numpy as np
import torch

from fast_kinematic_simulator_b200 import workloads as W

K = 64
SHAPES = [(1, 1 << 20), (64, 65536), (4096, 65536)]
PAIRWISE_MAX = 65535


def _u32(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint32).view(np.int32)).cuda()


def _configs(name, stride, n, rng):
    if name == "se2_arena":
        return np.stack([rng.uniform(0, 10, n), rng.uniform(0, 10, n), rng.uniform(-np.pi, np.pi, n)], axis=1)
    return rng.uniform(-np.pi, np.pi, (n, stride))


def existing_path(sim, dr, m, n_q):
    """(ids, distances) [n_q][K] through pairwise chunks, download and argpartition."""
    chunk = PAIRWISE_MAX - n_q
    q_ids = np.arange(m, m + n_q)
    blocks = []
    mat = torch.empty(PAIRWISE_MAX * PAIRWISE_MAX, dtype=torch.float64, device="cuda")
    for c0 in range(0, m, chunk):
        c = min(chunk, m - c0)
        ids = _u32(np.concatenate([np.arange(c0, c0 + c), q_ids]))
        n = c + n_q
        sim.end_states_pairwise_distance(dr, n, mat, ids)
        blocks.append(mat[:n * n].view(n, n)[:c, c:].cpu().numpy())
    d = np.ascontiguousarray(np.concatenate(blocks).T)  # [n_q][m]
    d[np.isnan(d)] = np.inf
    part = np.argpartition(d, K - 1, axis=1)[:, :K]
    dk = np.take_along_axis(d, part, axis=1)
    order = np.lexsort((part, dk), axis=1)
    ids = np.take_along_axis(part, order, axis=1).astype(np.uint32)
    return ids, np.take_along_axis(dk, order, axis=1)


def measure(name, n_q, m, reps):
    rng = np.random.default_rng(m + n_q)
    sim = W.make(name, n_particles=4).make_simulator()
    stride = sim.config_stride
    cand, queries = _configs(name, stride, m, rng), _configs(name, stride, n_q, rng)
    d_cand, d_q = torch.from_numpy(cand).cuda(), torch.from_numpy(queries).cuda()
    ids = torch.empty(n_q * K, dtype=torch.int32, device="cuda")
    dist = torch.empty(n_q * K, dtype=torch.float64, device="cuda")
    sim.nearest_configurations(d_cand, m, d_q, n_q, K, ids, dist)  # warm-up
    before = sim.launch_count
    sim.nearest_configurations(d_cand, m, d_q, n_q, K, ids, dist)
    launches = sim.launch_count - before
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        sim.nearest_configurations(d_cand, m, d_q, n_q, K, ids, dist)
        b.record()
    torch.cuda.synchronize()
    gpu_ms = float(np.median([a.elapsed_time(b) for a, b in ev]))
    got_ids = ids.cpu().numpy().view(np.uint32).reshape(n_q, K)
    got_d = dist.cpu().numpy().reshape(n_q, K)

    rec = np.zeros(m + n_q, dtype=sim.dtype)
    rec["cfg"] = np.concatenate([cand, queries])
    dr = torch.from_numpy(rec.view(np.uint8)).cuda()
    existing_path(sim, dr, min(m, 4096), n_q)  # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    want_ids, want_d = existing_path(sim, dr, m, n_q)
    host_ms = (time.perf_counter() - t0) * 1e3
    same = bool(np.array_equal(got_ids, want_ids) and got_d.tobytes() == want_d.tobytes())
    sim.close()
    del dr, d_cand, d_q
    torch.cuda.empty_cache()
    return dict(robot=name, queries=n_q, candidates=m, k=K, launches=launches, call_ms=gpu_ms, existing_path_ms=host_ms, same=same)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    card = q.stdout.strip().splitlines()[0] if q.stdout.strip() else "nvidia-smi unavailable"
    print("device:", torch.cuda.get_device_name(0), "|", card, flush=True)
    rows = []
    for name in ("se2_arena", "arm_table"):
        for n_q, m in SHAPES:
            r = measure(name, n_q, m, args.reps)
            rows.append(r)
            print(json.dumps(r), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(dict(card=card, rows=rows), f, indent=1)
    assert all(r["same"] for r in rows), "the two paths disagree"


if __name__ == "__main__":
    main()
