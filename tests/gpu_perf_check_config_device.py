"""Developer aid (not a test): fks_check_config_collision_device against the host call fks_check_config_collision.
Prints the card and its power limit, then per workload (arm_table: uniform joint values; se3_narrow_passage: 4 096 random
poses repeated), 2^20 configurations, inflation 0.5:
- the device call's time: the median of CUDA events around each of 20 warmed calls on configurations already on the device
  (they stay in L2 between calls: 2^20 arm configurations are 59 MB and fit in the 126 MB of L2, SE(3) ones are 101 MB);
- the host call's time: host clock around the whole call (H2D copy, kernel, D2H copy, synchronise), best of 3;
- whether both gave the same bytes.
Usage: python tests/gpu_perf_check_config_device.py [--reps R] [--out FILE.json]"""
import argparse
import json
import subprocess
import sys
import time

sys.path.insert(0, ".")
import numpy as np
import torch

from fast_kinematic_simulator_b200 import workloads as W

N = 1 << 20
INFLATION = 0.5


def _configs(name, n, rng):
    if name == "arm_table":
        return rng.uniform(-2.8, 2.8, (n, 7))
    base = np.stack([W._se3_config(np.array([rng.uniform(-0.6, 0.6), rng.uniform(-1.6, 1.2), rng.uniform(-0.5, 0.5)]),
                                   rng.normal(0, 0.6, 3)) for _ in range(4096)])
    return base[rng.integers(0, 4096, n)]


def measure(name, reps):
    sim = W.make(name, n_particles=4).make_simulator()
    cfg = np.ascontiguousarray(_configs(name, N, np.random.default_rng(5)))
    d_cfg = torch.from_numpy(cfg).cuda()
    d_out = torch.empty(N, dtype=torch.uint8, device="cuda")
    for _ in range(3):
        sim.check_config_collision_device(d_cfg, N, d_out, INFLATION)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        sim.check_config_collision_device(d_cfg, N, d_out, INFLATION)
        b.record()
    torch.cuda.synchronize()
    device_ms = float(np.median([a.elapsed_time(b) for a, b in ev]))
    got = d_out.cpu().numpy()

    sim.check_config_collision(cfg[:1024], INFLATION)
    host_ms = 1e9
    for _ in range(3):
        t0 = time.perf_counter()
        want = sim.check_config_collision(cfg, INFLATION)
        host_ms = min(host_ms, (time.perf_counter() - t0) * 1e3)
    same = got.tobytes() == want.view(np.uint8).tobytes()
    sim.close()
    return dict(workload=name, configurations=N, inflation=INFLATION, config_mb=cfg.nbytes / 1e6, device_call_ms=device_ms,
                host_call_ms=host_ms, colliding=float(want.mean()), same=same)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    card = q.stdout.strip().splitlines()[0] if q.stdout.strip() else "nvidia-smi unavailable"
    print("device:", torch.cuda.get_device_name(0), "|", card, flush=True)
    rows = []
    for name in ("arm_table", "se3_narrow_passage"):
        r = measure(name, args.reps)
        rows.append(r)
        print(json.dumps(r), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(dict(card=card, rows=rows), f, indent=1)
    assert all(r["same"] for r in rows), "the device and host calls disagree"


if __name__ == "__main__":
    main()
