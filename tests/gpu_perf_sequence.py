"""Developer aid (not a test): a plan of M legs as ONE sequence call (fks_forward_simulate_sequence) against M chained
single calls -- host-buffer calls, and device calls whose end configurations are copied into the next call's starts on the
device.  Prints ms per plan and particle-microsteps/s, and checks at full size that the sequence and the chain agree."""
import subprocess
import sys
import time

sys.path.insert(0, ".")
import numpy as np
import torch

from fast_kinematic_simulator_b200 import capi, workloads as W


def plan(w, m):
    """M legs alternating between the workload's target and where the particles started (one target per leg)"""
    back = w.starts[:1]
    return np.ascontiguousarray(np.stack([w.targets[:1] if k % 2 == 0 else back for k in range(m)]))


def timed(fn, reps):
    fn()  # warm-up of every shape the timed calls use
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t0)
    return best * 1e3


def run(name, n, m, reps=3):
    w = W.make(name, n_particles=n)
    legs = plan(w, m)
    sim = w.make_simulator()
    stride, rec = sim.config_stride, sim.result_stride
    out = {}

    def sequence():
        out["seq"] = sim.forward_simulate_sequence(w.starts, legs, True, capi.NOISE_PHILOX).records

    def host_chain():
        at, recs = w.starts, []
        for k in range(m):
            r = sim.forward_simulate_robots(at, legs[k], True, capi.NOISE_PHILOX, first_particle_id=k * n)
            recs.append(r.records)
            at = r.configs
        out["chain"] = np.stack(recs)

    dev = torch.device("cuda")
    d_starts0 = torch.from_numpy(w.starts).to(dev)
    d_starts = torch.empty_like(d_starts0)
    d_legs = torch.from_numpy(legs).to(dev)
    d_res = torch.empty((m, n, rec), dtype=torch.uint8, device=dev)

    def device_chain():
        d_starts.copy_(d_starts0)
        for k in range(m):
            sim.forward_simulate_device(d_starts, d_legs[k], n, 1, d_res[k], True, capi.NOISE_PHILOX, first_particle_id=k * n)
            d_starts.copy_(d_res[k][:, :stride * 8].view(torch.float64))  # the end configurations start the next leg

    t_seq = timed(sequence, reps)
    t_host = timed(host_chain, reps)
    t_dev = timed(device_chain, reps)
    seq = out["seq"]
    assert seq.tobytes() == out["chain"].tobytes(), "sequence and chain of host calls differ"
    assert seq.tobytes() == d_res.cpu().numpy().tobytes(), "sequence and chain of device calls differ"
    micro = int(seq["n_microsteps"].sum())
    for label, t in (("one sequence call", t_seq), ("%d chained host calls" % m, t_host), ("%d chained device calls" % m, t_dev)):
        print("%-18s %6d particles x %d legs  %-24s %9.2f ms  %.3e particle-microsteps/s" % (name, n, m, label, t, micro / t * 1e3),
              flush=True)
    sim.close()


if __name__ == "__main__":
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    print("device:", torch.cuda.get_device_name(0), "|", q.stdout.strip().splitlines()[0] if q.stdout.strip() else "nvidia-smi unavailable")
    run("arm_table", 65536, 4)
    run("arm_table", 2368, 4)
    run("se2_arena", 128, 8, reps=10)
