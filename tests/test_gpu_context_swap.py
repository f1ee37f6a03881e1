"""Particle contexts that move between warps: at these sizes every context of a CTA's pool is parked in the global context
store and picked up again, by whichever warp the census assigns, many times per launch (bulk copies, fks_kernels.cu
context_swap).  A copy that is not complete or not ordered before the next reader shows up as a record that changes between
launches or streams, or that differs from the same particle simulated where its context never leaves its warp."""
import numpy as np
import pytest
import torch

from fast_kinematic_simulator_b200 import capi, workloads as W

import parity
from oracle import oracle_binding as OB

pytestmark = pytest.mark.gpu

# at least 8 particles per pool context: 148 CTAs x 48 contexts = 7 104 contexts
CASES = [("arm_table", 65536), ("se3_narrow_passage", 65536), ("se2_arena", 65536)]


@pytest.mark.parametrize("name,n", CASES)
def test_records_do_not_depend_on_launch_stream_or_warp(name, n):
    w = W.make(name, n_particles=n)
    sim = w.make_simulator()
    ref = sim.forward_simulate_robots(w.starts, w.targets, True, capi.NOISE_PHILOX).records.copy()
    assert sim.forward_simulate_robots(w.starts, w.targets, True, capi.NOISE_PHILOX).records.tobytes() == ref.tobytes()
    # device-resident calls on two streams of their own
    dev = torch.device("cuda")
    ds, dt = torch.from_numpy(w.starts).to(dev), torch.from_numpy(w.targets).to(dev)
    outs = [torch.empty(n * sim.result_stride, dtype=torch.uint8, device=dev) for _ in range(2)]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    torch.cuda.synchronize()
    for out, st in zip(outs, streams):
        sim.forward_simulate_device(ds, dt, n, w.targets.shape[0], out, True, capi.NOISE_PHILOX, stream=st.cuda_stream)
    torch.cuda.synchronize()
    for out in outs:
        assert out.cpu().numpy().tobytes() == ref.tobytes()
    # calls of at most one particle per SM: one warp per CTA, so no context ever moves to another warp
    step = 148
    for a in range(0, 1184, step):
        s, t = w.subset(step, a)
        part = sim.forward_simulate_robots(s, t, True, capi.NOISE_PHILOX, first_particle_id=a).records
        assert part.tobytes() == ref[a:a + step].tobytes(), (name, a)
    sim.close()


@pytest.mark.parametrize("name", [c[0] for c in CASES])
def test_oracle_parity_inside_a_large_batch(name):
    """m particles in injection mode, each simulated 128 times inside one batch of 128 m particles (the tapes repeated).
    Every copy must be byte for byte the record of the same particle simulated in a batch of m alone, and those records
    must meet the oracle at the bar of the parity tests: the oracle also injects the solution of every solve whose
    condition estimate exceeds 100 (as test_gpu_parity.py does for the arm, whose rank-deficient solves otherwise amplify
    last-bit differences of their input), no particle may differ without a reason the oracle enumerates, and for the arm
    every flag and counter must be the oracle's and no decision tape may fall out of step."""
    m, k = 256, 128
    w = W.make(name, n_particles=m)
    starts, targets = w.subset(m, 0)
    orc = parity.make_oracle(w)
    OB.lib().oracle_set_decision_cond_limit(orc._h, 100.0)
    ref, tape, sens = OB.run_with_tape(orc, starts, targets, True)
    draws, offs, dec, doffs = tape
    offs, doffs = offs.astype(np.uint64), doffs.astype(np.uint64)
    big_tape = (np.tile(draws, k),
                np.concatenate([offs[:-1] + np.uint64(j) * offs[-1] for j in range(k)] + [np.uint64(k) * offs[-1:]]),
                np.tile(dec, k),
                np.concatenate([doffs[:-1] + np.uint64(j) * doffs[-1] for j in range(k)] + [np.uint64(k) * doffs[-1:]]))
    big_starts = np.tile(starts, (k, 1))
    big_targets = targets if targets.shape[0] == 1 else np.tile(targets, (k, 1))
    sim = w.make_simulator()
    alone = sim.forward_simulate_robots(starts, targets, True, capi.NOISE_INJECTED, tape)
    small = alone.records.copy()
    gpu = sim.forward_simulate_robots(big_starts, big_targets, True, capi.NOISE_INJECTED, big_tape)
    for j in range(k):
        assert gpu.records[j * m:(j + 1) * m].tobytes() == small.tobytes(), (name, j)
    rep = parity.compare(alone, ref, sens, with_decisions=True)
    print(parity.describe(rep, sens))
    assert len(rep["bad_insensitive"]) == 0
    assert rep["n_match"] >= 0.99 * m, rep["n_match"]
    if name.startswith("arm") or rep["n_match"] == m:
        assert rep["discrete_ok"].all() and rep["n_desync"] == 0
    sim.close()
