"""Sequence calls on the GPU (fks_forward_simulate_sequence): one launch that runs every particle through M legs must return,
byte for byte, what M chained single calls return (leg k from leg k-1's end states, particle ids first + k * n), in every
noise mode; in injection mode it must meet the oracle parity bar leg by leg."""
import os
import subprocess

import numpy as np
import pytest

from fast_kinematic_simulator_b200 import capi, workloads as W

import parity
import sequence_chain as SC

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def three_legs(w, n, per_particle=False, offset=0):
    """contact target -> back to the start -> a third waypoint between them; (3, n_targets, stride)"""
    starts, t = w.subset(n, offset)
    target = np.broadcast_to(t, starts.shape) if t.shape[0] == 1 else t
    third = 0.5 * (starts + target)
    if w.kind == capi.ROBOT_SE3:
        third = np.array(target)
        third[:, [3, 7, 11]] = 0.5 * (starts[:, [3, 7, 11]] + target[:, [3, 7, 11]])
    legs = np.stack([target, starts, third])
    if not per_particle:
        legs = legs[:, :1]
    return starts, np.ascontiguousarray(legs)


def chain(sim, starts, legs, allow_contacts, noise_mode, first=0, tapes=None):
    n = starts.shape[0]
    out, at = [], starts
    for k in range(legs.shape[0]):
        r = sim.forward_simulate_robots(at, legs[k], allow_contacts, noise_mode, tapes[k] if tapes else None, first + k * n)
        out.append(r.records)
        at = r.configs
    return np.stack(out)


CASES = [("se2_arena", 128), ("se3_narrow_passage", 1024), ("arm_table", 2048), ("arm_elbow", 512), ("arm_selfcollision", 256),
         ("gantry", 256)]


@pytest.mark.parametrize("name,n", CASES)
@pytest.mark.parametrize("noise_mode", [capi.NOISE_PHILOX, capi.NOISE_NONE])
def test_sequence_equals_chained_single_calls(name, n, noise_mode):
    w = W.gantry(n) if name == "gantry" else W.make(name, n_particles=n)
    sim = w.make_simulator()
    for per_particle, allow_contacts in ((False, True), (True, True), (False, False)):
        starts, legs = three_legs(w, n, per_particle)
        sim.reset_statistics()
        seq = sim.forward_simulate_sequence(starts, legs, allow_contacts, noise_mode, first_particle_id=7)
        s_stats = sim.get_statistics()
        sim.reset_statistics()
        ref = chain(sim, starts, legs, allow_contacts, noise_mode, first=7)
        c_stats = sim.get_statistics()
        assert seq.records.shape == (3, n)
        bad = np.nonzero(seq.records.view(np.uint8).reshape(3, n, -1) != ref.view(np.uint8).reshape(3, n, -1))
        assert bad[0].size == 0, (per_particle, allow_contacts, sorted(set(zip(bad[0].tolist(), bad[1].tolist())))[:8])
        assert s_stats == c_stats, (per_particle, allow_contacts)
        if allow_contacts and name != "arm_selfcollision":
            assert ((seq.flags[0] & capi.FLAG_DID_CONTACT) != 0).any()
        if not allow_contacts and name in ("se2_arena", "arm_table"):
            assert ((seq.flags[0] & capi.FLAG_ENDED_BY_NOCONTACT) != 0).any()  # a stopped leg hands on its end state
    sim.close()


def test_one_leg_is_forward_simulate_robots():
    w = W.arm_table(1024)
    sim = w.make_simulator()
    one = sim.forward_simulate_sequence(w.starts, w.targets[None], True, capi.NOISE_PHILOX, first_particle_id=3)
    ref = sim.forward_simulate_robots(w.starts, w.targets, True, capi.NOISE_PHILOX, first_particle_id=3)
    assert one.records.shape == (1, 1024) and one.records[0].tobytes() == ref.records.tobytes()


@pytest.mark.parametrize("name,n,min_insensitive", [("se2_arena", 128, 0.25), ("arm_elbow", 512, 0.5), ("gantry", 256, 0.5),
                                                    ("se3_narrow_passage", 512, 0.5)])
def test_sequence_oracle_parity_injected(name, n, min_insensitive):
    """oracle chain (mt19937, decision tapes) -> the GPU sequence with the merged tape; per leg the parity bar of
    test_gpu_parity; and the GPU chain with the per-leg tapes equals the sequence byte for byte."""
    w = W.gantry(n) if name == "gantry" else W.make(name, n_particles=n)
    starts, legs = three_legs(w, n)
    orc = parity.make_oracle(w)
    ref, tapes, merged, sens = SC.run_sequence_with_tape(orc, starts, legs, True)
    sim = w.make_simulator()
    seq = sim.forward_simulate_sequence(starts, legs, True, capi.NOISE_INJECTED, merged)
    from fast_kinematic_simulator_b200.simulator import SimulationResults

    for k in range(3):
        rep = parity.compare(SimulationResults(seq.records[k]), ref[k], sens[k], with_decisions=True)
        print("leg", k, parity.describe(rep, sens[k]))
        assert len(rep["bad_insensitive"]) == 0, (k, rep["bad_insensitive"][:16])
        # sensitivity carries over to every later leg (the leg starts from a possibly different end state), so the share of
        # insensitive particles is pinned on the first leg; every leg must still reproduce nearly all particles
        if k == 0:
            assert rep["n_insensitive"] >= min_insensitive * n, rep["n_insensitive"]
        assert rep["n_match"] >= 0.99 * n, (k, rep["n_match"])
        assert ((seq.records[k]["flags"] & capi.FLAG_DECISION_DESYNC)[sens[k] == 0] == 0).all(), k
    gpu_chain = chain(sim, starts, legs, True, capi.NOISE_INJECTED, tapes=tapes)
    assert gpu_chain.tobytes() == seq.records.tobytes()


def test_device_variant_on_a_side_stream_and_partition_of_a_leg():
    import torch

    w = W.se3_narrow_passage(1000)
    sim = w.make_simulator()
    starts, legs = three_legs(w, 1000, per_particle=True)
    host = sim.forward_simulate_sequence(starts, legs, True, capi.NOISE_PHILOX, first_particle_id=11)
    n, rec = 1000, sim.result_stride
    d_starts = torch.from_numpy(starts).cuda()
    d_legs = torch.from_numpy(legs).cuda()
    d_res = torch.zeros(3 * n * rec, dtype=torch.uint8, device="cuda")
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        sim.forward_simulate_sequence_device(d_starts, d_legs, n, n, 3, d_res, True, capi.NOISE_PHILOX, first_particle_id=11,
                                             stream=side.cuda_stream)
    side.synchronize()
    dev = d_res.cpu().numpy().view(sim.dtype).reshape(3, n)
    assert dev.tobytes() == host.records.tobytes()
    for k in range(3):
        order = torch.zeros(n, dtype=torch.int32, device="cuda")
        n0, n1 = sim.end_states_partition(d_res.data_ptr() + k * n * rec, n, order)
        contact = (host.flags[k] & capi.FLAG_DID_CONTACT) != 0
        assert (n0, n1) == (int((~contact).sum()), int(contact.sum()))
        o = order.cpu().numpy()
        assert np.array_equal(o[:n0], np.nonzero(~contact)[0]) and np.array_equal(o[n0:], np.nonzero(contact)[0])


def test_multi_gpu_sequence_equals_single_gpu():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from fast_kinematic_simulator_b200.simulator import MultiGpuParticleContactSimulator

    n = 301  # not divisible by the device count
    w = W.arm_elbow(n)
    starts, legs = three_legs(w, n, per_particle=True)
    single = w.make_simulator()
    multi = MultiGpuParticleContactSimulator(w.environment(), w.robot, torch.cuda.device_count())
    a = single.forward_simulate_sequence(starts, legs, True, capi.NOISE_PHILOX, first_particle_id=5)
    b = multi.forward_simulate_sequence(starts, legs, True, capi.NOISE_PHILOX, first_particle_id=5)
    assert a.records.tobytes() == b.records.tobytes()
    orc = parity.make_oracle(w)
    _, _, merged, _ = SC.run_sequence_with_tape(orc, starts, legs[:, :1], True)
    a = single.forward_simulate_sequence(starts, legs[:, :1], True, capi.NOISE_INJECTED, merged)
    b = multi.forward_simulate_sequence(starts, legs[:, :1], True, capi.NOISE_INJECTED, merged)
    assert a.records.tobytes() == b.records.tobytes()


def test_validation():
    w = W.se2_arena(8)
    sim = w.make_simulator()
    starts, legs = three_legs(w, 8)
    stride = sim.config_stride
    out = np.empty((3, 8), dtype=sim.dtype)

    def call(n=8, n_targets=1, n_legs=3, targets=legs, noise=capi.NOISE_PHILOX, first=0):
        return capi.lib.fks_forward_simulate_sequence(sim._h, starts.ctypes.data, None if targets is None else targets.ctypes.data, n,
                                                      n_targets, n_legs, 1, noise, None, first, out.ctypes.data)

    assert call() == capi.OK
    assert call(n_legs=0) == capi.ERR_INVALID_ARGUMENT
    assert call(targets=None) == capi.ERR_INVALID_ARGUMENT
    assert call(n_targets=2) == capi.ERR_INVALID_ARGUMENT
    assert call(noise=capi.NOISE_INJECTED) == capi.ERR_INVALID_ARGUMENT
    assert call(first=2 ** 64 - 24) == capi.ERR_INVALID_ARGUMENT
    assert call(first=2 ** 64 - 25) == capi.OK
    assert call(n_legs=2 ** 31) == capi.ERR_INVALID_ARGUMENT  # rejected before the buffers of 2^31 legs are sized
    launches = sim.launch_count
    assert call(n=0) == capi.OK and sim.launch_count == launches
    assert stride == 3
    with pytest.raises(capi.FksError):
        sim.forward_simulate_sequence(starts, np.ones((3, 2, 3)), True)


def test_cpp_adapter_sequence_example(tmp_path):
    lib = os.path.join(ROOT, "fast_kinematic_simulator_b200")
    exe = str(tmp_path / "fksgpu_example_sequence")
    subprocess.check_call(["/usr/bin/g++", "-std=c++11", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "forward_simulate_sequence.cpp"), "-L" + lib, "-lfksgpu", "-Wl,-rpath," + lib,
                           "-o", exe])
    r = subprocess.run([exe], capture_output=True, text=True)
    print(r.stdout)
    assert r.returncode == 0 and "ok" in r.stdout and "FAILED" not in r.stdout, r.stdout + r.stderr
