"""Linked robots past the 7-DoF arm on the GPU (tests/wide_robots.py): 8, 11 and 15 DoF, 16 links, branching trees with
fixed joints inside branches and joints numbered out of depth-first order.  These shapes run code the arm never reaches:
the solver's second column slot (colpiv_qr_lanes<2>), noise batches of 32 / D microsteps, FK over arbitrary parent /
child nibbles, Jacobian columns masked by non-contiguous ancestor sets, up to 105 self-collision pairs in four
broad-phase chunks, and shared-memory layouts with fewer warps per CTA.  Each layer is compared with the oracle:
collision checks, one traced particle, whole batches in injection and Philox mode, then the consumers of a batch."""
import re

import numpy as np
import pytest
import torch

import cluster_reference as CR
import parity
import wide_robots as WR
from fast_kinematic_simulator_b200 import capi, simulator as S
from oracle import oracle_binding as OB

pytestmark = pytest.mark.gpu

CHECKED_ROBOTS = ["chain8", "chain15", "dual_arm", "dual_arm_all_pairs", "tree_fixed"]


def _threads_per_cta(sim):
    return int(re.search(r"(\d+) threads/CTA", sim.kernel_info).group(1))


def _persistent_grid(sim):
    return int(re.search(r"persistent grid (\d+)", sim.kernel_info).group(1))


def _workload_of_robot(name):
    return {"chain8": lambda: WR.chain(8, 4), "chain15": lambda: WR.chain(15, 4), "dual_arm": lambda: WR.dual_arm(4),
            "dual_arm_all_pairs": lambda: WR.dual_arm(4, "folded"), "tree_fixed": lambda: WR.tree_fixed(4)}[name]()


# ------------------------------------------------------------------------------------------------
# collision checks
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", CHECKED_ROBOTS)
@pytest.mark.parametrize("inflation", [0.0, 1.5])
def test_check_config_collision_matches_oracle(name, inflation):
    w = _workload_of_robot(name)
    rng = np.random.default_rng(23)
    cfg = rng.uniform(-2.8, 2.8, (2000, w.robot.n_dof))
    sim = w.make_simulator()
    orc = parity.make_oracle(w)
    got, ref = sim.check_config_collision(cfg, inflation), orc.check_config_collision(cfg, inflation)
    assert np.array_equal(got, ref), np.nonzero(got != ref)[0][:10]
    assert 0.02 < got.mean() < 0.999
    if name.startswith("dual_arm"):
        # the arms folded into each other, lifted off the obstacles: only the cross-branch pairs collide
        left, right = WR.FOLD_TARGET
        q = np.tile(WR._interleave(0.0, left, right), (256, 1)) + rng.normal(0.0, 0.05, (256, 15))
        g2, r2 = sim.check_config_collision(q, inflation), orc.check_config_collision(q, inflation)
        assert np.array_equal(g2, r2) and g2.mean() > 0.5
        apart = np.tile(WR._interleave(0.0, *WR.FOLD_START), (64, 1)) + rng.normal(0.0, 0.01, (64, 15))
        assert np.array_equal(sim.check_config_collision(apart, inflation), orc.check_config_collision(apart, inflation))
    sim.close()


# ------------------------------------------------------------------------------------------------
# one traced particle per robot (Philox noise): FK, actuation and noise at D = 8, 11, 15
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,pid", [("chain8_free", 3), ("tree_fixed_free", 1), ("tree_fixed_table", 5), ("dual_arm_free", 1),
                                      ("chain15_free", 0)])
def test_trace_matches_oracle(name, pid):
    """Philox draws differ from the oracle's in the last ulp (device libm), so a trace through solves whose round-off pivots
    are kept may part from the oracle's (the injected batches cover those); the tree's contact cuts nearly all of them."""
    w = WR.make(name, 8)
    t = w.targets[0]
    ref, rtr = parity.make_oracle(w).forward_simulate_traced(w.starts[pid], t, True, capi.NOISE_PHILOX, particle_id=pid)
    sim = w.make_simulator()
    got, gtr = sim.forward_simulate_robot_traced(w.starts[pid], t, True, capi.NOISE_PHILOX, particle_id=pid)
    assert len(gtr) == len(rtr) > 0
    for f in ("kind", "step", "microstep", "iteration"):
        assert np.array_equal(gtr[f], rtr[f]), f
    err = np.abs(gtr["values"] - rtr["values"]) / np.maximum(1.0, np.abs(rtr["values"]))
    assert err.max() <= parity.RTOL, err.max()
    assert got.records["flags"][0] & parity.SEMANTIC_FLAGS == ref["flags"][0] & parity.SEMANTIC_FLAGS
    if name in WR.CONTACT:
        assert (gtr["kind"] == capi.TRACE_RESOLUTION_STEP).any()
    batch = sim.forward_simulate_robots(w.starts[pid:pid + 1], t.reshape(1, -1), True, capi.NOISE_PHILOX, first_particle_id=pid)
    assert batch.records.tobytes() == got.records.tobytes()
    sim.close()


# ------------------------------------------------------------------------------------------------
# whole batches against the oracle
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(WR.CONTACT))
def test_contact_parity_with_ill_conditioned_solves_injected(name):
    """The bar of test_arm_table_parity_with_ill_conditioned_solves_injected: decision tape plus the solution of every
    solve whose condition estimate exceeds 100 injected, then every flag and counter of every particle identical, the
    statistics identical, no tape out of step, 99.9 % of the configurations within 1e-9 and all within 1e-7."""
    n = 1024
    w = WR.make(name, n)
    rep, gpu, ref, sens = parity.run_parity(w, n, decision_cond_limit=100.0)
    print(parity.describe(rep, sens))
    assert rep["discrete_ok"].all(), np.nonzero(~rep["discrete_ok"])[0][:10]
    assert rep["n_desync"] == 0
    assert rep["gpu_stats"] == rep["oracle_stats"]
    assert rep["n_match"] >= 0.999 * n, rep["n_match"]
    assert rep["cfg_err"].max() < 1e-7
    # the workload runs what it claims
    d = rep["decisions"]
    assert gpu.did_contact.all()
    assert ((d["flags"] & OB.DECISION_ROUNDOFF_PIVOT) != 0).sum() > 1000
    assert rep["n_overridden"] > 0  # the device's own solver decisions differed from the tape somewhere, and were overridden
    if name == "dual_arm_folded":
        assert rep["gpu_stats"]["unsuccessful_self_collision_resolves"] > 0


@pytest.mark.parametrize("name", list(WR.FREE))
def test_free_motion_philox_matches_oracle(name):
    """Philox noise on both sides over a whole batch: noise batches of 32 // D microsteps (4 at D = 8, 2 at D >= 11)."""
    n = 256
    w = WR.make(name, n)
    sim = w.make_simulator()
    gpu = sim.forward_simulate_robots(w.starts, w.targets, True, capi.NOISE_PHILOX)
    ref = parity.make_oracle(w).forward_simulate(w.starts, w.targets, True, capi.NOISE_PHILOX)
    assert np.array_equal(gpu.n_microsteps, ref["n_microsteps"])
    assert np.array_equal(gpu.flags & parity.SEMANTIC_FLAGS, ref["flags"] & parity.SEMANTIC_FLAGS)
    assert np.max(np.abs(gpu.configs - ref["cfg"])) < 1e-9
    assert not gpu.did_contact.any()
    sim.close()


# ------------------------------------------------------------------------------------------------
# layout independence
# ------------------------------------------------------------------------------------------------
def test_many_points_robot_gets_fewer_warps_per_cta():
    w = WR.many_points(4)
    assert w.robot.points.shape[0] >= 1024
    sim = w.make_simulator()
    assert _threads_per_cta(sim) < 24 * 32, sim.kernel_info
    sim.close()


@pytest.mark.parametrize("name", ["dual_arm_table", "tree_fixed_table", "chain8_table", "dual_arm_folded"])
def test_records_do_not_depend_on_warps_per_cta_or_call_split(name, monkeypatch):
    n = 600
    w = WR.make(name, n)
    ref = None
    for wpb in (None, "1", "3"):
        if wpb is None:
            monkeypatch.delenv("FKS_WARPS_PER_BLOCK", raising=False)
        else:
            monkeypatch.setenv("FKS_WARPS_PER_BLOCK", wpb)
        sim = w.make_simulator()
        if wpb is not None:
            assert _threads_per_cta(sim) == 32 * int(wpb), sim.kernel_info
        rec = sim.forward_simulate_robots(w.starts, w.targets, True, capi.NOISE_PHILOX).records.copy()
        if ref is None:
            ref = rec
            # the same batch in three calls, each keyed by its first particle id
            parts = [sim.forward_simulate_robots(w.starts[a:b], w.targets, True, capi.NOISE_PHILOX, first_particle_id=a).records
                     for a, b in ((0, 100), (100, 357), (357, n))]
            assert np.concatenate(parts).tobytes() == ref.tobytes()
        else:
            assert rec.tobytes() == ref.tobytes(), wpb
        sim.close()
    assert ((ref["flags"] & capi.FLAG_DID_CONTACT) != 0).all()


@pytest.mark.parametrize("name", ["dual_arm_table", "many_points"])
def test_records_do_not_depend_on_launch_stream_at_eight_particles_per_context(name):
    """At least 8 particles per pool context (2 per warp), so every context is parked and loaded again many times per
    launch (test_gpu_context_swap.py), with the context and tall-system ranges of these layouts."""
    probe = WR.dual_arm(4) if name == "dual_arm_table" else WR.many_points(4)
    sim0 = probe.make_simulator()
    contexts = 2 * (_threads_per_cta(sim0) // 32) * _persistent_grid(sim0)
    sim0.close()
    n = 8 * contexts
    w = WR.dual_arm(n) if name == "dual_arm_table" else WR.many_points(n)
    sim = w.make_simulator()
    ref = sim.forward_simulate_robots(w.starts, w.targets, True, capi.NOISE_PHILOX).records.copy()
    assert sim.forward_simulate_robots(w.starts, w.targets, True, capi.NOISE_PHILOX).records.tobytes() == ref.tobytes()
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
    # calls of at most one particle per SM: no context ever moves to another warp
    for a in (0, 148 * 7):
        part = sim.forward_simulate_robots(w.starts[a:a + 148], w.targets, True, capi.NOISE_PHILOX, first_particle_id=a).records
        assert part.tobytes() == ref[a:a + 148].tobytes(), a
    sim.close()


# ------------------------------------------------------------------------------------------------
# consumers of a batch at D = 15
# ------------------------------------------------------------------------------------------------
def test_end_state_consumers_at_fifteen_dof():
    n = 1024
    w = WR.dual_arm(n)
    sim = w.make_simulator()
    st = torch.cuda.current_stream()
    dr = torch.empty(n * sim.result_stride, dtype=torch.uint8, device="cuda")
    sim.forward_simulate_device(torch.from_numpy(w.starts).cuda(), torch.from_numpy(w.targets).cuda(), n, 1, dr, True, capi.NOISE_PHILOX,
                                stream=st.cuda_stream)
    torch.cuda.synchronize()
    rec = dr.cpu().numpy().view(sim.dtype)
    # pairwise distances against the oracle's ComputeConfigurationDistanceTo
    ids = np.arange(0, n, 3, dtype=np.uint32)[:300]
    m = len(ids)
    out = torch.empty(m, m, dtype=torch.float64, device="cuda")
    sim.end_states_pairwise_distance(dr, m, out, torch.from_numpy(ids.view(np.int32)).cuda(), stream=st.cuda_stream)
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    want = parity.make_oracle(w).pairwise_config_distance(rec["cfg"][ids])
    assert np.allclose(got, want, rtol=4e-15, atol=0.0), float(np.max(np.abs(got - want)))
    # clustering of two segments of those records against the reference fed the GPU matrices
    segs = [ids[:170], ids[170:]]  # one segment past the shared-memory limit (160), one below it
    mats = []
    for s in segs:
        o = torch.empty(len(s), len(s), dtype=torch.float64, device="cuda")
        sim.end_states_pairwise_distance(dr, len(s), o, torch.from_numpy(s.view(np.int32)).cuda(), stream=st.cuda_stream)
        torch.cuda.synchronize()
        mats.append(o.cpu().numpy())
    offsets = np.array([0, len(segs[0]), m], dtype=np.uint64)
    vals = np.concatenate([x[np.triu_indices(len(x), 1)] for x in mats])
    for lk in (CR.LINKAGE_SINGLE, CR.LINKAGE_COMPLETE):
        t = float(np.quantile(vals, 0.05 if lk == CR.LINKAGE_SINGLE else 0.3, method="lower"))
        labels = torch.full((m,), -1, dtype=torch.int32, device="cuda")
        counts = sim.end_states_cluster(dr, offsets, labels, t, lk, torch.from_numpy(ids.view(np.int32)).cuda(), stream=st.cuda_stream)
        torch.cuda.synchronize()
        want_labels, want_counts = CR.cluster_segments(mats, lk, t)
        assert np.array_equal(counts, want_counts) and np.array_equal(labels.cpu().numpy().view(np.uint32), want_labels)
        assert 1 < want_counts.sum() < m
    # three legs in one call equal the chain of single calls
    legs = np.stack([w.targets[0], w.starts[0], w.targets[0] + 0.05])
    s0 = w.starts[:256]
    seq = sim.forward_simulate_sequence(s0, legs, True, capi.NOISE_PHILOX, first_particle_id=9)
    at = s0
    for k in range(3):
        single = sim.forward_simulate_robots(at, legs[k].reshape(1, -1), True, capi.NOISE_PHILOX, first_particle_id=9 + k * 256).records
        assert seq.records[k].tobytes() == single.tobytes(), k
        at = np.ascontiguousarray(single["cfg"])
    sim.close()


# ------------------------------------------------------------------------------------------------
# argument errors
# ------------------------------------------------------------------------------------------------
def _refused(robot, match):
    with pytest.raises(capi.FksError, match=match):
        S.GpuRobot(robot, 0)


def test_robot_descriptions_past_the_limits_are_refused():
    # 16 DoF: the solver keeps D + 1 <= 16 columns (the oracle takes this description: test_oracle_wide_robots.py)
    _refused(WR.sixteen_dof_robot(), "count out of range")
    # 17 links (16 joints, one of them fixed: 15 DoF)
    r = WR.chain_robot(16)
    r.joints[5] = dict(r.joints[5], type=WR.FIXED, lower=0.0, upper=0.0)
    r.axes, r.n_dof = r.axes[:15], 15
    assert r.n_links == 17
    _refused(r, "count out of range")
    # a link no joint leads to
    r = WR.chain_robot(15)
    r.joints, r.axes, r.n_dof = r.joints[:-1], r.axes[:-1], 14
    _refused(r, "needs a parent joint")
    # a joint listed before the joint that places its parent link
    r = WR.dual_arm_robot()
    r.joints[1], r.joints[3] = r.joints[3], r.joints[1]
    _refused(r, "kinematic order")
    # the robots of these tests are accepted
    for name in ("chain15", "dual_arm", "tree_fixed", "many_points"):
        S.GpuRobot(WR.ROBOTS[name](), 0).close()
