"""The oracle on linked robots past the 7-DoF arm (tests/wide_robots.py): 8 and 15 DoF chains, a dual arm whose joints are
numbered alternately between its branches, a 16-link tree with fixed joints inside its branches.  Kinematics against an
independent numpy model of the tree, and the precondition of the GPU parity bar on these robots."""
import ctypes as C

import numpy as np
import pytest

import parity
import wide_robots as WR
from fast_kinematic_simulator_b200 import capi
from oracle import oracle_binding as OB

SIZES = {name: (r.n_links, len(r.joints), r.n_dof) for name, r in ((n, f()) for n, f in WR.ROBOTS.items())}


def _kinematics(robot, q, link=0, point=(0.0, 0.0, 0.0)):
    """oracle_robot_kinematics -> (L, 3, 4) link transforms, 3 x D Jacobian of `point` (link frame) on `link`, stored cfg"""
    d = robot.to_c()
    L, D = robot.n_links, robot.n_dof
    q = np.ascontiguousarray(q, dtype=np.float64)
    p = np.ascontiguousarray(point, dtype=np.float64)
    T, Jm, cfg = np.zeros(12 * L), np.zeros(3 * D), np.zeros(D)
    assert OB.lib().oracle_robot_kinematics(C.addressof(d), q.ctypes.data, link, p.ctypes.data, T.ctypes.data, Jm.ctypes.data,
                                            cfg.ctypes.data) == 0
    return T.reshape(L, 3, 4), Jm.reshape(3, D), cfg


def pivots_from_second_slot(d):
    """per recorded solve: how many of its first `rank` pivots are columns >= 8"""
    nib = (d["order"][:, None] >> (np.uint64(4) * np.arange(16, dtype=np.uint64))) & np.uint64(0xF)
    return ((nib >= 8) & (np.arange(16)[None, :] < d["rank"][:, None])).sum(axis=1)


def test_robot_sizes():
    assert SIZES["chain8"] == (9, 8, 8)
    assert SIZES["chain15"] == (16, 15, 15)
    assert SIZES["dual_arm"] == SIZES["dual_arm_all_pairs"] == (16, 15, 15)
    assert SIZES["tree_fixed"] == (16, 15, 11)
    assert WR.ROBOTS["many_points"]().points.shape[0] >= 1024
    n_pairs = {name: int((f().allowed == 0).sum()) // 2 for name, f in WR.ROBOTS.items()}
    assert n_pairs["dual_arm"] == 49 and n_pairs["dual_arm_all_pairs"] == 105 and n_pairs["chain15"] == 91
    # the dual arm's joints are not depth-first: the left arm's ancestors are every second joint
    r = WR.dual_arm_robot()
    assert WR.ancestors(r, 14) == {0, 1, 3, 5, 7, 9, 11, 13}
    # the tree: DoF index != joint index past the first fixed joint, and fixed joints have children
    t = WR.tree_robot()
    act = WR.active_joints(t)
    assert act != list(range(t.n_dof))
    fixed_with_children = [i for i, j in enumerate(t.joints) if j["type"] == WR.FIXED and any(k["parent"] == j["child"] for k in t.joints)]
    assert len(fixed_with_children) >= 3


@pytest.mark.parametrize("name", ["chain8", "chain15", "dual_arm", "tree_fixed"])
def test_link_transforms_match_numpy_tree_fk(name):
    robot = WR.ROBOTS[name]()
    rng = np.random.default_rng(5)
    lo = np.array([j["lower"] for j in robot.joints if j["type"] != WR.FIXED])
    hi = np.array([j["upper"] for j in robot.joints if j["type"] != WR.FIXED])
    for _ in range(20):
        q = rng.uniform(lo - 0.2, hi + 0.2)  # past the limits too: clamped (continuous joints wrap)
        T, _, cfg = _kinematics(robot, q)
        want = WR.fk(robot, q)[:, :3]
        assert np.max(np.abs(T - want)) < 1e-12, name
        assert np.allclose(cfg, [v for v, j in zip(WR.joint_values(robot, q), robot.joints) if j["type"] != WR.FIXED], rtol=0, atol=1e-15)


@pytest.mark.parametrize("name", ["chain8", "chain15", "dual_arm", "tree_fixed"])
def test_point_jacobian_against_central_differences_and_ancestor_mask(name):
    robot = WR.ROBOTS[name]()
    rng = np.random.default_rng(7)
    act = WR.active_joints(robot)
    for _ in range(3):
        q = rng.uniform(-1.2, 1.2, robot.n_dof)
        # prismatic joints inside their limits: the clamp has no derivative
        q[[a for a, ji in enumerate(act) if robot.joints[ji]["type"] == WR.PRISMATIC]] = 0.03
        for link in range(robot.n_links):
            p = robot.points[robot.point_link == link][5]
            _, Jm, _ = _kinematics(robot, q, link, p)

            def pos(qq):
                T = WR.fk(robot, qq)[link]
                return T[:3, :3] @ p + T[:3, 3]

            h = 1e-6
            num = np.stack([(pos(q + h * e) - pos(q - h * e)) / (2 * h) for e in np.eye(robot.n_dof)], axis=1)
            assert np.max(np.abs(Jm - num)) < 1e-8, (name, link)
            anc = WR.ancestors(robot, link)
            for a, ji in enumerate(act):
                if ji not in anc:
                    assert np.all(Jm[:, a] == 0.0), (name, link, a)  # exactly zero, not small
                elif robot.joints[ji]["type"] == WR.PRISMATIC:
                    # a prismatic column is the joint axis in the world frame
                    jd = robot.joints[ji]
                    R = (WR.fk(robot, q)[jd["parent"]] @ np.vstack([np.asarray(jd["transform"]).reshape(3, 4), [0, 0, 0, 1]]))[:3, :3]
                    assert np.allclose(Jm[:, a], R @ np.asarray(jd["axis"]), rtol=0, atol=1e-15)


def test_prismatic_and_fixed_joints_are_placed_like_the_numpy_model():
    t = WR.tree_robot()
    q = np.zeros(11)
    base, _, _ = _kinematics(t, q)
    for lift in (0.0, 0.1, 0.3, 0.5):  # 0.5 is past the upper limit 0.3
        q[0] = lift
        T, _, cfg = _kinematics(t, q)
        assert cfg[0] == min(lift, 0.3)
        assert np.allclose(T[1:, :, 3] - base[1:, :, 3], [0.0, 0.0, min(lift, 0.3)], rtol=0, atol=1e-15)
        assert np.array_equal(T[0], base[0])
    # a fixed joint's child is the parent times the joint transform, whatever the configuration
    rng = np.random.default_rng(9)
    for _ in range(5):
        q = rng.uniform(-1.0, 1.0, 11)
        q[0] = 0.1
        T, _, _ = _kinematics(t, q)
        for j in t.joints:
            if j["type"] == WR.FIXED:
                Tp = np.vstack([T[j["parent"]], [0, 0, 0, 1]])
                Jt = np.vstack([np.asarray(j["transform"]).reshape(3, 4), [0, 0, 0, 1]])
                assert np.max(np.abs(T[j["child"]] - (Tp @ Jt)[:3])) < 1e-15
    # the chain's prismatic joint (DoF 2) moves every later link along joint 2's axis
    c = WR.chain_robot(8)
    q = np.full(8, 0.3)
    q[2] = 0.0
    T0, _, _ = _kinematics(c, q)
    q[2] = 0.07
    T1, _, _ = _kinematics(c, q)
    axis = T0[3][:, 2]
    assert np.allclose(T1[3:, :, 3] - T0[3:, :, 3], 0.07 * axis, rtol=0, atol=1e-14)
    assert np.array_equal(T1[:3], T0[:3])


@pytest.mark.parametrize("name", list(WR.CONTACT))
def test_contact_workloads_are_insensitive_with_ill_conditioned_solves_injected(name):
    """The precondition of the GPU parity bar at these shapes (test_gpu_wide_robots.py): with the decision tape and the
    solution of every solve whose condition estimate exceeds 100 injected, the oracle names no reason for any particle of
    the batch to differ -- no ill-conditioned solve, threshold or rank decision left to amplify round-off.  The only reason
    tolerated is a grid coordinate within 1e-9 of a cell boundary (a few particles in a thousand, at random), which a
    last-bit difference flips with a probability of about 1e-7.  Also checks that each workload runs what it claims."""
    n = 1024
    w = WR.make(name, n)
    orc = parity.make_oracle(w)
    OB.lib().oracle_set_decision_cond_limit(orc._h, 100.0)
    ref, tape, sens = OB.run_with_tape(orc, w.starts, w.targets, True)
    left = sens & ~np.uint32(OB.SENS_COVERED_BY_DECISION_TAPE)
    reasons = {OB.SENS_NAMES[b] for b in range(len(OB.SENS_NAMES)) for s in np.unique(left) if (int(s) >> b) & 1}
    assert reasons <= {"cell_boundary"}, reasons
    assert (left != 0).sum() <= 0.015 * n, (left != 0).sum()
    d = OB.decision_records(tape, w.robot.n_dof)
    assert ((ref["flags"] & capi.FLAG_DID_CONTACT) != 0).all()
    assert ((d["flags"] & OB.DECISION_ROUNDOFF_PIVOT) != 0).sum() > 1000
    assert ((d["flags"] & OB.DECISION_OVERRIDE_SOLUTION) != 0).sum() > 1000
    if w.robot.n_dof >= 9:  # pivots taken from the solver's second column slot (columns 8 ..) occur
        assert (pivots_from_second_slot(d) > 0).sum() > 100
    if name == "dual_arm_folded":
        stats = dict(zip(capi.STAT_NAMES, orc.statistics().tolist()))
        assert stats["unsuccessful_self_collision_resolves"] > 0 and (sens & OB.SENS_SELF_COLLISION).any()


@pytest.mark.parametrize("name", list(WR.FREE))
def test_free_workloads_touch_nothing(name):
    w = WR.make(name, 128)
    ref = parity.make_oracle(w).forward_simulate(w.starts, w.targets, True, OB.ORACLE_NOISE_MT19937)
    assert not ((ref["flags"] & capi.FLAG_DID_CONTACT) != 0).any()
    assert (ref["n_microsteps"] > 0).all()


def test_oracle_accepts_sixteen_dof():
    """The description with 16 DoF that the product refuses (its solver keeps D + 1 <= 16 columns) is one the oracle's model
    takes: the limit is the product's own."""
    r = WR.sixteen_dof_robot()
    assert (r.n_links, len(r.joints), r.n_dof) == (16, 16, 16)
    w = WR.chain(15, 4)
    orc = OB.OracleSimulator(w.environment().desc, r.to_c(), capi.default_solver_params())
    assert orc.stride == 16
