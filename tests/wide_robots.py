"""Linked robots past the 7-DoF arm, up to the C ABI's limits (16 links, 15 DoF, trees rooted at link 0), for the parity
tests.  Each builder returns a `Workload`, so `parity.run_parity` takes it unchanged; they live beside the other parity
helpers rather than in `workloads.py`, so the benchmark and its workload table do not change.

- `chain(D)`: a serial chain of D + 1 links (revolute, one prismatic, a continuous last joint); pairs more than two links
  apart may not collide.
- `dual_arm`: a waist joint and two 7-DoF arms (16 links, 15 joints, 15 DoF).  Joints and links are numbered alternately
  between the arms, so the order is kinematic but not depth-first and a link's ancestor joints are not a contiguous range.
- `tree_fixed`: 16 links that branch at two levels, fixed joints in the middle of branches and a prismatic lift (11 DoF:
  a DoF index is not its joint index).

`fk` is an independent numpy model of the tree: T_child = T_parent * joint transform * motion(value), the joints in the
order given."""
import numpy as np

from fast_kinematic_simulator_b200 import capi, workloads as W
from fast_kinematic_simulator_b200.robots import RobotDescription, make_transform

RES = 0.04
BASE_OFFSET = np.array([0.011, 0.007, 0.013])  # keeps the bases off the voxel lattice
REVOLUTE, PRISMATIC, FIXED, CONTINUOUS = capi.JOINT_REVOLUTE, capi.JOINT_PRISMATIC, capi.JOINT_FIXED, capi.JOINT_CONTINUOUS
Z, Y, X = (0.0, 0.0, 1.0), (0.0, 1.0, 0.0), (1.0, 0.0, 0.0)


def link_points(length, rings=3, radius=0.04):
    """`rings` rings of 8 points around the link's z axis, between 10 % and 90 % of its length."""
    return np.array([(radius * np.cos(2 * np.pi * k / 8), radius * np.sin(2 * np.pi * k / 8), z)
                     for z in np.linspace(0.1 * length, 0.9 * length, rings) for k in range(8)])


def _joint(parent, child, kind, offset, axis, lower=-2.9, upper=2.9, rotation=None):
    return dict(parent=parent, child=child, type=kind, transform=make_transform(offset, rotation), axis=axis, lower=lower, upper=upper)


def _robot(joints, lengths, allowed, base, rings=3):
    L = len(lengths)
    pts = np.concatenate([link_points(lengths[l], rings) for l in range(L)])
    plink = np.repeat(np.arange(L, dtype=np.int32), 8 * rings)
    n_dof = sum(1 for j in joints if j["type"] != FIXED)
    axes = [W._axis(1.0, kp=2.0, prop=0.1, minn=0.005) for _ in range(n_dof)]
    return RobotDescription(capi.ROBOT_LINKED, pts, plink, axes, n_links=L, joints=joints, base_transform=make_transform(tuple(base)),
                            allowed_self_collision=allowed)


def _allowed_beyond(L, gap):
    """every pair of links whose indices differ by more than `gap` is disallowed"""
    i = np.arange(L)
    return (np.abs(i[:, None] - i[None, :]) <= gap).astype(np.uint8)


# ------------------------------------------------------------------------------------------------
# numpy model
# ------------------------------------------------------------------------------------------------
_rot = W._rot


def joint_values(robot, q):
    """per joint: the value its motion uses (continuous wrapped, others clamped, fixed 0 clamped)"""
    vals, a = [], 0
    for j in robot.joints:
        if j["type"] == FIXED:
            vals.append(min(max(0.0, j["lower"]), j["upper"]))
            continue
        v = float(q[a])
        a += 1
        if j["type"] == CONTINUOUS:
            v = np.arctan2(np.sin(v), np.cos(v))
        else:
            v = min(max(v, j["lower"]), j["upper"])
        vals.append(v)
    return vals


def fk(robot, q):
    """(L, 4, 4) link transforms"""
    T = np.zeros((robot.n_links, 4, 4))
    T[0] = np.eye(4)
    T[0][:3] = robot.base.reshape(3, 4)
    for j, v in zip(robot.joints, joint_values(robot, q)):
        Jt = np.eye(4)
        Jt[:3] = np.asarray(j["transform"]).reshape(3, 4)
        M = np.eye(4)
        if j["type"] in (REVOLUTE, CONTINUOUS):
            M[:3, :3] = _rot(j["axis"], v)
        elif j["type"] == PRISMATIC:
            M[:3, 3] = np.asarray(j["axis"]) * v
        T[j["child"]] = T[j["parent"]] @ Jt @ M
    return T


def ancestors(robot, link):
    """joint indices on the path from the root to `link`"""
    parent_joint = {j["child"]: i for i, j in enumerate(robot.joints)}
    out = set()
    while link in parent_joint:
        i = parent_joint[link]
        out.add(i)
        link = robot.joints[i]["parent"]
    return out


def active_joints(robot):
    """DoF index -> joint index"""
    return [i for i, j in enumerate(robot.joints) if j["type"] != FIXED]


# ------------------------------------------------------------------------------------------------
# robots
# ------------------------------------------------------------------------------------------------
def chain_robot(D, rings=3):
    """Serial chain, L = D + 1.  Joint 0 turns about z, joint 2 is prismatic along the link, the last joint is continuous,
    the others are revolute about z and y in turn; links shorten with D so the reach stays about the 7-DoF arm's."""
    L = D + 1
    ell = 1.81 / D
    joints = []
    for j in range(D):
        offset = (0.0, 0.0, ell if j > 0 else 0.3)
        if j == 2:
            joints.append(_joint(j, j + 1, PRISMATIC, offset, Z, -0.05, 0.1))
        elif j == D - 1:
            joints.append(_joint(j, j + 1, CONTINUOUS, offset, Z, -np.pi, np.pi))
        else:
            joints.append(_joint(j, j + 1, REVOLUTE, offset, Z if j % 2 == 0 else Y))
    lengths = [0.3] + [ell] * D
    return _robot(joints, lengths, _allowed_beyond(L, 2), BASE_OFFSET + (0.0, 0.0, W.ARM_BASE_Z - 0.3), rings)


SHOULDER = 0.25


def dual_arm_robot(all_pairs=False, rings=3):
    """Waist (link 0 -> 1) and two 7-DoF arms on shoulders at y = +-0.25.  Arm joint k of the left arm is joint 1 + 2k with
    child link 2 + 2k, of the right arm joint 2 + 2k with child link 3 + 2k.  Cross-arm pairs (49) may not collide; with
    `all_pairs` no two links without a joint between them may (105 pairs)."""
    L = 16
    joints = [_joint(0, 1, REVOLUTE, (0.0, 0.0, 0.3), Z)]
    for k in range(7):
        for side, y in ((0, SHOULDER), (1, -SHOULDER)):
            child = 2 + 2 * k + side
            parent = 1 if k == 0 else child - 2
            offset = (0.0, y, 0.3) if k == 0 else (0.0, 0.0, W.ARM_LINK_LENGTH)
            joints.append(_joint(parent, child, CONTINUOUS if k == 6 else REVOLUTE, offset, Z if k % 2 == 0 else Y,
                                 -np.pi if k == 6 else -2.9, np.pi if k == 6 else 2.9))
    side = np.array([-1, -1] + [l % 2 for l in range(2, L)])
    allowed = np.ones((L, L), np.uint8)
    cross = (side[:, None] >= 0) & (side[None, :] >= 0) & (side[:, None] != side[None, :])
    allowed[cross] = 0
    if all_pairs:
        allowed[:] = 0
        np.fill_diagonal(allowed, 1)
        for j in joints:
            allowed[j["parent"], j["child"]] = allowed[j["child"], j["parent"]] = 1
    return _robot(joints, [0.3] * L, allowed, BASE_OFFSET + (0.0, 0.0, 0.3), rings)


def tree_robot(rings=3):
    """16 links, 15 joints, 11 DoF.  Link 0 -> 1 prismatic lift, 1 -> 2 waist; branch B from link 2: y, z, FIXED (tilted),
    y, continuous z; branch A from link 2: y, FIXED, then two sub-branches from A's fixed link: (y, FIXED, y) and
    (z, y, FIXED).  Joints listed breadth-first across the branches."""
    tilt = _rot(Y, 0.3)
    spec = [  # name, parent name, type, offset, axis, rotation
        ("lift", "base", PRISMATIC, (0.0, 0.0, 0.1), Z, None),
        ("waist", "lift", REVOLUTE, (0.0, 0.0, 0.2), Z, None),
        ("B1", "waist", REVOLUTE, (0.0, -0.2, 0.2), Y, None),
        ("A1", "waist", REVOLUTE, (0.0, 0.2, 0.2), Y, None),
        ("B2", "B1", REVOLUTE, (0.0, 0.0, 0.25), Z, None),
        ("A2", "A1", FIXED, (0.0, 0.0, 0.25), Z, tilt),
        ("B3", "B2", FIXED, (0.0, 0.0, 0.25), Z, _rot(X, 0.2)),
        ("Aa1", "A2", REVOLUTE, (0.0, 0.1, 0.2), Y, None),
        ("Ab1", "A2", REVOLUTE, (0.0, -0.1, 0.2), Z, None),
        ("B4", "B3", REVOLUTE, (0.0, 0.0, 0.2), Y, None),
        ("Aa2", "Aa1", FIXED, (0.0, 0.0, 0.2), Z, _rot(Y, -0.4)),
        ("Ab2", "Ab1", REVOLUTE, (0.0, 0.0, 0.2), Y, None),
        ("B5", "B4", CONTINUOUS, (0.0, 0.0, 0.25), Z, None),
        ("Aa3", "Aa2", REVOLUTE, (0.0, 0.0, 0.2), Y, None),
        ("Ab3", "Ab2", FIXED, (0.0, 0.0, 0.2), Z, _rot(Z, 0.5)),
    ]
    link = {"base": 0}
    joints = []
    for name, parent, kind, offset, axis, rot in spec:
        link[name] = len(link)
        lo, hi = {PRISMATIC: (0.0, 0.3), CONTINUOUS: (-np.pi, np.pi), FIXED: (0.0, 0.0)}.get(kind, (-2.9, 2.9))
        joints.append(_joint(link[parent], link[name], kind, offset, axis, lo, hi, rot))
    lengths = [0.1, 0.2, 0.2, 0.25, 0.25, 0.25, 0.2, 0.2, 0.2, 0.25, 0.2, 0.2, 0.25, 0.2, 0.2, 0.2]
    L = len(lengths)
    allowed = np.zeros((L, L), np.uint8)
    for a in range(L):
        for b in range(L):
            # links that share a joint or a parent may touch
            allowed[a, b] = a == b or any({j["parent"], j["child"]} == {a, b} for j in joints) or \
                any(j["child"] == a and k["child"] == b and j["parent"] == k["parent"] for j in joints for k in joints)
    return _robot(joints, lengths, allowed, BASE_OFFSET + (0.0, 0.0, 0.3), rings)


def sixteen_dof_robot():
    """`chain_robot(15)` plus a sixteenth active joint that drives the last link once more: 16 DoF on 16 links"""
    r = chain_robot(15)
    r.joints.append(_joint(14, 15, REVOLUTE, (0.0, 0.0, 1.81 / 15), Y))
    r.axes.append(dict(r.axes[-1]))
    r.n_dof = 16
    return r


# ------------------------------------------------------------------------------------------------
# workloads (the arm's room with its table at resolution 0.04)
# ------------------------------------------------------------------------------------------------
def _workload(name, robot, start, target, n, sigma, description, seed=1003):
    rng = np.random.Generator(np.random.MT19937(seed))
    start = np.asarray(start, dtype=np.float64)
    starts = start[None, :] + rng.normal(0.0, sigma, (n, len(start)))
    return W.Workload(name, capi.ROBOT_LINKED, W.arm_room_obstacles(), RES, robot, starts, np.asarray(target, dtype=np.float64).reshape(1, -1),
                      description)


def _spread(arm7, D):
    """the 7-DoF arm's configuration stretched over a D-joint chain: the sum of its y bends split evenly over the chain's y
    joints, its first and last values on the chain's first and last joints"""
    q = np.zeros(D)
    ys = [j for j in range(1, D - 1) if j % 2 == 1]
    q[ys] = (arm7[1] + arm7[3] + arm7[5]) / len(ys)
    q[0], q[D - 1] = arm7[0], arm7[6]
    return q


def _interleave(waist, left, right):
    q = [waist]
    for k in range(7):
        q += [left[k], right[k]]
    return np.array(q)


# scale factors of the arm's start and target over the chain: the last link's lowest point 7 cm above the table top at the
# start, 12 cm below it at the target (found by bisection on the numpy model)
_CHAIN_TABLE = {8: (0.8436, 0.7786), 15: (1.0112, 0.9441)}
ARM_FREE_START = np.array([0.0, 0.5, 0.0, 0.9, 0.0, 0.5, 0.0])
ARM_FREE_TARGET = np.array([0.4, 0.6, 0.3, 1.0, 0.2, 0.6, 0.5])


def chain(D, n_particles=1024, scenario="table", rings=3):
    """`table`: the last link is driven into the table; `free`: a raised chain moves through free space."""
    robot = chain_robot(D, rings)
    if scenario == "table":
        s0, s1 = _CHAIN_TABLE[D]
        start, target = s0 * _spread(W.ARM_START, D), s1 * _spread(W.ARM_TARGET, D)
    else:
        start, target = 0.8 * _spread(ARM_FREE_START, D), 0.8 * _spread(ARM_FREE_TARGET, D)
    target[2] = 0.05  # the prismatic joint extends
    return _workload("chain%d_%s" % (D, scenario), robot, start, target, n_particles, 0.02,
                     "%d-DoF serial chain (%d links), %s" % (D, D + 1, scenario))


def dual_arm(n_particles=1024, scenario="table", rings=3):
    """`table`: the left arm does what the 7-DoF arm does in `arm_table`, the right arm mirrors it behind the robot;
    `free`: both arms raised and moving in free space; `folded`: the arms swing towards each other until they cross (every
    non-adjacent pair disallowed, so the crossing links collide)."""
    robot = dual_arm_robot(all_pairs=scenario == "folded", rings=rings)
    if scenario == "table":
        start, target = _interleave(0.0, W.ARM_START, -W.ARM_START), _interleave(0.1, W.ARM_TARGET, -W.ARM_TARGET)
    elif scenario == "free":
        start, target = _interleave(0.0, ARM_FREE_START, -ARM_FREE_START), _interleave(0.3, ARM_FREE_TARGET, -ARM_FREE_TARGET)
    else:
        start, target = _interleave(0.0, *FOLD_START), _interleave(0.0, *FOLD_TARGET)
    return _workload("dual_arm_%s" % scenario, robot, start, target, n_particles, 0.02,
                     "waist + two 7-DoF arms (16 links, 15 DoF, joints interleaved), %s" % scenario)


# both arms reach forward; the left one turns towards -y at the shoulder, the right one towards +y, until their forearms cross
FOLD_START = (np.array([-0.05, 0.7, 0.0, 0.8, 0.0, 0.0, 0.0]), np.array([0.05, 0.7, 0.0, 0.8, 0.0, 0.0, 0.0]))
FOLD_TARGET = (np.array([-0.3, 0.7, 0.0, 0.8, 0.0, 0.0, 0.0]), np.array([0.3, 0.7, 0.0, 0.8, 0.0, 0.0, 0.0]))

# branch B's last link 7 cm above the table at the start, 12 cm below at the target
_TREE_TABLE = (1.1094, 1.2714)


def tree_fixed(n_particles=1024, scenario="table", rings=3):
    """`table`: branch B (DoF 2 and 7) reaches down onto the table while the lift rises; `free`: every joint moves a
    little in free space."""
    robot = tree_robot(rings)
    start, target = np.zeros(11), np.zeros(11)
    if scenario == "table":
        start[[2, 7]], target[[2, 7]] = _TREE_TABLE[0], _TREE_TABLE[1]
        target[0], target[1] = 0.02, 0.1
    else:
        start[:] = [0.05, 0.0, 0.3, -0.3, 0.2, 0.3, 0.2, 0.3, 0.3, 0.0, 0.3]
        target[:] = [0.2, 0.5, 0.5, -0.5, 0.4, 0.5, -0.2, 0.6, 0.5, 2.0, 0.5]
    return _workload("tree_fixed_%s" % scenario, robot, start, target, n_particles, 0.02,
                     "16-link tree, 11 DoF, fixed joints inside branches, prismatic lift, %s" % scenario)


def many_points(n_particles=1024):
    """`dual_arm` in free space with 72 points per link (1 152 points): the simulator gives it fewer warps per CTA"""
    return dual_arm(n_particles, "free", rings=9)


# contact workloads of the parity tests and the sizes they run at
CONTACT = {"chain8_table": lambda n: chain(8, n), "chain15_table": lambda n: chain(15, n), "dual_arm_table": lambda n: dual_arm(n),
           "tree_fixed_table": lambda n: tree_fixed(n), "dual_arm_folded": lambda n: dual_arm(n, "folded")}
FREE = {"chain8_free": lambda n: chain(8, n, "free"), "chain15_free": lambda n: chain(15, n, "free"),
        "dual_arm_free": lambda n: dual_arm(n, "free"), "tree_fixed_free": lambda n: tree_fixed(n, "free")}
ROBOTS = {"chain8": lambda: chain_robot(8), "chain15": lambda: chain_robot(15), "dual_arm": dual_arm_robot,
          "dual_arm_all_pairs": lambda: dual_arm_robot(True), "tree_fixed": tree_robot, "many_points": lambda: dual_arm_robot(rings=9)}


def make(name, n_particles):
    return {**CONTACT, **FREE}[name](n_particles)
