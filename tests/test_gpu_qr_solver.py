"""The device's contact solver (fks_debug_qr_solve = the colpiv_qr_lanes the simulate kernel calls) against the oracle's
restatement of Eigen's ColPivHouseholderQR solve (spcs.hpp:1990-1998) ON THE SAME SYSTEMS: the stacked Jacobians the
oracle met while simulating the BASELINE workloads, plus random and degenerate ones.  The device follows Eigen operation
for operation with unfused arithmetic, so the solutions must be BIT-identical -- including the round-off coin flips of
rank-deficient systems (a kept round-off pivot gives the same garbage on both sides)."""
import numpy as np
import pytest

from fast_kinematic_simulator_b200 import capi, simulator as S, workloads as W
from oracle import oracle_binding as OB

import parity
import wide_robots as WR

pytestmark = pytest.mark.gpu


def _captured(name, n):
    w = WR.make(name, n) if name in WR.CONTACT else W.make(name, n_particles=n)
    orc = parity.make_oracle(w)
    OB.lib().oracle_debug_capture_systems(1 << 20)
    OB.run_with_tape(orc, w.starts, w.targets, True)
    systems = OB.captured_systems()
    OB.lib().oracle_debug_capture_systems(0)
    return systems


@pytest.mark.parametrize("name,n", [("arm_table", 512), ("se3_narrow_passage", 1024), ("se2_arena", 128), ("arm_selfcollision", 64),
                                    ("gantry", 128), ("chain8_table", 256), ("chain15_table", 256), ("dual_arm_table", 256),
                                    ("tree_fixed_table", 256), ("dual_arm_folded", 256)])
def test_device_solver_returns_the_oracles_bits(name, n):
    systems = _captured(name, n)
    assert len(systems) > 500
    x, flags = S.debug_qr_solve(systems)
    ref = np.array([OB.qr_solve_info(A, b)[0] for A, b in systems])
    info = np.array([OB.qr_solve_info(A, b)[3] for A, b in systems])
    same = np.all(x.view(np.uint64) == ref.view(np.uint64), axis=1) | np.all(x == ref, axis=1)  # (-0.0 == 0.0)
    print("%s: %d systems, rows up to %d, %d with a round-off pivot (%d kept), bit-identical %d" % (
        name, len(systems), max(A.shape[0] for A, _ in systems), int((info & 1).sum()), int(((info & 2) != 0).sum()), int(same.sum())))
    assert same.all(), np.nonzero(~same)[0][:10]
    if name == "arm_table" or (name in WR.CONTACT and name != "tree_fixed_table"):
        assert ((info & 2) != 0).sum() > 20  # kept round-off pivots are in the sample, and reproduce
    if name in WR.CONTACT:  # (the tree meets round-off pivots in most solves and keeps almost none)
        assert (info & 1).sum() > 500
    if systems[0][0].shape[1] >= 9:  # D >= 9: pivots from the second column slot are in the sample
        order = np.array([OB.qr_solve_info(A, b)[2] for A, b in systems], dtype=np.uint64)
        assert (((order[:, None] >> (np.uint64(4) * np.arange(4, dtype=np.uint64))) & np.uint64(0xF)) >= 8).any(axis=1).sum() > 20


def _random_and_degenerate(rng, cols, rows_list):
    systems = []
    for rows in rows_list:
        A = rng.normal(size=(rows, cols))
        systems.append((A, rng.normal(size=rows)))
        A2 = A.copy()
        A2[:, -1] = A2[:, 0] * 2.0  # exactly dependent columns
        systems.append((A2, rng.normal(size=rows)))
        A3 = A.copy()
        A3[:, 1] = 0.0  # a structurally zero column (a joint that does not move the point)
        systems.append((A3, rng.normal(size=rows)))
        systems.append((np.zeros((rows, cols)), rng.normal(size=rows)))
        if cols >= 9:
            # the second column slot (columns 8 ..): the first pivot there, a dependent pair across the slots, a zero column
            A4 = A.copy()
            A4[:, cols - 1] *= 8.0
            systems.append((A4, rng.normal(size=rows)))
            A5 = A.copy()
            A5[:, 8] = A5[:, 2] * -3.0
            A5[:, 8] *= 4.0  # and the larger of the pair: the pivot comes from slot 1, its partner's norm is downdated to zero
            systems.append((A5, rng.normal(size=rows)))
            A6 = A.copy()
            A6[:, 8] = 0.0
            A6[:, cols - 1] = 0.0
            systems.append((A6, rng.normal(size=rows)))
            A7 = A.copy()
            A7[:, 9 if cols > 9 else 8] = A7[:, 0] + A7[:, 8 if cols > 9 else 1]  # a dependent triple spanning both slots
            systems.append((A7, rng.normal(size=rows)))
            A8 = A[:, ::-1] * np.geomspace(1.0, 1e-6, cols)[None, ::-1]  # norms growing with the column: pivots from slot 1 first
            systems.append((np.ascontiguousarray(A8), rng.normal(size=rows)))
    return systems


ROWS = (1, 2, 3, 5, 6, 7, 8, 9, 24, 31, 32, 33, 63, 64, 65, 200, 1152)


def test_device_solver_on_random_and_degenerate_systems():
    """Random and degenerate systems.  From cols = 8 on the device keeps a second column per quad (colpiv_qr_lanes<2>,
    the right-hand side at cols = 8); from cols = 9 on, pivots come from that slot too."""
    for cols in (3, 6, 7, 4, 8, 9, 11, 15):
        rng = np.random.default_rng(11 if cols <= 7 else 11 + cols)
        systems = _random_and_degenerate(rng, cols, ROWS)
        x, flags = S.debug_qr_solve(systems)
        ref = np.array([OB.qr_solve_info(A, b)[0] for A, b in systems])
        same = np.all((x.view(np.uint64) == ref.view(np.uint64)) | (x == ref), axis=1)
        assert same.all(), (cols, np.nonzero(~same)[0][:10])
        if cols >= 9:  # the first pivot came from slot 1 in at least two systems per row count
            first = np.array([OB.qr_solve_info(A, b)[2] & 0xF for A, b in systems])
            assert (first >= 8).sum() >= 2 * len(ROWS), cols
