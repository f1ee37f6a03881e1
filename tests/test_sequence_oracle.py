"""Sequence calls without a GPU: the reference chain on the CPU oracle, the merged per-particle tapes it produces, the
Python wrappers' input shapes, and the C++ example that compares a sequence with a chain of single calls."""
import os
import subprocess

import numpy as np
import pytest

from fast_kinematic_simulator_b200 import capi, workloads as W
from fast_kinematic_simulator_b200.simulator import sequence_inputs
from oracle import oracle_binding as OB

import parity
import sequence_chain as SC

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _tape(per_particle_draws, per_particle_records, n_dof):
    """tape of n particles from lists of draws / decision records (lists of word lists)"""
    draws = np.concatenate([np.asarray(d, dtype=np.float64) for d in per_particle_draws])
    offs = np.concatenate([[0], np.cumsum([len(d) for d in per_particle_draws])]).astype(np.uint64)
    recs = [np.asarray(r, dtype=np.uint64).reshape(-1, 2 + n_dof) for r in per_particle_records]
    dec = np.concatenate([r.reshape(-1) for r in recs])
    dec_offs = np.concatenate([[0], np.cumsum([len(r) for r in recs])]).astype(np.uint64)
    return draws, offs, dec, dec_offs


def test_merge_tapes_concatenates_each_particles_legs():
    n_dof = 2

    def rec(rank, rows, value):
        return [rank | (rows << 16), 0x10, np.float64(value).view(np.uint64), np.float64(-value).view(np.uint64)]

    leg0 = _tape([[1.0, 2.0], [], [3.0]], [[rec(2, 6, 0.5)], [], [rec(1, 3, 1.5), rec(2, 9, 2.5)]], n_dof)
    leg1 = _tape([[4.0], [5.0, 6.0, 7.0], []], [[], [rec(2, 12, 3.5)], [rec(1, 6, 4.5)]], n_dof)
    draws, offs, dec, dec_offs = SC.merge_tapes([leg0, leg1], 3, n_dof)
    assert offs.tolist() == [0, 3, 6, 7]
    assert draws.tolist() == [1.0, 2.0, 4.0, 5.0, 6.0, 7.0, 3.0]
    assert dec_offs.tolist() == [0, 1, 2, 5]
    d = OB.decision_records((draws, offs, dec, dec_offs), n_dof)
    assert d["rank"].tolist() == [2, 2, 1, 2, 1]
    assert d["rows"].tolist() == [6, 12, 3, 9, 6]
    assert d["solution"][:, 0].tolist() == [0.5, 3.5, 1.5, 2.5, 4.5]
    assert d["solution"][:, 1].tolist() == [-0.5, -3.5, -1.5, -2.5, -4.5]


def test_merge_tapes_without_decisions():
    t0 = ([1.0, 2.0, 3.0], np.array([0, 1, 3], dtype=np.uint64))
    t1 = ([4.0, 5.0], np.array([0, 2, 2], dtype=np.uint64))
    draws, offs, dec, dec_offs = SC.merge_tapes([t0, t1], 2, 3)
    assert draws.tolist() == [1.0, 4.0, 5.0, 2.0, 3.0] and offs.tolist() == [0, 3, 5]
    assert dec.size == 0 and dec_offs.tolist() == [0, 0, 0]


def test_sensitivity_propagates_to_later_legs():
    sens = np.array([[0, 1, 0, 0], [0, 0, 4, 0], [2, 0, 0, 0]], dtype=np.uint32)
    out = SC.propagate_sensitivity(sens)
    assert out.tolist() == [[0, 1, 0, 0], [0, 1, 4, 0], [2, 1, 4, 0]]


def test_oracle_chain_is_the_single_calls_chained():
    """run_sequence_with_tape on the CPU oracle: leg k starts where leg k-1 ended (replaying leg k from there with its
    recorded tape reproduces its records); the merged tape holds exactly the per-leg spans."""
    w = W.se2_arena(16)
    starts = w.starts
    legs = np.stack([w.targets[0], w.starts[0], np.array([-1.0, -1.5, 0.4])])
    orc = parity.make_oracle(w)
    rec, tapes, merged, sens = SC.run_sequence_with_tape(orc, starts, legs, True, OB.ORACLE_NOISE_MT19937, 100)
    assert rec.shape == (3, 16) and sens.shape == (3, 16) and len(tapes) == 3
    assert ((rec[0]["flags"] & capi.FLAG_DID_CONTACT) != 0).all()
    at = starts
    for k in range(3):
        ref = parity.make_oracle(w).forward_simulate(at, legs[k], True, capi.NOISE_INJECTED, tapes[k], 100 + 16 * k)
        assert np.array_equal(ref, rec[k]), k
        at = rec[k]["cfg"]
    assert int(merged[1][-1]) == sum(int(t[1][-1]) for t in tapes) and int(merged[1][-1]) > 0
    assert int(merged[3][-1]) == sum(int(t[3][-1]) for t in tapes)
    for i in (0, 7, 15):
        expect = np.concatenate([t[0][int(t[1][i]):int(t[1][i + 1])] for t in tapes])
        assert np.array_equal(merged[0][int(merged[1][i]):int(merged[1][i + 1])], expect)
    assert np.array_equal(sens[1:] & sens[:-1], sens[:-1])  # marks never disappear


def test_sequence_inputs_shapes():
    starts = np.zeros((5, 3))
    s, t = sequence_inputs(starts, np.ones((4, 3)), 3)
    assert s.shape == (5, 3) and t.shape == (4, 1, 3)
    s, t = sequence_inputs(starts.reshape(-1), np.ones((2, 5, 3)), 3)
    assert s.shape == (5, 3) and t.shape == (2, 5, 3) and t.flags["C_CONTIGUOUS"]
    s, t = sequence_inputs(starts, np.ones((2, 5, 3))[:, ::2], 3)
    assert t.shape == (2, 3, 3) and t.flags["C_CONTIGUOUS"]
    with pytest.raises(ValueError):
        sequence_inputs(starts, np.ones((2, 4)), 3)
    with pytest.raises(ValueError):
        sequence_inputs(starts, np.ones(3), 3)
    with pytest.raises(ValueError):
        sequence_inputs(starts, np.ones((1, 2, 5, 3)), 3)


def test_sequence_entry_points_are_declared():
    for name in ("fks_forward_simulate_sequence", "fks_forward_simulate_sequence_device", "fks_multi_forward_simulate_sequence"):
        assert name in capi.EXPORTS and hasattr(capi.lib, name)


def test_sequence_example_compiles_and_fails_loudly_without_a_gpu(tmp_path):
    import torch

    lib = os.path.join(ROOT, "fast_kinematic_simulator_b200")
    exe = str(tmp_path / "fksgpu_example_sequence")
    subprocess.check_call(["/usr/bin/g++", "-std=c++11", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "forward_simulate_sequence.cpp"), "-L" + lib, "-lfksgpu", "-Wl,-rpath," + lib,
                           "-o", exe])
    r = subprocess.run([exe], capture_output=True, text=True)
    if torch.cuda.is_available():
        assert r.returncode == 0 and "ok" in r.stdout, r.stdout
    else:
        assert r.returncode == 3 and "no CUDA device" in r.stdout, r.stdout
