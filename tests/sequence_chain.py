"""Reference side of the sequence-call tests: a sequence of M legs is, by definition, M chained single calls in which leg k
starts from leg k-1's end states and uses the particle ids first_particle_id + k * n.  These helpers run that chain on the CPU
oracle (recording its noise and decision tapes) and turn the per-leg tapes into the one-span-per-particle tape a sequence
call consumes (include/fksgpu.h, fks_forward_simulate_sequence)."""
import numpy as np

from oracle import oracle_binding as OB


def leg_targets(targets_seq, stride):
    """(M, n_targets, stride) view of the targets of a sequence ((M, stride) = one target per leg)."""
    t = np.ascontiguousarray(targets_seq, dtype=np.float64)
    return t.reshape(t.shape[0], -1, stride)


def merge_tapes(tapes, n, n_dof):
    """Per-leg tapes (draws, offsets, decision words, decision offsets) of a chain over n particles -> one tape whose span of
    particle i is its leg-0 span, then its leg-1 span, ...  (draws and decision records alike)."""
    words = 2 + n_dof
    draws, dec = [], []
    offs = np.zeros(n + 1, dtype=np.uint64)
    dec_offs = np.zeros(n + 1, dtype=np.uint64)
    for i in range(n):
        d_i, r_i = 0, 0
        for t in tapes:
            lo, hi = int(t[1][i]), int(t[1][i + 1])
            draws.append(np.asarray(t[0], dtype=np.float64)[lo:hi])
            d_i += hi - lo
            if len(t) >= 4:
                lo, hi = int(t[3][i]), int(t[3][i + 1])
                dec.append(np.asarray(t[2], dtype=np.uint64)[lo * words:hi * words])
                r_i += hi - lo
        offs[i + 1] = offs[i] + d_i
        dec_offs[i + 1] = dec_offs[i] + r_i
    draws = np.concatenate(draws) if draws else np.zeros(0)
    dec = np.concatenate(dec) if dec else np.zeros(0, dtype=np.uint64)
    return draws, offs, dec, dec_offs


def propagate_sensitivity(sens):
    """(M, n) per-leg sensitivity masks -> a particle sensitive at leg k stays marked for every later leg: its end state may
    differ there, and every later leg starts from it."""
    return np.bitwise_or.accumulate(np.asarray(sens, dtype=np.uint32), axis=0)


def n_dof_of_stride(stride):
    """actuated axes of a robot from its configuration stride (include/fksgpu.h: SE(2) 3 / 3, SE(3) 12 / 6, linked n / n)"""
    return 6 if stride == 12 else stride


def run_sequence_with_tape(oracle, starts, targets_seq, allow_contacts=True, noise_mode=OB.ORACLE_NOISE_MT19937, first_particle_id=0):
    """The chain of oracle forward_simulate calls a sequence call stands for, with tapes recorded.  Returns
    (records (M, n), per-leg tapes, merged tape, sensitivity (M, n) propagated over the legs)."""
    starts = np.ascontiguousarray(starts, dtype=np.float64).reshape(-1, oracle.stride)
    targets = leg_targets(targets_seq, oracle.stride)
    n, m = starts.shape[0], targets.shape[0]
    records = np.empty((m, n), dtype=oracle.dtype)
    tapes, sens = [], np.zeros((m, n), dtype=np.uint32)
    at = starts
    for k in range(m):
        rec, tape, s = OB.run_with_tape(oracle, at, targets[k], allow_contacts, noise_mode, first_particle_id + k * n)
        records[k], sens[k] = rec, s
        tapes.append(tape)
        at = np.ascontiguousarray(rec["cfg"])
    return records, tapes, merge_tapes(tapes, n, n_dof_of_stride(oracle.stride)), propagate_sensitivity(sens)
