"""End-state records on the device for the tests of the calls that consume them (partition, pairwise distances, clustering,
groups, nearest configurations): simulated batches, records of chosen configurations, and the GPU's own pairwise matrices."""
import numpy as np
import torch

from fast_kinematic_simulator_b200 import capi, workloads as W


def stream():
    return torch.cuda.current_stream().cuda_stream


def u32(a):
    """a device int32 tensor holding the uint32 values of a"""
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint32).view(np.int32)).cuda()


def simulated(name, n):
    """(workload, simulator, device records, host copy of the records) of one Philox batch of n particles of a workload"""
    w = W.make(name, n_particles=n)
    sim = w.make_simulator()
    dr = torch.empty(n * sim.result_stride, dtype=torch.uint8, device="cuda")
    sim.forward_simulate_device(torch.from_numpy(w.starts).cuda(), torch.from_numpy(w.targets).cuda(), n, w.targets.shape[0], dr, True,
                                capi.NOISE_PHILOX, stream=stream())
    torch.cuda.synchronize()
    return w, sim, dr, dr.cpu().numpy().view(sim.dtype)


def records(sim, cfg, contact=None):
    """(device buffer, host array) of records of sim's layout with configurations cfg and, when given, these contact flags"""
    rec = np.zeros(len(cfg), dtype=sim.dtype)
    rec["cfg"] = cfg
    if contact is not None:
        rec["flags"] = np.where(contact, capi.FLAG_DID_CONTACT, 0)
    return torch.from_numpy(rec.view(np.uint8).copy()).cuda(), rec


def synthetic_se2(cfg, contact=None):
    """SE(2) records written straight into a device buffer: (simulator, device records, host records)"""
    sim = W.make("se2_arena", n_particles=4).make_simulator()
    dr, rec = records(sim, cfg, contact)
    return sim, dr, rec


def gpu_matrix(sim, dr, ids):
    """fks_end_states_pairwise_distance over the records ids, on the host"""
    m = len(ids)
    if m == 0:
        return np.zeros((0, 0))
    out = torch.empty(m, m, dtype=torch.float64, device="cuda")
    sim.end_states_pairwise_distance(dr, m, out, u32(ids), stream=stream())
    torch.cuda.synchronize()
    return out.cpu().numpy()
