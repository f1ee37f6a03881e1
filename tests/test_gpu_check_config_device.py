"""fks_check_config_collision_device: CheckConfigCollision on device buffers.  The bytes must equal the host call's
(fks_check_config_collision, checked against the oracle in test_gpu_check_config.py) for every input, size and stream, the
call must write nothing past n, and it must be ordered with the simulator's batch calls, which share its scratch slots.
The last test runs one planner extension step (sample, reject colliding samples, nearest tree state, simulate) on the
device and through the host, and requires the same next batch."""
import ctypes as C
import re

import numpy as np
import pytest
import torch

from fast_kinematic_simulator_b200 import capi, workloads as W

import device_records as DR
from test_gpu_check_config import _configs

pytestmark = pytest.mark.gpu

SENTINEL = 0xAB


def _folded(rng, n):
    """folded arms: self collisions only (the arm lifted away from the obstacles)"""
    return np.tile(np.array([0.0, 0.3, 0.0, 2.6, 0.0, 2.6, 0.0]), (n, 1)) + rng.normal(0.0, 0.05, (n, 7))


def host_bytes(sim, cfg, inflation=0.0):
    """the host call's output bytes, as they come from the library"""
    cfg = np.ascontiguousarray(cfg, dtype=np.float64).reshape(-1, sim.config_stride)
    out = np.full(len(cfg), SENTINEL, dtype=np.uint8)
    capi.check(capi.lib.fks_check_config_collision(sim._h, cfg.ctypes.data, len(cfg), float(inflation), out.ctypes.data))
    return out.tobytes()


def device_check(sim, d_cfg, n, inflation=0.0, stream=None):
    """d_out of n + 1 bytes, the last one a sentinel, after an asynchronous device call"""
    d_out = torch.full((n + 1,), SENTINEL, dtype=torch.uint8, device="cuda")
    sim.check_config_collision_device(d_cfg, n, d_out, inflation, stream=DR.stream() if stream is None else stream)
    return d_out


def device_bytes(d_out, n):
    torch.cuda.synchronize()
    h = d_out.cpu().numpy()
    assert h[n] == SENTINEL, "the call wrote past n"
    return h[:n].tobytes()


@pytest.mark.parametrize("name", ["se2_arena", "se3_narrow_passage", "arm_table"])
@pytest.mark.parametrize("inflation", [0.0, 1.5])
def test_same_bytes_as_the_host_call(name, inflation):
    w = W.make(name, n_particles=4)
    rng = np.random.default_rng(11)
    cfg = _configs(w, 2000, rng)
    if name == "arm_table":
        cfg = np.concatenate([cfg, _folded(rng, 64)])
    sim = w.make_simulator()
    got = device_bytes(device_check(sim, torch.from_numpy(cfg).cuda(), len(cfg), inflation), len(cfg))
    assert got == host_bytes(sim, cfg, inflation)
    flags = np.frombuffer(got, np.uint8)
    assert 0.02 < flags[:2000].mean() < 0.999  # the sample mixes free and colliding configurations
    if name == "arm_table":
        assert flags[2000:].any()  # self collisions of the folded arms
    sim.close()


def _warps_of_a_full_grid(sim):
    """warps of check_config_kernel's largest grid: the persistent grid of full CTAs (fks_sim_kernel_info)"""
    info = sim.kernel_info
    threads = int(re.search(r"(\d+) threads/CTA", info).group(1))
    grid = int(re.search(r"persistent grid (\d+)", info).group(1))
    return grid * threads // 32


def test_sizes_launch_counts_and_nothing_written_past_n():
    w = W.arm_table(4)
    sim = w.make_simulator()
    rng = np.random.default_rng(3)
    big = 1 << 20
    assert big > _warps_of_a_full_grid(sim)  # the grid-stride loop runs more than once
    cfg = np.concatenate([_configs(w, big - 256, rng), _folded(rng, 256)])
    d_cfg = torch.from_numpy(cfg).cuda()
    for n in (1, 31, 33, big):
        before = sim.launch_count
        d_out = device_check(sim, d_cfg, n, 0.5)
        assert sim.launch_count == before + 1
        assert device_bytes(d_out, n) == host_bytes(sim, cfg[:n], 0.5), n
    # nothing to check: no launch, nothing written, buffers may be null
    before = sim.launch_count
    d_out = device_check(sim, d_cfg, 0)
    sim.check_config_collision_device(None, 0, None)
    assert sim.launch_count == before
    assert device_bytes(d_out, 0) == b""
    sim.close()


def test_edge_inputs():
    sim = W.se2_arena(4).make_simulator()
    nan = np.nan
    cfg = np.array([[100.0, 100.0, 0.0],   # outside the grid: out-of-bounds points are free (spcs.hpp:943-955)
                    [1.0, 0.0, 0.0],       # centre of the interior box
                    [nan, nan, nan], [nan, 0.0, 0.0], [0.0, nan, 0.0], [0.0, 0.0, nan]])
    got = device_bytes(device_check(sim, torch.from_numpy(cfg).cuda(), len(cfg)), len(cfg))
    assert got == host_bytes(sim, cfg)
    assert got[:2] == b"\x00\x01"
    sim.close()
    w = W.arm_table(4)
    sim = w.make_simulator()
    q = np.concatenate([_folded(np.random.default_rng(4), 4), np.zeros((1, 7))])
    q[0, :] = nan
    q[1, 3] = nan
    q[2, 0] = nan
    got = device_bytes(device_check(sim, torch.from_numpy(q).cuda(), len(q)), len(q))
    assert got == host_bytes(sim, q)
    sim.close()


def test_streams():
    w = W.arm_table(4)
    sim = w.make_simulator()
    rng = np.random.default_rng(5)
    cfg = np.concatenate([_configs(w, 4000, rng), _folded(rng, 96)])
    n = len(cfg)
    want = host_bytes(sim, cfg, 0.5)
    d_cfg = torch.from_numpy(cfg).cuda()
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        a = device_check(sim, d_cfg, n, 0.5, stream=side.cuda_stream)
    assert device_bytes(a, n) == want
    assert device_bytes(device_check(sim, d_cfg, n, 0.5, stream=0), n) == want  # the default stream
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s1):
        a = device_check(sim, d_cfg, n, 0.5, stream=s1.cuda_stream)
    with torch.cuda.stream(s2):
        b = device_check(sim, d_cfg[: n // 2], n // 2, 0.5, stream=s2.cuda_stream)
    assert device_bytes(a, n) == want and device_bytes(b, n // 2) == want[: n // 2]
    sim.close()


def _check_and_simulate(check_first):
    """A device simulate of 16 384 arm particles on stream A and a device check on stream B issued while the other is in
    flight (in either order), then a host check: all three must give their standalone results."""
    n = 16384
    w = W.arm_table(n)
    sim = w.make_simulator()
    rng = np.random.default_rng(8)
    n_dev = (1 << 20) if check_first else (1 << 16)
    cfg = np.concatenate([_configs(w, n_dev - 4096, rng), _folded(rng, 4096)])  # folded arms write self-collision keys
    cfg_host = np.concatenate([_configs(w, 3000, rng), _folded(rng, 1000)])
    ds, dt = torch.from_numpy(w.starts).cuda(), torch.from_numpy(w.targets).cuda()
    d_cfg = torch.from_numpy(cfg).cuda()
    dr = torch.empty(n * sim.result_stride, dtype=torch.uint8, device="cuda")
    sim.forward_simulate_device(ds, dt, n, w.targets.shape[0], dr, True, capi.NOISE_PHILOX, first_particle_id=5, stream=DR.stream())
    torch.cuda.synchronize()
    want_rec = dr.cpu().numpy().tobytes()
    want_dev, want_host = host_bytes(sim, cfg, 0.5), host_bytes(sim, cfg_host, 0.5)
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    dr.fill_(0)
    torch.cuda.synchronize()

    def simulate():
        with torch.cuda.stream(sa):
            sim.forward_simulate_device(ds, dt, n, w.targets.shape[0], dr, True, capi.NOISE_PHILOX, first_particle_id=5,
                                        stream=sa.cuda_stream)

    def check():
        with torch.cuda.stream(sb):
            return device_check(sim, d_cfg, n_dev, 0.5, stream=sb.cuda_stream)

    if check_first:
        d_out = check()
        simulate()
    else:
        simulate()
        d_out = check()
    got_host = host_bytes(sim, cfg_host, 0.5)
    torch.cuda.synchronize()
    assert dr.cpu().numpy().tobytes() == want_rec
    assert device_bytes(d_out, n_dev) == want_dev
    assert got_host == want_host
    sim.close()


def test_a_check_issued_during_a_simulate_waits_for_it():
    _check_and_simulate(check_first=False)


def test_a_simulate_issued_during_a_check_waits_for_it():
    _check_and_simulate(check_first=True)


def test_invalid_arguments():
    sim = W.se2_arena(4).make_simulator()
    d_cfg = torch.zeros(4, 3, dtype=torch.float64, device="cuda")
    d_out = torch.zeros(4, dtype=torch.uint8, device="cuda")

    def refused(s=sim, **kw):
        args = dict(d_configs=d_cfg, n=4, d_out=d_out, inflation_ratio=0.0)
        args.update(kw)
        with pytest.raises(capi.FksError) as e:
            s.check_config_collision_device(**args)
        assert e.value.code == capi.ERR_INVALID_ARGUMENT

    before = sim.launch_count
    refused(d_configs=None)
    refused(d_out=None)
    refused(inflation_ratio=float("nan"))
    assert sim.launch_count == before
    closed = W.se2_arena(4).make_simulator()
    closed.close()
    refused(s=closed)  # a null simulator
    with pytest.raises(capi.FksError) as e:
        capi.check(capi.lib.fks_check_config_collision_device(None, None, 0, 0.0, None, None))
    assert e.value.code == capi.ERR_INVALID_ARGUMENT
    sim.check_config_collision_device(d_cfg, 4, d_out)  # a valid call after the refusals
    torch.cuda.synchronize()
    assert sim.launch_count == before + 1
    sim.close()


def _bounds(w):
    if w.kind == capi.ROBOT_SE2:
        return torch.tensor([-4.5, -4.5, -3.1], dtype=torch.float64, device="cuda"), torch.tensor([4.5, 4.5, 3.1], dtype=torch.float64, device="cuda")
    lo = torch.full((w.robot.n_dof,), -2.8, dtype=torch.float64, device="cuda")
    return lo, -lo


def _extension_step(name, n, n_samples, on_device):
    """One RRT-style extension: a first batch as the tree, seeded samples, the free ones, the nearest tree state to each, and
    the next batch from there towards them.  Returns the next batch's records and the number of free samples."""
    w, sim, dr, _ = DR.simulated(name, n)
    stride = sim.config_stride
    tree = dr.view(torch.float64).view(n, sim.result_stride // 8)[:, :stride]  # the records' configurations, strided
    g = torch.Generator(device="cuda")
    g.manual_seed(1234)
    lo, hi = _bounds(w)
    samples = lo + (hi - lo) * torch.rand(n_samples, stride, generator=g, dtype=torch.float64, device="cuda")
    if on_device:
        collides = torch.empty(n_samples, dtype=torch.uint8, device="cuda")
        sim.check_config_collision_device(samples, n_samples, collides, stream=DR.stream())
        free = samples[collides == 0]
    else:
        h = samples.cpu().numpy()
        free = torch.from_numpy(np.ascontiguousarray(h[~sim.check_config_collision(h)])).cuda()
    m = len(free)
    cand = tree.contiguous()
    ids = torch.empty(m, dtype=torch.int32, device="cuda")
    dist = torch.empty(m, dtype=torch.float64, device="cuda")
    sim.nearest_configurations(cand, n, free, m, 1, ids, dist, stream=DR.stream())
    starts = cand[ids.long()]
    dr2 = torch.empty(m * sim.result_stride, dtype=torch.uint8, device="cuda")
    sim.forward_simulate_device(starts, free, m, m, dr2, True, capi.NOISE_PHILOX, first_particle_id=n, stream=DR.stream())
    torch.cuda.synchronize()
    out = dr2.cpu().numpy().tobytes()
    sim.close()
    return out, m


@pytest.mark.parametrize("name,n,n_samples", [("se2_arena", 600, 1000), ("arm_table", 512, 1000)])
def test_one_extension_step_on_the_device_equals_the_host_step(name, n, n_samples):
    device_records, m = _extension_step(name, n, n_samples, True)
    host_records, m_host = _extension_step(name, n, n_samples, False)
    assert 0 < m < n_samples and m == m_host  # some samples are rejected, some kept
    assert len(device_records) == len(host_records) and device_records == host_records
