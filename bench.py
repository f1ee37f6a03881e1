#!/usr/bin/env python
"""Benchmark of the batched particle forward-simulate path (BASELINE.json metric:
particle-microsteps/sec with contact resolution).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload arm_table] [--particles P] [--impl reference]
                    [--dump-outputs DIR]

A "step" is ONE ForwardSimulateRobots call (simple_particle_contact_simulator.hpp:788) over one batch of
synthetic particles: 25 controller steps x their microsteps x contact resolution per particle.  Default
workload: BASELINE config 3, the 7-DoF linked arm with 65,536 particles PER GPU (weak scaling; at N GPUs the
job simulates N x 65,536 particles, and for N > 1 every step ends with the NCCL all-gather of end-state records
the north star names).  Noise is counter-based Philox keyed by global particle id.

value   = particle-microsteps / s, whole job, inputs resident in HBM, device-timed (CUDA events), max over ranks.
e2e     = the same metric with HOST buffers (pinned) through the C ABI: H2D of starts/targets + kernels + D2H of the
          result records inside the timed region; at N > 1 the records of ALL ranks are gathered (ncclAllGather) and
          read back on every rank inside it.
config5 = BASELINE config 5 in the same line: 1,048,576 arm particles IN TOTAL split over the N GPUs (strong scaling),
          all-gather of the end states included, device-timed.  A fixed-size leg: one warm-up call and two timed calls
          whatever --steps and --warmup say (--config5-particles 0 skips it).
--steps K sets the number of timed steps of value and of e2e; --warmup W the untimed steps before them.
roofline= the simulate kernel against the unit ncu shows binding for the workload.
--impl reference times the CPU restatement of the reference (oracle/, all host threads) on a bounded sample; that arm
never loads libfksgpu.so.
--dump-outputs DIR writes the end-state records of the last device-timed step (all ranks' records at N > 1) to
DIR/<field>.npy as float64, so that two builds can be compared output for output on the same seeded inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "particle-microsteps/sec (with contact resolution)"
UNIT = "particle-microsteps/s"
DEFAULT_PARTICLES = {"arm_table": 65536, "se3_narrow_passage": 16384, "se2_arena": 128, "se3_highres": 65536,
                     "arm_elbow": 65536, "arm_selfcollision": 4096}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="arm_table")
    ap.add_argument("--particles", type=int, default=0, help="particles per GPU (default: the BASELINE config's count)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config5-particles", type=int, default=1048576, help="total particles of the strong-scaling leg (0 = skip it)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU work budget of the cpu_baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the end-state records of the last timed step to DIR/<field>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm (the reference arm sizes its sample by timing)")
    return args


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def summary(self):
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for k, nm in enumerate(names):
                if len(s) > 4 + k and s[4 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


def algorithmic_work(stats, P, D, J):
    """SURVEY.md 8(d): ALGORITHMIC bytes, FP64 flops and SDF / normal-table gathers of a batch from its counters.
    bytes = 4 P per microstep + (28 P + 4 P) per resolver iteration + 56 per corrected point + (16 D + 16) per step;
    flops = (FK + 39 P) per microstep + (3 FK + 174 P + 12 D P) per iteration + (40 + 6 D^2) per corrected point;
    gathers = P per microstep + 8 P per iteration (one 4-byte SDF value per point per check, 7 per distance estimate)."""
    M = stats["total_microsteps"]
    I = stats["total_resolver_iterations"]
    K = stats["total_corrected_points"]
    S = stats["successful_resolves"] + stats["unsuccessful_resolves"]
    fk = 130 * J + 40 * J if J else (20 if D == 3 else 0)
    nbytes = 4 * P * M + 32 * P * I + 56 * K + (16 * D + 16) * S
    flops = (fk + 39 * P) * M + (3 * fk + P * (36 + 12 * D + 21 + 30) + 36 * P + 39 * P) * I + (40 + 6 * D * D) * K
    gathers = P * M + 8 * P * I
    return nbytes, flops, gathers


DUMP_LIMIT_BYTES = 64_000_000  # all files of one dump together, .npy headers included
NPY_HEADER_BYTES = 1024  # bound on one .npy header (numpy pads it to a multiple of 64 bytes: 128 for these arrays)


def dump_outputs(path, records):
    """One float64 .npy per field of the end-state records, plus particle_id.npy.  A batch whose dump would exceed
    DUMP_LIMIT_BYTES is represented by a fixed, seeded sample of its particles (the ids are in particle_id.npy)."""
    os.makedirs(path, exist_ok=True)
    n = len(records)
    per_particle = 8 * (1 + sum(int(np.prod(records.dtype[f].shape)) for f in records.dtype.names))
    budget = DUMP_LIMIT_BYTES - (1 + len(records.dtype.names)) * NPY_HEADER_BYTES
    ids = np.arange(n)
    if n * per_particle > budget:
        ids = np.sort(np.random.default_rng(0).choice(n, budget // per_particle, replace=False))
    np.save(os.path.join(path, "particle_id.npy"), ids.astype(np.float64))
    for f in records.dtype.names:
        np.save(os.path.join(path, f + ".npy"), records[f][ids].astype(np.float64))


def oracle_simulator(w, threads):
    """The CPU oracle for workload `w`, environment built by the oracle's own restatement of BuildCompleteEnvironment:
    nothing of the product is loaded on this path."""
    from fast_kinematic_simulator_b200 import abi
    from oracle import oracle_binding as OB

    env = OB.build_environment(w.obstacles, w.resolution)
    desc, keep = abi.env_desc_from_arrays(env)
    orc = OB.OracleSimulator(desc, w.robot.to_c(), abi.default_solver_params(), 25.0, 42, threads)
    orc._keep_env = keep
    return orc


def run_reference(args, rank, world):
    """The reference's CPU implementation of the path: here the oracle port (the reference itself cannot be
    compiled without Eigen/ROS/arc_utilities/sdf_tools, DESIGN.md), all host threads, bounded sample per step."""
    if rank != 0:
        return
    from fast_kinematic_simulator_b200 import abi, workloads as W

    n_per_gpu = args.particles or DEFAULT_PARTICLES.get(args.workload, 65536)
    w = W.make(args.workload, n_particles=min(n_per_gpu, 8192))
    # all host threads (torchrun exports OMP_NUM_THREADS=1: ask for the cores explicitly)
    orc = oracle_simulator(w, host_threads())
    # calibrate the sample so that one step is ~4 s of CPU work
    n0 = min(128, w.n_particles)
    s0, t0 = w.subset(n0)
    t = time.perf_counter()
    orc.forward_simulate(s0, t0, True, abi.NOISE_PHILOX)
    dt = max(time.perf_counter() - t, 1e-3)
    n = int(max(n0, min(w.n_particles, n0 * 4.0 / dt)))
    starts, targets = w.subset(n)
    times, micro = [], 0
    for it in range(args.warmup + args.steps):
        t = time.perf_counter()
        rec = orc.forward_simulate(starts, targets, True, abi.NOISE_PHILOX)
        dt = time.perf_counter() - t
        if it >= args.warmup:
            times.append(dt)
            micro = int(rec["n_microsteps"].sum())
    total = sum(times)
    value = micro * len(times) / total
    sample = "first %d of %d particles of workload %s per step, Philox noise, %d OpenMP threads" % (n, n_per_gpu, w.name, orc.num_threads)
    loaded = [l.split()[-1] for l in open("/proc/self/maps") if ".so" in l and ("fks" in l)]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": w.name, "particles_per_step": n, "description": w.description,
                   "note": "CPU restatement of the reference (oracle port, environment built by the oracle too); the reference "
                           "itself needs Eigen/ROS/arc_utilities/sdf_tools",
                   "native_libraries": sorted(set(os.path.basename(x) for x in loaded))},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": orc.num_threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    from fast_kinematic_simulator_b200 import capi, workloads as W

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n_local = args.particles or DEFAULT_PARTICLES.get(args.workload, 65536)
    w = W.make(args.workload, n_particles=n_local)
    if world > 1:
        # weak scaling: every rank simulates its own contiguous shard of the (world * n_local)-particle job;
        # starts are regenerated per shard with a shard-specific seed
        w = W.make(args.workload, n_particles=n_local, seed=1003 + rank) if args.workload != "se2_arena" else w
    sim = w.make_simulator(device=local_rank)
    sim.enable_kernel_timing(True)
    rd = w.robot
    P, D, J = rd.points.shape[0], rd.n_dof, len(rd.joints)
    stride, rec = sim.config_stride, sim.result_stride
    n_targets = w.targets.shape[0]
    first_id = rank * n_local

    dev = torch.device("cuda", local_rank)
    d_starts = torch.from_numpy(w.starts).to(dev)
    d_targets = torch.from_numpy(w.targets).to(dev)
    d_results = torch.empty(n_local * rec, dtype=torch.uint8, device=dev)
    d_gather = torch.empty(world * n_local * rec, dtype=torch.uint8, device=dev) if world > 1 else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    stream = torch.cuda.current_stream()

    def device_step(ds=d_starts, n=n_local, first=first_id, out=d_results, gather=d_gather):
        sim.forward_simulate_device(ds, d_targets, n, n_targets if n_targets == 1 else n, out, True, capi.NOISE_PHILOX,
                                    first_particle_id=first, stream=stream.cuda_stream)
        if world > 1:
            dist.all_gather_into_tensor(gather, out)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing ---------------------------------------------------------------
    for _ in range(args.warmup):
        device_step()
    barrier()
    sim.reset_statistics()
    launches0 = sim.launch_count
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kernel_ms = []  # per step: device time of the simulate kernel
    barrier()
    for i in range(args.steps):
        flush.fill_(i & 0xFF)  # L2 flush between timed iterations (outside the timed events)
        ev[i][0].record(stream)
        device_step()
        ev[i][1].record(stream)
        kernel_ms.append(sim.kernel_times_ms())  # waits for this step's kernels; the events above are on the stream
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, (d_gather if world > 1 else d_results).cpu().numpy().view(sim.dtype))
    step_ms = sum(a.elapsed_time(b) for a, b in ev)
    stats = sim.get_statistics()
    launches = sim.launch_count - launches0
    if rank == 0:
        sampler.stop_flag.set()
        sampler.join()

    # ---- end to end with host (pinned) buffers: H2D, kernels, gather over the ranks, D2H, all inside the timed region ----
    h_starts = torch.from_numpy(w.starts).pin_memory()
    h_targets = torch.from_numpy(w.targets).pin_memory()
    if world == 1:
        h_results = torch.empty(n_local * rec, dtype=torch.uint8).pin_memory()
        out = h_results.numpy().view(sim.dtype)
        hs, ht = h_starts.numpy(), h_targets.numpy()

        def e2e_step():
            return int(sim.forward_simulate_robots(hs, ht, True, capi.NOISE_PHILOX, first_particle_id=first_id, out=out).n_microsteps.sum())
    else:
        h_all = torch.empty(world * n_local * rec, dtype=torch.uint8).pin_memory()
        view = h_all.numpy().view(sim.dtype)

        def e2e_step():
            d_starts.copy_(h_starts, non_blocking=True)
            d_targets.copy_(h_targets, non_blocking=True)
            device_step()
            h_all.copy_(d_gather, non_blocking=True)
            torch.cuda.synchronize()
            return int(view["n_microsteps"][rank * n_local:(rank + 1) * n_local].sum())
    for _ in range(max(1, args.warmup // 2)):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        micro_e2e = e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0

    # ---- BASELINE config 5: 1,048,576 arm particles in total over the N GPUs (strong scaling), all-gather included ----
    c5 = None
    if args.config5_particles > 0 and args.workload == "arm_table":
        n5 = args.config5_particles // world
        w5 = W.make("arm_table", n_particles=n5, seed=2003 + rank)
        s5 = torch.from_numpy(w5.starts).to(dev)
        r5 = torch.empty(n5 * rec, dtype=torch.uint8, device=dev)
        g5 = torch.empty(world * n5 * rec, dtype=torch.uint8, device=dev) if world > 1 else None
        device_step(s5, n5, rank * n5, r5, g5)  # warm-up (allocates the hand-over buffers for this size)
        barrier()
        st0 = sim.get_statistics()
        e5 = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        reps5 = 2
        e5[0].record(stream)
        for _ in range(reps5):
            device_step(s5, n5, rank * n5, r5, g5)
        e5[1].record(stream)
        barrier()
        st1 = sim.get_statistics()
        c5 = [e5[0].elapsed_time(e5[1]) / reps5, float(st1["total_microsteps"] - st0["total_microsteps"]) / reps5]
        del s5, r5, g5

    # ---- reduce over ranks: max time, sum of work ------------------------------------------------
    kms = [sum(k[j] for k in kernel_ms) / len(kernel_ms) for j in range(len(kernel_ms[0]))]
    vals = torch.tensor([step_ms, e2e_s, c5[0] if c5 else 0.0], dtype=torch.float64, device=dev)
    work = torch.tensor([float(stats[k]) for k in capi.STAT_NAMES] + [float(micro_e2e), c5[1] if c5 else 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        dist.all_reduce(work, op=dist.ReduceOp.SUM)
    step_ms, e2e_s, c5_ms = [float(x) for x in vals.tolist()]
    tot = {k: int(v) for k, v in zip(capi.STAT_NAMES, work.tolist()[:-2])}
    micro_e2e_total, c5_micro = int(work.tolist()[-2]), work.tolist()[-1]

    if rank == 0:
        value = tot["total_microsteps"] / (step_ms * 1e-3)
        e2e_value = micro_e2e_total * args.steps / e2e_s
        # Roofline of the (single) kernel of the call, per launch, from THIS rank's counters and the device time of the kernel
        nbytes, flops, gathers = algorithmic_work(stats, P, D, J)
        k_s = kms[0] * 1e-3
        kname = "simulate_kernel<%d, false>" % w.kind
        peak, how = measured_peaks()
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                traffic = json.load(f).get(w.name)
        sdf_bytes = 4 * int(np.prod(w.environment().shape))
        import ctypes as C
        fp, ga, gh = C.c_double(), C.c_double(), C.c_double()
        have_fp = capi.lib.fks_measure_fp64_peak(local_rank, C.byref(fp)) == 0
        have_g = capi.lib.fks_measure_gather_rate(local_rank, 64 << 20, C.byref(ga)) == 0 and \
            capi.lib.fks_measure_gather_rate(local_rank, 2 << 30, C.byref(gh)) == 0
        hbm_resident = sdf_bytes > (100 << 20)
        roof_hbm = {"bound": "hbm", "achieved": nbytes / args.steps / k_s / 1e9, "peak": peak, "unit": "GB/s",
                    "frac": nbytes / args.steps / k_s / 1e9 / peak, "traffic": traffic, "peak_source": how, "kernel": kname,
                    "kernel_ms_per_launch": 1e3 * k_s, "algorithmic_bytes_per_launch": nbytes // args.steps}
        if hbm_resident or not have_g:
            roofline = dict(roof_hbm, note="the SDF (%d MB) does not fit the L2: its gathers are HBM traffic" % (sdf_bytes >> 20))
        else:
            g_rate = gathers / args.steps / k_s
            roofline = {"bound": "l2_gather", "achieved": g_rate / 1e9, "peak": ga.value / 1e9, "unit": "Ggather/s (4-byte, L2-resident)",
                        "frac": g_rate / ga.value, "traffic": traffic,
                        "peak_source": "random 4-byte __ldg gathers over an L2-resident 64 MiB array, measured in this job (fks_measure_gather_rate)",
                        "kernel": kname, "kernel_ms_per_launch": 1e3 * k_s, "algorithmic_gathers_per_launch": gathers // args.steps,
                        "algorithmic_bytes_per_launch": nbytes // args.steps,
                        "note": "the %.1f MB SDF is L2-resident (persisting window): DRAM is idle (traffic = measured DRAM bytes of one launch), "
                                "the binding units are the L2 gather path and the FP64 pipe; see roofline_hbm / roofline_fp64 for the other "
                                "denominators" % (sdf_bytes / 1e6)}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": w.name, "particles_per_gpu": n_local, "particles_total": n_local * world,
                       "description": w.description, "noise": "philox4x32-10 truncated normal, keyed by global particle id",
                       "controller_hz": 25, "forward_simulation_time_s": 1.0, "l2": "flushed between timed steps (256 MiB fill)",
                       "collective": "ncclAllGather of %d-byte end-state records" % rec if world > 1 else "none (1 GPU)",
                       "microsteps_per_step": tot["total_microsteps"] // args.steps,
                       "resolver_iterations_per_step": tot["total_resolver_iterations"] // args.steps},
            "clocks": sampler.summary(),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(world * (n_local + n_targets) * stride * 8),
                    "d2h_bytes_per_step": int(world * n_local * rec * (world if world > 1 else 1)), "ms_per_step": 1e3 * e2e_s / args.steps,
                    "includes": "H2D of starts/targets, kernels, %sD2H of the records" % ("ncclAllGather of all ranks' records, " if world > 1 else "")},
            "gpu_launches": int(launches),
            "kernel_ms_per_step": kms[0],
            "roofline": roofline,
            "roofline_hbm": roof_hbm,
            "kernel_info": sim.kernel_info,
        }
        if have_fp:
            af = flops / args.steps / k_s
            line["roofline_fp64"] = {"achieved": af / 1e12, "peak": fp.value / 1e12, "unit": "TFLOP/s", "frac": af / fp.value,
                                     "peak_source": "dependent-free DFMA micro-benchmark in this job",
                                     "algorithmic_flops_per_launch": flops // args.steps}
        if have_g:
            line["gather_peaks"] = {"l2_resident_gathers_per_s": ga.value, "hbm_resident_gathers_per_s": gh.value}
        if c5 is not None:
            line["config5"] = {"workload": "arm_table", "particles_total": (args.config5_particles // world) * world, "scaling": "strong",
                               "ms_per_step": c5_ms, "value": c5_micro / (c5_ms * 1e-3), "unit": UNIT,
                               "collective": "ncclAllGather of end-state records" if world > 1 else "none (1 GPU)"}
        if not args.no_cpu_baseline and world == 1:  # reported at N = 1 only
            line["cpu_baseline"] = cpu_baseline(args, w)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def cpu_baseline(args, w):
    """The oracle port on this box's host cores, bounded sample of the same workload (rank 0, N = 1 shape)."""
    from fast_kinematic_simulator_b200 import abi

    orc = oracle_simulator(w, host_threads())
    n0 = min(256, w.n_particles)
    s0, t0 = w.subset(n0)
    t = time.perf_counter()
    orc.forward_simulate(s0, t0, True, abi.NOISE_PHILOX)
    dt = max(time.perf_counter() - t, 1e-3)
    n = int(max(n0, min(w.n_particles, n0 * args.cpu_seconds / dt)))
    starts, targets = w.subset(n)
    t = time.perf_counter()
    rec = orc.forward_simulate(starts, targets, True, abi.NOISE_PHILOX)
    dt = time.perf_counter() - t
    return {"value": float(rec["n_microsteps"].sum()) / dt, "unit": UNIT, "cores": orc.num_threads, "kind": "port",
            "sample": "first %d of %d particles of %s, one call, Philox noise, %.1f s" % (n, w.n_particles, w.name, dt)}


if __name__ == "__main__":
    main()
