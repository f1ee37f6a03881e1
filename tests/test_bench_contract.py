"""bench.py on a CPU box: the reference arm runs the oracle port WITHOUT loading the product library and prints the
contract's JSON line; the product arm refuses to run without a GPU (no CPU fallback).  --dump-outputs writes the records of
the last timed step (on the GPU: the records the simulator returns for the same inputs)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line_and_never_loads_the_product():
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0", "--workload", "se2_arena"],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in line, key
    assert line["impl"] == "reference" and line["gpu_launches"] == 0 and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    libs = line["config"]["native_libraries"]
    assert "libfks_oracle.so" in libs and not any("fksgpu" in x for x in libs), libs


def test_other_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"], cwd=ROOT,
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_product_arm_fails_loudly_without_a_gpu():
    import torch

    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, "bench.py", "--steps", "1", "--warmup", "0"], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)


def test_dump_outputs_stay_within_the_size_limit(tmp_path, monkeypatch):
    import bench
    from fast_kinematic_simulator_b200.simulator import result_dtype

    names = ["cfg.npy", "flags.npy", "n_microsteps.npy", "n_resolver_iters.npy", "n_steps.npy", "particle_id.npy"]
    limit = 100 * 12 * 8 + len(names) * bench.NPY_HEADER_BYTES  # room for the arrays of 100 particles and every header
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", limit)
    # 160 particles: the arrays alone fit the limit, with the headers they do not
    for n, kept in ((100, 100), (160, 100), (1000, 100)):
        rec = np.zeros(n, dtype=result_dtype(7))
        rec["cfg"] = np.arange(7 * n, dtype=np.float64).reshape(n, 7)
        rec["n_microsteps"] = np.arange(n)
        a, b = tmp_path / ("a%d" % n), tmp_path / ("b%d" % n)
        bench.dump_outputs(str(a), rec)
        bench.dump_outputs(str(b), rec)
        assert sorted(os.listdir(a)) == names
        assert sum(os.path.getsize(a / f) for f in names) <= limit
        ids = np.load(a / "particle_id.npy")
        assert len(ids) == kept and np.all(np.diff(ids) > 0)
        for f in names:
            x, y = np.load(a / f), np.load(b / f)
            assert x.dtype == np.float64 and np.array_equal(x, y)
        assert np.array_equal(np.load(a / "cfg.npy"), rec["cfg"][ids.astype(int)])
        assert np.array_equal(np.load(a / "n_microsteps.npy"), ids)


@pytest.mark.gpu
def test_dump_outputs_are_the_records_of_the_timed_path(tmp_path):
    from fast_kinematic_simulator_b200 import capi, workloads as W

    r = subprocess.run([sys.executable, "bench.py", "--workload", "arm_table", "--particles", "700", "--steps", "3", "--warmup", "1",
                        "--config5-particles", "0", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    w = W.arm_table(700)
    ref = w.make_simulator().forward_simulate_robots(w.starts, w.targets, True, capi.NOISE_PHILOX).records
    # the microsteps counted over the timed loop, divided by --steps, are those of one batch: the loop ran --steps times
    assert line["steps"] == 3 and line["config"]["microsteps_per_step"] == int(ref["n_microsteps"].sum())
    assert np.array_equal(np.load(tmp_path / "particle_id.npy"), np.arange(700))
    for f in ref.dtype.names:
        assert np.array_equal(np.load(tmp_path / (f + ".npy")), ref[f].astype(np.float64)), f
