"""Developer aid (not a test): A/B of two in-tree library builds on bench.py, alternating A B A B ... in one job.

    python tests/gpu_perf_ab.py A.so B.so [--runs 3] [--out DIR] [-- <bench.py arguments>]

A and B are libraries built in the tree (the default build fast_kinematic_simulator_b200/libfksgpu.so, or variants of
build_variant.sh); each run is a bench.py subprocess with FKSGPU_LIBRARY set to one of them.  Default bench arguments:
--gpus 1 --no-cpu-baseline --config5-particles 0.  Prints the card name, power limit and max SM clock (read-only
nvidia-smi query), every run's ms_per_step and kernel_ms_per_step, the mean and spread per side, and whether the
end-state records (bench.py --dump-outputs) of every run are byte-identical to the first A run's.
"""
import argparse
import filecmp
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, check=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError) as e:
        out = "unavailable (%s)" % e
    return out


def bench_once(lib, bench_args, dump_dir):
    env = dict(os.environ, FKSGPU_LIBRARY=os.path.abspath(lib))
    cmd = [sys.executable, os.path.join(ROOT, "bench.py")] + bench_args + ["--dump-outputs", dump_dir]
    p = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True)
    if p.returncode != 0:
        sys.stderr.write(p.stdout + p.stderr)
        raise SystemExit("bench.py failed with %s" % lib)
    line = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    return line["ms_per_step"], line.get("kernel_ms_per_step")


def same_dump(d0, d1):
    f0, f1 = sorted(os.listdir(d0)), sorted(os.listdir(d1))
    return f0 == f1 and all(filecmp.cmp(os.path.join(d0, f), os.path.join(d1, f), shallow=False) for f in f0)


def main():
    argv = sys.argv[1:]
    bench_args = ["--gpus", "1", "--no-cpu-baseline", "--config5-particles", "0"]
    if "--" in argv:
        i = argv.index("--")
        argv, bench_args = argv[:i], argv[i + 1:]
    ap = argparse.ArgumentParser()
    ap.add_argument("a")
    ap.add_argument("b")
    ap.add_argument("--runs", type=int, default=3, help="runs per side")
    ap.add_argument("--out", default=None, help="directory for the output dumps (default: a temporary one)")
    args = ap.parse_args(argv)
    out = args.out or tempfile.mkdtemp(prefix="fks_ab_")
    print("gpu:", gpu_info(), flush=True)
    print("bench.py", " ".join(bench_args), flush=True)
    res = {"A": [], "B": []}
    dumps = []
    for r in range(args.runs):
        for side, lib in (("A", args.a), ("B", args.b)):
            d = os.path.join(out, "%s%d" % (side, r))
            ms, kms = bench_once(lib, bench_args, d)
            res[side].append((ms, kms))
            dumps.append(d)
            print("%s run %d: ms_per_step %.3f  kernel_ms_per_step %s" % (side, r, ms, "%.3f" % kms if kms is not None else "-"),
                  flush=True)
    for side, lib in (("A", args.a), ("B", args.b)):
        v = [m for m, _ in res[side]]
        print("%s %s: mean %.3f ms, min %.3f, max %.3f" % (side, os.path.basename(lib), sum(v) / len(v), min(v), max(v)),
              flush=True)
    ma = sum(m for m, _ in res["A"]) / args.runs
    mb = sum(m for m, _ in res["B"]) / args.runs
    print("B vs A: %+.2f %% ms_per_step; every B run faster than every A run: %s" % (
        100.0 * (mb - ma) / ma, max(m for m, _ in res["B"]) < min(m for m, _ in res["A"])), flush=True)
    print("outputs byte-identical across all runs:", all(same_dump(dumps[0], d) for d in dumps[1:]), flush=True)


if __name__ == "__main__":
    main()
