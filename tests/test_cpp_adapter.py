"""The C++ host adapter (include/fksgpu_simulator.hpp, include/fksgpu_glue.hpp) compiles with a plain C++11 compiler against
the C ABI and behaves like the reference interface: CPU box -> loud failure (no fallback), GPU box -> the scenarios of
examples/ end where they should for all three robot kinds, through the single-GPU class, the several-GPU class and the
SimulatorInterface base.  The glue templates are checked against mock types with the reference's call-site API."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "fast_kinematic_simulator_b200")
PROGRAMS = {
    "se2": os.path.join(ROOT, "examples", "forward_simulate_se2.cpp"),
    "linked_se3": os.path.join(ROOT, "examples", "forward_simulate_linked_se3.cpp"),
    "glue_mock": os.path.join(ROOT, "tests", "cpp", "glue_mock_test.cpp"),
}


def build(name, directory):
    exe = str(directory / ("fksgpu_example_" + name))
    subprocess.check_call(["/usr/bin/g++", "-std=c++11", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"), PROGRAMS[name],
                           "-L" + LIB, "-lfksgpu", "-Wl,-rpath," + LIB, "-o", exe])
    return exe


@pytest.mark.parametrize("name", ["se2", "linked_se3"])
def test_adapter_compiles_and_fails_loudly_without_a_gpu(name, tmp_path):
    import torch

    r = subprocess.run([build(name, tmp_path)], capture_output=True, text=True)
    if torch.cuda.is_available():
        assert r.returncode == 0, r.stdout
    else:
        assert r.returncode == 3 and "no CUDA device" in r.stdout


def test_glue_templates_against_mock_reference_types(tmp_path):
    r = subprocess.run([build("glue_mock", tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["se2", "linked_se3"])
def test_adapter_on_gpu(name, tmp_path):
    r = subprocess.run([build(name, tmp_path)], capture_output=True, text=True)
    print(r.stdout)
    assert r.returncode == 0 and "ok" in r.stdout and "FAILED" not in r.stdout, r.stdout + r.stderr
