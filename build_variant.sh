#!/bin/bash
# developer aid: builds fast_kinematic_simulator_b200/libfksgpu_<name>.so from fks_kernels.cu compiled with extra flags
#   ./build_variant.sh timers -DFKS_PHASE_TIMERS      (per-phase clock counters, read by tests/gpu_perf.py)
#   FKSGPU_LIBRARY=$PWD/fast_kinematic_simulator_b200/libfksgpu_<name>.so python tests/gpu_perf.py ...
set -e
name=$1; shift
cd "$(dirname "$0")/fast_kinematic_simulator_b200/csrc"
make -j4 > /dev/null
mkdir -p build_$name
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC,-fopenmp -I../../include -I. "$@" -c fks_kernels.cu -o build_$name/fks_kernels.o
nvcc -gencode arch=compute_100a,code=sm_100a -shared -Xcompiler -fopenmp -o ../libfksgpu_$name.so build_$name/fks_kernels.o build/fks_consumers.o build/fks_api.o build/fks_multi.o build/fks_env_builder.o build/environment_builder.o -lgomp -ldl
