#!/bin/bash
# tcgen05 int8 path: MMA mechanics in isolation, then the scoring kernel's parity tests and a first timing
mkdir -p gpurun_out
mkdir -p build_tools && nvcc -gencode arch=compute_100a,code=sm_100a -O2 -o build_tools/i8_mma_proto tools/i8_mma_proto.cu || exit 1
timeout 60 ./build_tools/i8_mma_proto > gpurun_out/i8_proto.log 2>&1; echo "proto exit $?"; tail -5 gpurun_out/i8_proto.log
timeout 600 python -m pytest tests/test_gpu_score_i8.py -x -q > gpurun_out/pytest_i8.log 2>&1; echo "pytest exit $?"; tail -25 gpurun_out/pytest_i8.log
timeout 300 python tools/bench_i8.py > gpurun_out/bench_i8.log 2>&1; echo "bench exit $?"; tail -8 gpurun_out/bench_i8.log
timeout 400 python -m pytest tests/test_gpu_linear.py -x -q > gpurun_out/pytest_linear.log 2>&1; echo "linear exit $?"; tail -15 gpurun_out/pytest_linear.log
