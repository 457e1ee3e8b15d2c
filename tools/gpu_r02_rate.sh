#!/bin/bash
mkdir -p gpurun_out
mkdir -p build_tools && nvcc -gencode arch=compute_100a,code=sm_100a -O2 -o build_tools/umma_rate tools/umma_rate.cu || exit 1
timeout 120 ./build_tools/umma_rate > gpurun_out/umma_rate.log 2>&1; echo "exit $?"; cat gpurun_out/umma_rate.log
