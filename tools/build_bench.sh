#!/bin/bash
# builds tools/smooth_bench (development aid); extra nvcc flags are passed through
cd "$(dirname "$0")/.." && nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -I pressurepoissonsolver_b200/csrc "$@" tools/smooth_bench.cu -o tools/smooth_bench
