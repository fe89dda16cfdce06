#!/bin/bash
# build_ab/lib<NAME>.so with extra nvcc flags:  scripts/build_variant.sh R64 "-maxrregcount=64"
set -e
mkdir -p build_ab
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -fmad=false -prec-div=true -prec-sqrt=true -ftz=false \
  -Xcompiler -fPIC,-mfma,-ffp-contract=off -shared -cudart static $2 -o build_ab/lib$1.so \
  marlnav_b200/csrc/marlnav_kernels.cu marlnav_b200/csrc/marlnav_rollout.cu
echo built build_ab/lib$1.so
