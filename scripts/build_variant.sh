#!/bin/bash
# build_ab/lib<NAME>.so with extra nvcc flags:  scripts/build_variant.sh R64 "-maxrregcount=64"
set -e
mkdir -p build_ab
python -c 'import sys; from marlnav_b200.build import compile_library; compile_library(sys.argv[1], sys.argv[2].split())' "build_ab/lib$1.so" "$2"
echo built build_ab/lib$1.so
