#!/bin/bash
# tools/build_variant.sh <tag> [extra nvcc flags for gemm_small.cu ...]
# Links quanta_b200/csrc/build/variants/lib<tag>.so from the regular objects plus a gemm_small.cu compiled with the
# given flags (-DQUANTA_SMALL_TRACE: timeline stamps).  For tools/ab_small.sh
# and tools/trace_small.py; the variants are git-ignored and travel with the gpurun snapshot.
set -e
cd "$(dirname "$0")/../quanta_b200/csrc"
tag=$1; shift
make -j8 > /dev/null
mkdir -p build/variants
nvcc "$@" -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -Xcompiler -fvisibility=hidden \
     --expt-relaxed-constexpr -c gemm_small.cu -o build/variants/gemm_small_$tag.o
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o build/variants/lib$tag.so \
     $(ls build/*.o | grep -v "build/gemm_small.o") build/variants/gemm_small_$tag.o -cudart shared
echo built build/variants/lib$tag.so
