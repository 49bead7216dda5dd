#!/bin/bash
# Build libstheno_b200.so (sm_100a only) in-tree: stheno.jl_b200/libstheno_b200.so
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC,-O2 -Xptxas -v"
mkdir -p ../../build
for f in assemble gemm_nt ozaki potrf solve api; do
  $NVCC $FLAGS -c $f.cu -o ../../build/$f.o 2> ../../build/$f.ptxas.log || { cat ../../build/$f.ptxas.log; exit 1; }
done
$NVCC -shared -o ../libstheno_b200.so ../../build/assemble.o ../../build/gemm_nt.o ../../build/ozaki.o ../../build/potrf.o ../../build/solve.o ../../build/api.o -lcudart -ldl
echo "built $(cd ..; pwd)/libstheno_b200.so"
# test hooks over the Ozaki launchers (tests/test_gpu_ozaki_exact.py): linked against the library above, not a copy
$NVCC $FLAGS -shared -o ../../build/liboz_hooks.so ../../tests/csrc/oz_hooks.cu -L.. -lstheno_b200 -lcudart \
  -Xlinker -rpath,'$ORIGIN/../stheno.jl_b200' 2> ../../build/oz_hooks.ptxas.log || { cat ../../build/oz_hooks.ptxas.log; exit 1; }
echo "built $(cd ../..; pwd)/build/liboz_hooks.so"
