#!/bin/bash
# Build libhydra_pspec_b200.so (sm_100a) and the host-only math shim, in-tree.
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC"
for f in hp_kernels hp_zgemm hp_solve hp_solve3 hp_fft hp_fft2 hp_pertime hp_ptlow hp_eigh hp_moments hp_engine hp_testhooks; do
  if [ ! -f $f.o ] || [ $f.cu -nt $f.o ] || [ hp_kernels.cuh -nt $f.o ] || [ hp_mma.cuh -nt $f.o ] || [ hp_math.h -nt $f.o ] || [ hp_diag.cuh -nt $f.o ] || [ hp_async.cuh -nt $f.o ] || [ ../../include/hydra_pspec_b200.h -nt $f.o ]; then
    $NVCC $FLAGS -c $f.cu -o $f.o &
  fi
done
wait
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -o libhydra_pspec_b200.so hp_kernels.o hp_zgemm.o hp_solve.o hp_solve3.o hp_fft.o hp_fft2.o hp_pertime.o hp_ptlow.o hp_eigh.o hp_moments.o hp_engine.o hp_testhooks.o -lcudart
g++ -O2 -shared -fPIC -o libhp_math_host.so hp_math_host.cpp
echo "built $(pwd)/libhydra_pspec_b200.so"
