#!/bin/bash
# Experiments: build the library with extra -D flags into libhydra_pspec_b200_<tag>.so (select it with HP_LIB_PATH).
#   ./build_variant.sh w24 -DHP_S3_WARPS=24
set -e
cd "$(dirname "$0")"
tag=$1; shift
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC $*"
mkdir -p build_$tag
for f in hp_kernels hp_zgemm hp_solve hp_solve3 hp_fft hp_fft2 hp_pertime hp_ptlow hp_eigh hp_engine hp_testhooks; do
  $NVCC $FLAGS -c $f.cu -o build_$tag/$f.o &
done
wait
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -o libhydra_pspec_b200_$tag.so build_$tag/*.o -lcudart
rm -rf build_$tag
echo "built libhydra_pspec_b200_$tag.so"
