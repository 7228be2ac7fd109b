#!/bin/bash
# Builds libnerfactor_b200.so in-tree (sm_100a only; no torch headers).
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xptxas -v"
mkdir -p build
objs=""
for f in nf_api nf_mlp_simt nf_mlp_api nf_integrate nf_integrate_bwd nf_stage_a nf_mlp_tc nf_sigma_tc nf_sigma_grad nf_sigma_grad_tc nf_nerf_tc nf_train nf_train_tc nf_point_tc nf_selftest nf_raymarch nf_stageb; do
  if [ ! -f build/$f.o ] || [ $f.cu -nt build/$f.o ] || [ nf_common.cuh -nt build/$f.o ] || [ nf_tc_ptx.cuh -nt build/$f.o ] || [ ../../include/nerfactor_b200.h -nt build/$f.o ]; then
    $NVCC $FLAGS -c $f.cu -o build/$f.o 2> build/$f.log || { cat build/$f.log; exit 1; }
  fi
  objs="$objs build/$f.o"
done
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -o ../libnerfactor_b200.so $objs
echo "built $(cd .. && pwd)/libnerfactor_b200.so"
