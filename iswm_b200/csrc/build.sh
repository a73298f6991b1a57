#!/bin/bash
# Builds libiswm_b200.so in-tree for sm_100a (cross-compiles without a GPU).
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 --expt-relaxed-constexpr -Xcompiler -fPIC"
mkdir -p build
pids=()
for f in lib loss_metric elementwise bn_dual stem_pool sgd_pack scale_crop shape_metrics tail_fused tta quant tc_host conv_igemm conv_wgrad peer_allreduce; do
  if [ -f $f.cu ]; then
    if [ ! -f build/$f.o ] || [ $f.cu -nt build/$f.o ] || [ common.cuh -nt build/$f.o ] || [ ew_common.cuh -nt build/$f.o ] || [ metric_common.cuh -nt build/$f.o ] || [ scale_math.h -nt build/$f.o ] || [ ../../include/iswm_b200.h -nt build/$f.o ] || { [ -f tc_common.cuh ] && [ tc_common.cuh -nt build/$f.o ]; }; then
      $NVCC $FLAGS $EXTRA -c $f.cu -o build/$f.o &
      pids+=($!)
    fi
  fi
done
for p in "${pids[@]}"; do wait $p; done
$NVCC -shared -o ../libiswm_b200.so build/*.o -gencode arch=compute_100a,code=sm_100a
echo "built $(realpath ../libiswm_b200.so)"
