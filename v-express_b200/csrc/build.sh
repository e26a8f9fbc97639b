#!/bin/bash
# Build libvxb200.so in-tree for sm_100a (cross-compiles without a GPU).
set -e
cd "$(dirname "$0")"
OUT=../lib
mkdir -p $OUT build
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -O3 --expt-relaxed-constexpr"
pids=()
for f in vx_*.cu; do
  o=build/${f%.cu}.o
  if [ ! -f $o ] || [ $f -nt $o ] || [ vx_ptx.cuh -nt $o ] || [ vx_host.h -nt $o ] || [ vx_bringup.h -nt $o ] || [ ../../include/vxb200.h -nt $o ]; then
    ( $NVCC $FLAGS ${VX_PTXAS_V:+-Xptxas -v} -I../../include -c $f -o $o ) &
    pids+=($!)
  fi
done
for p in "${pids[@]}"; do wait $p; done
$NVCC -shared -o $OUT/libvxb200.so build/vx_*.o -lcudart
echo "built $OUT/libvxb200.so"
