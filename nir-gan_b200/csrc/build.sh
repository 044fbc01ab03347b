#!/bin/bash
# Build libnirgan_b200.so for sm_100a (in-tree; the .so travels to the GPU box with the snapshot).
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -Xptxas -v --expt-relaxed-constexpr"
mkdir -p build
pids=()
for f in host api conv_simt conv_tc wgrad_tc head_tc elementwise backward postprocess scene; do
  ( $NVCC $FLAGS -c $f.cu -o build/$f.o > build/$f.log 2>&1 || { cat build/$f.log; exit 1; } ) &
  pids+=($!)
done
rc=0
for p in "${pids[@]}"; do wait $p || rc=1; done
[ $rc -eq 0 ] || exit 1
$NVCC -shared -o libnirgan_b200.so build/host.o build/api.o build/conv_simt.o build/conv_tc.o build/wgrad_tc.o build/head_tc.o build/elementwise.o build/backward.o build/postprocess.o build/scene.o -lcudart_static -ldl -lpthread -lrt
echo "built $(pwd)/libnirgan_b200.so"
