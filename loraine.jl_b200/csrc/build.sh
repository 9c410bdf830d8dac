#!/bin/bash
# Builds libloraine_b200.so (sm_100a only) next to the Python host package.
set -e
cd "$(dirname "$0")"
OUT=../libloraine_b200.so
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC"
mkdir -p ../build
pids=()
for f in gemm chol chol_i8 eig ops pairs solver pcg dist group model debug ddlp dddist; do
  [ -f $f.cu ] || continue
  if [ ! -f ../build/$f.o ] || [ $f.cu -nt ../build/$f.o ] || [ -n "$(find . -name '*.cuh' -newer ../build/$f.o 2>/dev/null)" ] || [ -n "$(find ../../include -name '*.h' -newer ../build/$f.o 2>/dev/null)" ]; then
    $NVCC $FLAGS $EXTRA_INC -c $f.cu -o ../build/$f.o &
    pids+=($!)
  fi
done
for p in "${pids[@]}"; do wait $p; done
$NVCC -shared -o $OUT ../build/*.o -ldl $EXTRA_LIBS
echo "built $OUT"
