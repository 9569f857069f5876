#!/bin/bash
# Builds eigd_b200/libeigd_b200.so for sm_100a (cross-compiles without a GPU).
set -e
cd "$(dirname "$0")"
SRC=eigd_b200/csrc
OUT=eigd_b200/libeigd_b200.so
mkdir -p build
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -Xcompiler -O3 ${EIGD_NVCC_EXTRA}"
pids=()
for f in dense sparse factor solve krylov block_krylov fe buckling stored_fe h8 h8_buckling t10; do
  $NVCC $FLAGS -c $SRC/$f.cu -o build/$f.o &
  pids+=($!)
done
for f in symbolic solve_plan; do
  g++ -O3 -std=c++17 -fPIC -c $SRC/$f.cpp -o build/$f.o &
  pids+=($!)
done
for p in "${pids[@]}"; do wait $p || exit 1; done
$NVCC -shared -o $OUT build/dense.o build/sparse.o build/factor.o build/solve.o build/krylov.o build/block_krylov.o build/fe.o build/buckling.o build/stored_fe.o build/h8.o build/h8_buckling.o build/t10.o build/symbolic.o build/solve_plan.o -lcudart
echo "built $OUT"
