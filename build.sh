#!/bin/bash
# Builds libcmbpo_b200.so in-tree for sm_100a (cross-compiles without a GPU).
set -e
cd "$(dirname "$0")"
PKG="constrained-model-based-policy-optimization_b200"
SRC="$PKG/csrc"
OUT="$PKG/libcmbpo_b200.so"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xcompiler -Wall --expt-relaxed-constexpr"
mkdir -p build
objs=""
for f in capi gae ens_f32 ens_tc rollout policy_pack archive train train_tc; do
  if [ ! -f build/$f.o ] || [ $SRC/$f.cu -nt build/$f.o ] || [ -n "$(find $SRC include -name '*.cuh' -newer build/$f.o -o -name '*.h' -newer build/$f.o)" ]; then
    echo "nvcc $f.cu"
    $NVCC $FLAGS ${PTXAS_V:+-Xptxas -v} -c $SRC/$f.cu -o build/$f.o
  fi
  objs="$objs build/$f.o"
done
# cuBLAS (train.cu only: plain batched GEMMs of the ensemble training step) is linked dynamically; torch has
# usually loaded the same soname already, the rpath covers a process that has not
$NVCC -shared -o $OUT $objs -cudart static -lcublas -Xlinker -rpath -Xlinker /usr/local/cuda/lib64
echo "built $OUT"
