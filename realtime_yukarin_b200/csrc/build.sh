#!/bin/bash
# Builds libryk.so for sm_100a (B200) in-tree.  Usage: ./build.sh [-j N]
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -Xcompiler -Wno-unused-variable --expt-relaxed-constexpr $RYK_NVCC_EXTRA"
OBJ=${RYK_OBJ_DIR:-_obj}
mkdir -p $OBJ
SRCS="api crepe conv_direct conv_tc conv_tc3 s1_fused unet world_analysis world_harvest world_synth features convert session"
pids=""
for s in $SRCS; do
  if [ ! -f $OBJ/$s.o ] || [ $s.cu -nt $OBJ/$s.o ] || [ -n "$(find . -maxdepth 1 \( -name '*.h' -o -name '*.cuh' \) -newer $OBJ/$s.o 2>/dev/null)" ] || [ ../../include/ryk.h -nt $OBJ/$s.o ]; then
    $NVCC $FLAGS -c $s.cu -o $OBJ/$s.o &
    pids="$pids $!"
  fi
done
for p in $pids; do wait $p; done
OBJS=""; for s in $SRCS; do OBJS="$OBJS $OBJ/$s.o"; done
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -o ${RYK_LIB_OUT:-libryk.so} $OBJS -L/usr/local/cuda/lib64 -lcufft -Xlinker -rpath -Xlinker /usr/local/cuda/lib64
OUT=${RYK_LIB_OUT:-libryk.so}

echo "built $(pwd)/${RYK_LIB_OUT:-libryk.so}"
