#!/bin/bash
# Build library variants for on-box A/B runs: tools/build_variants.sh NAME "-DRT_MINB=1 ..." [NAME2 "flags2" ...]
# The result is tools/variants/lib<NAME>.so, selected at run time with $ER3T_B200_LIB (tools/gpu_variants.sh).
cd "$(dirname "$0")/.."
mkdir -p tools/variants
while [ $# -ge 2 ]; do
  NAME=$1; FLAGS=$2; shift 2
  ( nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 --use_fast_math --shared -Xcompiler -fPIC $FLAGS \
      -o tools/variants/lib$NAME.so er3t_b200/csrc/b200rt.cu && echo "built $NAME ($FLAGS)" ) &
done
wait
