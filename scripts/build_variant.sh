#!/bin/bash
# Build a variant of the product library with extra compiler flags for A/B experiments:
#   bash scripts/build_variant.sh <name> "<extra nvcc flags>"   ->  build_variants/liblrs_pnp_<name>.so   (git-ignored)
set -e
cd "$(dirname "$0")/../lrs_pnp_dip_b200/csrc"
NAME=$1; EXTRA=$2
OUT=../../build_variants; mkdir -p $OUT/obj_$NAME
FLAGS="-O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC $EXTRA"
# every source the Makefile links into the product library; sparse_fused_tc.cu is the one built per variant
for f in $(sed -n 's/^SRCS := //p' Makefile); do
  f=${f%.cu}; [ $f = sparse_fused_tc ] && continue
  [ -f $OUT/obj_common/$f.o ] || { mkdir -p $OUT/obj_common; nvcc $FLAGS -c $f.cu -o $OUT/obj_common/$f.o & }
done
nvcc $FLAGS -Xptxas -v -c sparse_fused_tc.cu -o $OUT/obj_$NAME/sparse_fused_tc.o 2>&1 | grep -A1 "kernelILb0ELi256ELb1" | grep -E "registers|spill" || true
wait
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o $OUT/liblrs_pnp_$NAME.so $OUT/obj_common/*.o $OUT/obj_$NAME/sparse_fused_tc.o -lcuda
echo built $OUT/liblrs_pnp_$NAME.so
