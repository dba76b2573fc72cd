#!/bin/bash
# Build libmmunet_b200.so (sm_100a only) in-tree.  Usage: mm-unet_b200/csrc/build.sh [-j]
set -e
cd "$(dirname "$0")"
# Experiments: MMU_VARIANT=name MMU_EXTRA="-DMMU_V4_L2PF=0" build.sh builds ../mmunet_b200/libmmunet_b200_name.so in build_name/
# (select it at run time with MMU_LIB=<path>); the product library is the plain build.
OUT=../mmunet_b200/libmmunet_b200${MMU_VARIANT:+_$MMU_VARIANT}.so
BUILD=build${MMU_VARIANT:+_$MMU_VARIANT}
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 --expt-relaxed-constexpr -diag-suppress 128 -Xcompiler -fPIC $MMU_EXTRA"
mkdir -p $BUILD
pids=()
for f in capi selective_scan_fwd selective_scan_bwd causal_conv1d scan_order snake_sample group_norm narrow_mamba det_reduce resize_bilinear sw_stitch; do
  if [ ! -f $BUILD/$f.o ] || [ $f.cu -nt $BUILD/$f.o ] || [ common.cuh -nt $BUILD/$f.o ] || [ scan_tiles.cuh -nt $BUILD/$f.o ] || [ scan3.cuh -nt $BUILD/$f.o ] || [ scan3_fwd.cuh -nt $BUILD/$f.o ] || [ scan3_bwd.cuh -nt $BUILD/$f.o ] || [ scan4.cuh -nt $BUILD/$f.o ] || [ scan4_bwd.cuh -nt $BUILD/$f.o ] || [ scan5_fwd.cuh -nt $BUILD/$f.o ] || [ tma_map.cuh -nt $BUILD/$f.o ] || [ ../../include/mmunet_b200.h -nt $BUILD/$f.o ]; then
    nvcc $FLAGS -c $f.cu -o $BUILD/$f.o &
    pids+=($!)
  fi
done
for p in "${pids[@]}"; do wait $p; done
nvcc -shared -gencode arch=compute_100a,code=sm_100a -o $OUT $BUILD/*.o
echo "built $OUT"
