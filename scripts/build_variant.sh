#!/bin/bash
# Build a variant of the library for kernel experiments: build/libspgg_<tag>.so with extra -D flags.
# usage: bash scripts/build_variant.sh <tag> [-DSPGG_X_... ...]     (select it with SPGG_B200_LIB=build/libspgg_<tag>.so)
TAG=$1; shift
PKG=$(ls -d neighbor*_b200)
mkdir -p build/obj_$TAG
FLAGS="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -w"
for u in spgg_capi spgg_inst_general spgg_inst_lean spgg_clusters spgg_pairs spgg_blocks spgg_hist spgg_overlap; do
  nvcc $FLAGS "$@" -c $PKG/csrc/$u.cu -o build/obj_$TAG/$u.o &
done
wait
nvcc $FLAGS -shared -o build/libspgg_${TAG}.so build/obj_$TAG/*.o && echo "built build/libspgg_${TAG}.so"
