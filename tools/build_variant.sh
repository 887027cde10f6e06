#!/bin/bash
# Build an instrumented variant of the library next to the product one:
#   tools/build_variant.sh trace -DKPD_WS_TRACE        -> keypoint_diffusion_b200/libkpdiff_b200_trace.so
# Use it with KPD_LIB=keypoint_diffusion_b200/libkpdiff_b200_<name>.so python tools/...
# The sources are the Makefile's SRCS, so the variant links the same translation units as the product library.
set -e
name=$1; shift
root=$(cd "$(dirname "$0")/.." && pwd)
src=$root/keypoint_diffusion_b200/csrc
out=$root/build/$name
mkdir -p "$out"
srcs=$(make -s -C "$src" --eval 'print-srcs: ; @echo $(SRCS)' print-srcs)
objs=() pids=()
for f in $srcs; do
  o=$out/${f%.cu}.o
  objs+=("$o")
  /usr/local/cuda/bin/nvcc -O3 -std=c++17 -lineinfo -gencode arch=compute_100a,code=sm_100a -Xcompiler -fPIC "$@" -c "$src/$f" -o "$o" &
  pids+=($!)
done
for p in "${pids[@]}"; do wait "$p"; done
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -shared -o "$root/keypoint_diffusion_b200/libkpdiff_b200_$name.so" "${objs[@]}"
echo built "keypoint_diffusion_b200/libkpdiff_b200_$name.so"
