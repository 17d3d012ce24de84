#!/bin/bash
# Build an A/B variant of libikb200.so with extra -D flags for ONE source file, into gpurun_variants/ (git-ignored,
# travels to the GPU box).  Select it at run time with IKB200_LIB=gpurun_variants/<name>.so.
#   tools/build_variant.sh <name> <source.cu> [-DFOO=1 ...]
set -euo pipefail
name=$1; src=$2; shift 2
root=$(cd "$(dirname "$0")/.." && pwd)
csrc=$root/inversekinematicsann_b200/csrc
out=$root/gpurun_variants
mkdir -p "$out/obj_$name"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
ARCH="-gencode arch=compute_100a,code=sm_100a"
extra=""
case "$src" in fabrik.cu|fabrik_chain.cu) extra="--fmad=false" ;; esac  # as csrc/Makefile compiles them
$NVCC $ARCH -O3 -std=c++17 -lineinfo -Xcompiler -fPIC --expt-relaxed-constexpr $extra "$@" -c -o "$out/obj_$name/${src%.cu}.o" "$csrc/$src"
# every object the library links, from the Makefile's SRCS, so that the list cannot drift from it
srcs=$(make -s -C "$csrc" --no-print-directory --eval 'print-srcs: ; @echo $(SRCS)' print-srcs)
objs=""
for f in $srcs; do
  if [ "$f" = "$src" ]; then objs="$objs $out/obj_$name/${f%.cu}.o"; else objs="$objs $csrc/${f%.cu}.o"; fi
done
$NVCC $ARCH -shared -o "$out/$name.so" $objs
echo "$out/$name.so"
