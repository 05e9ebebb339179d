#!/bin/bash
# usage: SRC=<dir> tools/build_variant.sh <name>   -> nvdiffrecmc_b200/lib/variants/<name>.so
#        compiles the sources of another directory (e.g. an older revision checked out to /tmp; default: this tree) for same-box A/B
#        runs with MCS_LIB=nvdiffrecmc_b200/lib/variants/<name>.so.  The include path still points at this tree's include/mcshade.h,
#        so the variant must have the same C ABI.
set -e
root="$(cd "$(dirname "$0")/.." && pwd)"
src="${SRC:-$root/nvdiffrecmc_b200/csrc}"
name=$1
out="$root/nvdiffrecmc_b200/lib/variants"
mkdir -p "$out/obj_$name"
cd "$src"
for f in core elementwise denoise bvh envshade lossmesh light raster; do
  nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC -c $f.cu -o "$out/obj_$name/$f.o" &
done
wait
nvcc -shared -gencode arch=compute_100a,code=sm_100a -o "$out/$name.so" "$out"/obj_$name/*.o
rm -rf "$out/obj_$name"
echo built $name
