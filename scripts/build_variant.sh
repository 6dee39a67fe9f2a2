#!/bin/bash
# Builds a differently tuned copy of the library for A/B runs on the GPU box: scripts/build_variant.sh <name> "<nvcc -D flags>"
# -> variants/libcm_<name>.so (git-ignored; select it with CM_LIB_PATH). Only the given sources are recompiled with the flags.
set -e
name=$1; flags=$2; shift 2
srcs=${@:-cm_radix_sort.cu}
root=$(cd "$(dirname "$0")/.." && pwd)
mkdir -p "$root/variants/obj_$name"
objs=""
# every source the library links, in build.py's order (the other objects come from its build directory)
all=$(python3 -c "import runpy, sys; print(' '.join(runpy.run_path(sys.argv[1])['SOURCES']))" "$root/cloud_merger_b200/build.py")
for s in $all; do
  o="$root/cloud_merger_b200/build/${s%.cu}.o"
  for v in $srcs; do
    if [ "$v" == "$s" ]; then
      o="$root/variants/obj_$name/${s%.cu}.o"
      nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo --fmad=false -Xcompiler -fPIC -Xcompiler -fvisibility=hidden \
        -Xcudafe --diag_suppress=177 $flags -c "$root/cloud_merger_b200/csrc/$s" -o "$o"
    fi
  done
  objs="$objs $o"
done
nvcc -shared -gencode arch=compute_100a,code=sm_100a -cudart static -o "$root/variants/libcm_$name.so" $objs
echo "$root/variants/libcm_$name.so"
