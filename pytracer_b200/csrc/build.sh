#!/bin/bash
# Builds libpytracer_b200.so for sm_100a (B200) in-tree.  The fp64 kernels are compiled without
# multiply-add fusion so that they round like the reference's Python arithmetic.
set -euo pipefail
cd "$(dirname "$0")"
OUT=${RT_OUT:-../libpytracer_b200.so}
B=${RT_BUILD_DIR:-build}
ARCH="-gencode arch=compute_100a,code=sm_100a"
COMMON="${RT_EXTRA_FLAGS:-} -O3 -std=c++17 -lineinfo -Xcompiler -fPIC"
mkdir -p $B
pids=()
nvcc $ARCH $COMMON -c rt_kernels_f32.cu -o $B/rt_kernels_f32.o & pids+=($!)
nvcc $ARCH $COMMON --fmad=false -c rt_kernels_f64.cu -o $B/rt_kernels_f64.o & pids+=($!)
nvcc $ARCH $COMMON -c rt_api.cu -o $B/rt_api.o & pids+=($!)
nvcc $ARCH $COMMON --fmad=false -c rt_tonemap.cu -o $B/rt_tonemap.o & pids+=($!)
nvcc $ARCH $COMMON -c rt_adaptive.cu -o $B/rt_adaptive.o & pids+=($!)
for pid in "${pids[@]}"; do wait "$pid"; done  # set -e: a failed translation unit fails the build
nvcc $ARCH -shared -o $OUT $B/rt_kernels_f32.o $B/rt_kernels_f64.o $B/rt_api.o $B/rt_tonemap.o $B/rt_adaptive.o -lcudart_static -lpthread -ldl -lrt
[ -f $OUT ] && echo "built $(realpath $OUT)"
