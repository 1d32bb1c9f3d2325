#!/bin/bash
# Build a kernel variant of libuavca.so with extra -D flags (A/B experiments; load it with UAVCA_LIB=<path>).
#   tools/build_variant.sh NAME [-DUAVCA_ROLLOUT_MINB=6 ...]  ->  build/variants/libuavca_NAME.so
set -e
name=$1; shift
root=$(cd "$(dirname "$0")/.." && pwd)
mkdir -p "$root/build/variants"
cd "$root/gym_uav_collision_avoidance_b200/csrc"
/usr/local/cuda/bin/nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC "$@" \
  -shared -o "$root/build/variants/libuavca_$name.so" uavca_kernels.cu uavca_policy.cu uavca_capi.cu
echo "$root/build/variants/libuavca_$name.so"
