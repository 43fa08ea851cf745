#!/bin/bash
# usage: tools/build_variant.sh NAME "-DVX_ITEM_TASKS=256 ..."   -> variants/libvx_NAME.so (development: kernel tuning sweeps,
# loaded through VX_B200_LIB; the product always loads the in-tree library)
set -e
cd "$(dirname "$0")/../differential_projection_voxel_renderer_b200/csrc"
NAME=$1; FLAGS=$2
mkdir -p ../../variants build_$NAME
NVCC=/usr/local/cuda/bin/nvcc
COMMON="-O3 -std=c++17 -lineinfo -gencode arch=compute_100a,code=sm_100a -Xcompiler -fPIC -Xcompiler -fvisibility=hidden -I../../include"
$NVCC $COMMON -fmad=false $FLAGS -c vx_frame.cu -o build_$NAME/vx_frame.o
$NVCC $COMMON -fmad=false $FLAGS -c vx_ray.cu -o build_$NAME/vx_ray.o
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -o ../../variants/libvx_$NAME.so build/vx_context.o build/vx_mesh.o build_$NAME/vx_frame.o build/vx_misc.o build/vx_spanwalk.o build/vx_bary.o build/vx_multi.o build_$NAME/vx_ray.o
rm -rf build_$NAME
echo built variants/libvx_$NAME.so
