#!/bin/bash
# builds a kernel-variant library: tools/build_variant.sh NAME "-DRCC_K2_MIN_CTAS=2 ..."  -> robot_camera_calibration_b200/build/variants/librcc_ba_NAME.so
set -e
cd "$(dirname "$0")/.."
name=$1; defs=$2
pkg=robot_camera_calibration_b200
out=$pkg/build/variants; mkdir -p $out/$name
for f in assemble evaluate schur dense problem pnp; do
  /usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC,-fopenmp,-O3 \
    --expt-relaxed-constexpr $defs -c $pkg/csrc/$f.cu -o $out/$name/$f.o &
done
wait
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -shared -o $out/librcc_ba_$name.so $out/$name/*.o \
  -Xcompiler -fopenmp -lcusolver -lcublas -lnccl -lgomp -Xlinker -rpath,/usr/local/cuda/lib64
echo $out/librcc_ba_$name.so
