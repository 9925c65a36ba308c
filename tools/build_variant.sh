#!/bin/bash
# Experiment build of the library with arbitrary -D flags: tools/build_variant.sh NAME "-DPKF_FUSE=1 ..."  -> tools/variants/libposekf_NAME.so
set -e
cd "$(dirname "$0")/.."
mkdir -p tools/variants
out=tools/variants/libposekf_$1.so
nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false --shared -Xcompiler -fPIC -Xptxas -v \
  $2 -o $out poseestimationkf_b200/csrc/posekf_capi.cu poseestimationkf_b200/csrc/replay_general_innovation.cu 2> $out.log
echo "$out: $(grep -A2 'replay_tma2_kernelILi0ELb0ELb0ELb0E' $out.log | grep -oE 'Used [0-9]+ registers|[0-9]+ bytes spill stores' | paste -sd' ')"
