#!/bin/bash
# Experiment builds of the packed Wahba-only kernel: "minctas waves" -> tools/variants/libposekf_w{minctas}_{waves}.so
set -e
cd "$(dirname "$0")/.."
mkdir -p tools/variants
for cfg in "$@"; do
  set -- $cfg
  out=tools/variants/libposekf_w$1_$2.so
  nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false --shared -Xcompiler -fPIC -Xptxas -v \
    -DPKF_WAHBA2_MIN_CTAS=$1 -DPOSEKF_WAHBA2_WAVES=$2 -o $out poseestimationkf_b200/csrc/posekf_capi.cu poseestimationkf_b200/csrc/replay_general_innovation.cu 2> $out.log
  echo "$out: $(grep -A2 'wahba2_kernel' $out.log | grep -oE 'Used [0-9]+ registers|[0-9]+ bytes spill stores' | paste -sd' ')"
done
