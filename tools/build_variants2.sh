#!/bin/bash
# Experiment builds of the PACKED replay kernel: "steps stages minctas" -> tools/variants/libposekf_p{steps}_{stages}_{ctas}.so
set -e
cd "$(dirname "$0")/.."
mkdir -p tools/variants
for cfg in "$@"; do
  set -- $cfg
  out=tools/variants/libposekf_p$1_$2_$3_t${4:-64}.so
  nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false --shared -Xcompiler -fPIC -Xptxas -v \
    -DPKF_TMA2_STEPS=$1 -DPKF_TMA2_STAGES=$2 -DPKF_MIN_CTAS2=$3 -DPKF_THREADS2=${4:-64} -o $out poseestimationkf_b200/csrc/posekf_capi.cu poseestimationkf_b200/csrc/replay_general_innovation.cu 2> $out.log
  echo "$out: $(grep -A2 'replay_tma2_kernelILi0ELb0ELb0ELb0E' $out.log | grep -oE 'Used [0-9]+ registers|[0-9]+ bytes spill stores' | paste -sd' ')"
done
