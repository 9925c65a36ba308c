#!/bin/bash
# Experiment builds of the replay kernel with different TMA ring shapes / occupancy targets.
# usage: tools/build_variants.sh "steps stages minctas" ...   -> tools/variants/libposekf_s{steps}_g{stages}_c{ctas}.so
set -e
cd "$(dirname "$0")/.."
for cfg in "$@"; do
  set -- $cfg
  out=tools/variants/libposekf_s$1_g$2_c$3.so
  nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false --shared -Xcompiler -fPIC -Xptxas -v \
    -DPKF_TMA_STEPS=$1 -DPKF_TMA_STAGES=$2 -DPKF_MIN_CTAS=$3 -o $out poseestimationkf_b200/csrc/posekf_capi.cu poseestimationkf_b200/csrc/replay_general_innovation.cu 2> $out.log
  echo "$out: $(grep -A2 'replay_tma_kernelILi0ELb0ELb0' $out.log | grep -oE 'Used [0-9]+ registers|[0-9]+ bytes spill stores' | paste -sd' ')  ldg: $(grep -A2 'replay_ldg_kernelILi0ELb0ELb0' $out.log | grep -oE 'Used [0-9]+ registers|[0-9]+ bytes spill stores' | paste -sd' ')"
done
