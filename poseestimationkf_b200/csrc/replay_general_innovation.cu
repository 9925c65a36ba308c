// replay_general_innovation.cu -- launches of the general-matrix innovation kernels (GEN with INNOV, gated or not;
// DESIGN.md section 5, f12).  They are a device module of their own: build.py compiles this file and posekf_capi.cu in
// parallel, and the kernels of the other module are instantiated exactly as before.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/posekf.h"
#include "ekf_math.cuh"
#include "device_util.cuh"
#include "replay_kernels.cuh"
#include "replay_launch.cuh"

namespace pkf_host {
namespace {

// Launches with general Q and R and the innovation terms (posekf_replay_general_innovation_f32): the scalar BATCH GEN
// kernels with INNOV and AUX, gated or not, on the launch's staging (the TMA kernel for a packed staging).  Their pack is
// GenQRArgs, the GateArgs of a gated launch and an InnovStepArgs whose output may be null, and innov_acc is optional too:
// one set of kernels serves the sums, the per-step terms and the gate alone (the tangent gated kernel with neither).
template <int ALGO, bool TAN, bool GATE, typename... GA>
int launch_general_innov(const ReplayParams& p, bool lpf, bool use_tma, cudaStream_t st, const GA&... ga) {
  if constexpr (ALGO != WAHBA_PRECOMPUTED) {
    if (lpf) return launch_replay<ALGO, true, true, false, true, TAN, true, GATE, true>(p, use_tma, st, ga...);
  }
  return launch_replay<ALGO, false, true, false, true, TAN, true, GATE, true>(p, use_tma, st, ga...);
}

template <int ALGO>
int launch_general_innov_model(const ReplayParams& p, const GenQRArgs& gq, const GateArgs* gate, const InnovStepArgs& ia,
                               bool lpf, bool use_tma, int innov_model, cudaStream_t st) {
  const bool tan = innov_model == POSEKF_INNOV_TANGENT;
  if (gate) return tan ? launch_general_innov<ALGO, true, true>(p, lpf, use_tma, st, gq, *gate, ia)
                       : launch_general_innov<ALGO, false, true>(p, lpf, use_tma, st, gq, *gate, ia);
  return tan ? launch_general_innov<ALGO, true, false>(p, lpf, use_tma, st, gq, ia)
             : launch_general_innov<ALGO, false, false>(p, lpf, use_tma, st, gq, ia);
}

}  // namespace

int launch_general_innov_algo(const ReplayParams& p, const GenQRArgs& gq, const GateArgs* gate, const InnovStepArgs& ia, int algo,
                              bool lpf, bool use_tma, int innov_model, cudaStream_t st) {
  if (algo == POSEKF_WAHBA_QR2) return launch_general_innov_model<WAHBA_QR2>(p, gq, gate, ia, lpf, use_tma, innov_model, st);
  if (algo == POSEKF_WAHBA_PRECOMPUTED) return launch_general_innov_model<WAHBA_PRECOMPUTED>(p, gq, gate, ia, lpf, use_tma, innov_model, st);
  if (algo == POSEKF_WAHBA_JACOBI) return launch_general_innov_model<WAHBA_JACOBI>(p, gq, gate, ia, lpf, use_tma, innov_model, st);
  return POSEKF_EINVAL;
}

}  // namespace pkf_host
