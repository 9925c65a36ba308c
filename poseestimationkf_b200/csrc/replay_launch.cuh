// replay_launch.cuh -- host-side launch helpers of the replay kernels, shared by the library's two translation units:
// posekf_capi.cu (dispatch and the extern "C" surface) and replay_general_innovation.cu (the general-matrix innovation
// kernels, a device module of its own so that the two compile in parallel).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/posekf.h"
#include "replay_kernels.cuh"

namespace pkf_host {
using namespace pkf;
using namespace pkf_dev;

#define PKF_CUDA_TRY(expr)                           \
  do {                                               \
    cudaError_t _e = (expr);                         \
    if (_e != cudaSuccess) return (int)_e;           \
  } while (0)

inline int launch_status() {
  cudaError_t e = cudaPeekAtLastError();
  return e == cudaSuccess ? 0 : (int)e;
}

// ---------------------------------------------------------------------------------------------
// launch logic
// ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess) return nullptr;
    if (q != cudaDriverEntryPointSuccess) return nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}

// Tensor map over the stream [T][9][Ns] (float32) with a box of `columns` filters x 9 channels x `steps`
// timesteps; out-of-range columns / steps are zero-filled by the TMA unit.
inline int encode_stream_map(const ReplayParams& p, int columns, int steps, CUtensorMap* tmap) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return POSEKF_ENODEV;
  const cuuint64_t dims[3] = {(cuuint64_t)p.Ns, (cuuint64_t)kChannels, (cuuint64_t)p.T};
  const cuuint64_t strides[2] = {(cuuint64_t)p.Ns * sizeof(float), (cuuint64_t)p.Ns * kChannels * sizeof(float)};
  const cuuint32_t box[3] = {(cuuint32_t)columns, (cuuint32_t)kChannels, (cuuint32_t)steps};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(p.streams), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : POSEKF_EALIGN;
}

// ga: the gate's arguments (one GateArgs; GATE launches only) or the general Q and R (one GenQRArgs; GEN launches only);
// the others pass none
template <int ALGO, bool LPF, bool AUX, bool COMP, bool INNOV = false, bool TAN = false, bool BATCH = false, bool GATE = false,
          bool GEN = false, typename... GA>
int launch_replay(const ReplayParams& p, bool use_tma, cudaStream_t st, const GA&... ga) {
  const unsigned grid = (unsigned)((p.N + kThreads - 1) / kThreads);
  if (!use_tma) {
    replay_ldg_kernel<ALGO, LPF, AUX, COMP, INNOV, TAN, BATCH, GATE, GEN, GA...><<<grid, kThreads, 0, st>>>(p, ga...);
    return launch_status();
  }
  CUtensorMap tmap;
  if (int rc = encode_stream_map(p, kThreads, kTmaSteps, &tmap)) return rc;
  auto kern = replay_tma_kernel<ALGO, LPF, AUX, COMP, INNOV, TAN, BATCH, GATE, GEN, GA...>;
  // idempotent; set on every launch (cheap) so that it holds on every device of a multi-GPU process
  PKF_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(TmaSmem)));
  kern<<<grid, kThreads, sizeof(TmaSmem), st>>>(p, tmap, ga...);
  return launch_status();
}

// Launches with general Q and R and the innovation terms (replay_general_innovation.cu; DESIGN.md section 5, f12).
// gate: the gated kernels with these arguments (null: the ungated ones); ia: the per-step output, whose `out` may be null.
int launch_general_innov_algo(const ReplayParams& p, const GenQRArgs& gq, const GateArgs* gate, const InnovStepArgs& ia,
                              int algo, bool lpf, bool use_tma, int innov_model, cudaStream_t st);

}  // namespace pkf_host
