// posekf_capi.cu -- host dispatch + C ABI (include/posekf.h) of the batched quaternion EKF.
//
// Design (DESIGN.md has the long form):
//   * one filter per thread; X (4), upper-triangular P (10), the Wahba reference frame (12) and the
//     Q/R scalars live in registers for the whole launch -- a launch covers MANY timesteps;
//   * IMU samples are a structure-of-arrays stream [T][9][N] (filter index fastest), so a warp's
//     load of one channel of one step is one 128-byte line;
//   * staging: a TMA (cp.async.bulk.tensor.3d) ring of [TC][9][128] tiles in shared memory driven by
//     mbarriers (default), or plain coalesced LDG with a one-step register prefetch (unaligned input);
//   * template variants: Wahba solver (rank-2 QR / Jacobi), low-pass stage, auxiliary outputs
//     (trajectory, flip mask, tuning loss), compensated two-float state;
//   * no tensor cores (per-filter matrices are 4x4), no inter-thread communication on the step;
//   * filters are independent: multi-GPU = shard N, no collective on this path.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 --shared -Xcompiler -fPIC, with
// replay_general_innovation.cu (poseestimationkf_b200/build.py compiles the two in parallel and links them)
//
// Files: ekf_math.cuh (per-filter arithmetic, scalar and packed), device_util.cuh (TMA / mbarrier /
// streaming access helpers, tunables), replay_kernels.cuh (the three fused replay kernels),
// ops_kernels.cuh (stand-alone operators), replay_launch.cuh (launch helpers shared with
// replay_general_innovation.cu, which launches the general-matrix innovation kernels in a device module of its own),
// this file (launch logic and the extern "C" surface).
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <algorithm>
#include <vector>

#include "../../include/posekf.h"
#include "ekf_math.cuh"
#include "device_util.cuh"
#include "replay_kernels.cuh"
#include "ops_kernels.cuh"
#include "replay_launch.cuh"

using namespace pkf;
using namespace pkf_dev;
using namespace pkf_host;

namespace {

inline unsigned blocks_for(int64_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }

bool tma_eligible(const ReplayParams& p) {
  if ((reinterpret_cast<uintptr_t>(p.streams) & 15) != 0) return false;
  if ((reinterpret_cast<uintptr_t>(p.dt_cols) & 15) != 0) return false;   // (the TMA kernels read it with 8-byte loads)
  if (p.Ns % 4 != 0) return false;                        // global strides must be multiples of 16 bytes
  if (p.Ns != p.N && (p.Ns % kThreads) != 0) return false;   // a CTA's 128 columns must not wrap
  if (p.T > INT32_MAX || p.Ns > INT32_MAX) return false;
  return true;
}

bool packed_eligible(const ReplayParams& p) {
  // float2 accesses to the [k][N] state / constant arrays need N even and 8-byte aligned bases
  if ((p.N & 1) != 0) return false;
  if (p.Ns != p.N && (p.Ns % kTile2) != 0) return false;      // a CTA's columns must not wrap
  const void* ptrs[] = {p.acc_ref, p.mag_ref, p.q_scale, p.r_scale, p.state_x, p.state_x_lo, p.state_p, p.state_lpf};
  for (const void* q : ptrs) if ((reinterpret_cast<uintptr_t>(q) & 7) != 0) return false;
  if ((reinterpret_cast<uintptr_t>(p.loss_acc) & 7) != 0 || (reinterpret_cast<uintptr_t>(p.out_flip) & 1) != 0) return false;
  if ((reinterpret_cast<uintptr_t>(p.innov_acc) & 7) != 0) return false;
  return true;      // out_traj / truth are already required to be 16-byte aligned
}

template <int ALGO, bool LPF, bool AUX, bool COMP, bool INNOV = false, bool TAN = false, bool BATCH = false, bool GATE = false,
          typename... GA>
int launch_replay_packed(const ReplayParams& p, cudaStream_t st, const GA&... ga) {
  CUtensorMap tmap;
  if (int rc = encode_stream_map(p, kTile2, kTma2Steps, &tmap)) return rc;
  auto kern = replay_tma2_kernel<ALGO, LPF, AUX, COMP, INNOV, TAN, BATCH, GATE, GA...>;
  const int smem = (int)sizeof(Tma2Smem) + (BATCH ? (int)kBatchSmem2 : 0);
  PKF_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  const unsigned grid = (unsigned)((p.N + kTile2 - 1) / kTile2);
  kern<<<grid, kThreads2, smem, st>>>(p, tmap, ga...);
  return launch_status();
}

template <int ALGO, bool LPF, bool BATCH = false> int launch_replay_aux(const ReplayParams& p, bool use_tma, cudaStream_t st) {
  const bool aux = p.out_traj != nullptr || p.out_flip != nullptr || p.truth != nullptr;
  const bool comp = p.state_x_lo != nullptr;
  if (comp) return aux ? launch_replay<ALGO, LPF, true, true, false, false, BATCH>(p, use_tma, st) : launch_replay<ALGO, LPF, false, true, false, false, BATCH>(p, use_tma, st);
  return aux ? launch_replay<ALGO, LPF, true, false, false, false, BATCH>(p, use_tma, st) : launch_replay<ALGO, LPF, false, false, false, false, BATCH>(p, use_tma, st);
}

template <int ALGO, bool BATCH = false> int launch_packed_variant(const ReplayParams& p, bool lpf, cudaStream_t st) {
  const bool comp = p.state_x_lo != nullptr;
  const bool aux = p.out_traj != nullptr || p.out_flip != nullptr || p.truth != nullptr;
  if constexpr (BATCH) {
    // the precise packed step with per-step outputs or the low-pass, plus the copies a held lane needs, does not fit the
    // registers of 3 CTAs per SM: the scalar TMA kernel runs those (same results bit for bit)
    if (comp && (aux || lpf)) return lpf ? launch_replay_aux<ALGO, true, true>(p, true, st) : launch_replay_aux<ALGO, false, true>(p, true, st);
    if (lpf) return aux ? launch_replay_packed<ALGO, true, true, false, false, false, true>(p, st) : launch_replay_packed<ALGO, true, false, false, false, false, true>(p, st);
    if (aux) return launch_replay_packed<ALGO, false, true, false, false, false, true>(p, st);
    return comp ? launch_replay_packed<ALGO, false, false, true, false, false, true>(p, st) : launch_replay_packed<ALGO, false, false, false, false, false, true>(p, st);
  } else {
    if (lpf) {
      if (aux) return comp ? launch_replay_packed<ALGO, true, true, true>(p, st) : launch_replay_packed<ALGO, true, true, false>(p, st);
      return comp ? launch_replay_packed<ALGO, true, false, true>(p, st) : launch_replay_packed<ALGO, true, false, false>(p, st);
    }
    if (aux) return comp ? launch_replay_packed<ALGO, false, true, true>(p, st) : launch_replay_packed<ALGO, false, true, false>(p, st);
    return comp ? launch_replay_packed<ALGO, false, false, true>(p, st) : launch_replay_packed<ALGO, false, false, false>(p, st);
  }
}

// Launches with the innovation likelihood (TAN: its tangent-space form).  The packed kernel carries it without per-step
// outputs and low-pass (the (Q,R) sweep path, where the registers allow 12 warps per SM); every other combination runs
// in the scalar kernels on the same staging (TMA or LDG), whose results are the same bit for bit.
template <int ALGO, bool TAN = false, bool BATCH = false>
int launch_innovation(const ReplayParams& p, bool lpf, bool aux, bool use_tma, bool packed, cudaStream_t st) {
  const bool comp = p.state_x_lo != nullptr;
  if constexpr (ALGO != WAHBA_JACOBI) {
    if (packed && !lpf && !aux)
      return comp ? launch_replay_packed<ALGO, false, false, true, true, TAN, BATCH>(p, st) : launch_replay_packed<ALGO, false, false, false, true, TAN, BATCH>(p, st);
  }
  if constexpr (ALGO != WAHBA_PRECOMPUTED) {      // (the low-pass of a measurement stream belongs to its builder)
    if (lpf) return comp ? launch_replay<ALGO, true, true, true, true, TAN, BATCH>(p, use_tma, st) : launch_replay<ALGO, true, true, false, true, TAN, BATCH>(p, use_tma, st);
  }
  return comp ? launch_replay<ALGO, false, true, true, true, TAN, BATCH>(p, use_tma, st) : launch_replay<ALGO, false, true, false, true, TAN, BATCH>(p, use_tma, st);
}

template <bool TAN, bool BATCH = false>
int launch_innovation_algo(const ReplayParams& p, int algo, bool lpf, bool aux, bool use_tma, bool packed, cudaStream_t st) {
  if (algo == POSEKF_WAHBA_QR2) return launch_innovation<WAHBA_QR2, TAN, BATCH>(p, lpf, aux, use_tma, packed, st);
  if (algo == POSEKF_WAHBA_PRECOMPUTED) return launch_innovation<WAHBA_PRECOMPUTED, TAN, BATCH>(p, lpf, aux, use_tma, packed, st);
  if (algo == POSEKF_WAHBA_JACOBI) return launch_innovation<WAHBA_JACOBI, TAN, BATCH>(p, lpf, aux, use_tma, packed, st);
  return POSEKF_EINVAL;
}

// The kernels of a launch, chosen from its buffers.  BATCH: per-stream dt columns or lengths (ReplayParams::dt_cols /
// n_valid); every combination the other kernels accept has a BATCH twin on the same staging.
template <bool BATCH>
int launch_kernels(const ReplayParams& p, int algo, bool lpf, bool use_tma, bool packed, int innov_model, cudaStream_t st) {
  if (p.innov_acc) {
    const bool aux = p.out_traj != nullptr || p.out_flip != nullptr || p.truth != nullptr;
    return innov_model == POSEKF_INNOV_TANGENT ? launch_innovation_algo<true, BATCH>(p, algo, lpf, aux, use_tma, packed, st)
                                               : launch_innovation_algo<false, BATCH>(p, algo, lpf, aux, use_tma, packed, st);
  }
  if (packed)
    return algo == POSEKF_WAHBA_QR2 ? launch_packed_variant<WAHBA_QR2, BATCH>(p, lpf, st) : launch_packed_variant<WAHBA_PRECOMPUTED, BATCH>(p, lpf, st);
  if (algo == POSEKF_WAHBA_PRECOMPUTED) return lpf ? launch_replay_aux<WAHBA_PRECOMPUTED, true, BATCH>(p, use_tma, st) : launch_replay_aux<WAHBA_PRECOMPUTED, false, BATCH>(p, use_tma, st);
  if (algo == POSEKF_WAHBA_QR2) return lpf ? launch_replay_aux<WAHBA_QR2, true, BATCH>(p, use_tma, st) : launch_replay_aux<WAHBA_QR2, false, BATCH>(p, use_tma, st);
  if (algo == POSEKF_WAHBA_JACOBI) return lpf ? launch_replay_aux<WAHBA_JACOBI, true, BATCH>(p, use_tma, st) : launch_replay_aux<WAHBA_JACOBI, false, BATCH>(p, use_tma, st);
  return POSEKF_EINVAL;
}

// Launches with the innovation gate.  The scalar gated kernels are the BATCH kernels, which step exactly as the others
// when dt_cols and n_valid are null (bit for bit, see launch_kernels), so the gate adds one set of them, not two; they
// always have AUX (their per-step outputs are checked per pointer).  The packed kernel carries the plain variant with
// and without per-step outputs and the precise variant without them, all without low-pass and innovation sums (a
// trajectory replay and the (Q,R) sweep); with per-stream dt or lengths only the plain variant without per-step
// outputs, because the copies a held lane needs push the others past the 168 registers of 3 CTAs per SM.  Every other
// combination runs in the scalar kernels on the same staging (the TMA kernel for a packed staging), whose results are
// the same bit for bit.
template <int ALGO, bool TAN>
int launch_gated_innovation(const ReplayParams& p, const GateArgs& ga, bool lpf, bool use_tma, cudaStream_t st) {
  const bool comp = p.state_x_lo != nullptr;
  if constexpr (ALGO != WAHBA_PRECOMPUTED) {
    if (lpf) return comp ? launch_replay<ALGO, true, true, true, true, TAN, true, true>(p, use_tma, st, ga) : launch_replay<ALGO, true, true, false, true, TAN, true, true>(p, use_tma, st, ga);
  }
  return comp ? launch_replay<ALGO, false, true, true, true, TAN, true, true>(p, use_tma, st, ga) : launch_replay<ALGO, false, true, false, true, TAN, true, true>(p, use_tma, st, ga);
}

template <int ALGO>
int launch_gated(const ReplayParams& p, const GateArgs& ga, bool lpf, bool use_tma, bool packed, int innov_model, cudaStream_t st) {
  const bool comp = p.state_x_lo != nullptr;
  const bool aux = p.out_traj != nullptr || p.out_flip != nullptr || p.truth != nullptr || ga.out_gated != nullptr;
  if (p.innov_acc) return innov_model == POSEKF_INNOV_TANGENT ? launch_gated_innovation<ALGO, true>(p, ga, lpf, use_tma, st)
                                                              : launch_gated_innovation<ALGO, false>(p, ga, lpf, use_tma, st);
  // (the packed kernel reads gate_count as int2 and stores out_gated as uchar2)
  packed = packed && (reinterpret_cast<uintptr_t>(ga.gate_count) & 7) == 0 && (reinterpret_cast<uintptr_t>(ga.out_gated) & 1) == 0;
  if constexpr (ALGO != WAHBA_JACOBI) {
    const bool batch = p.dt_cols != nullptr || p.n_valid != nullptr;
    if (packed && !lpf && !comp && !aux) {
      return batch ? launch_replay_packed<ALGO, false, false, false, false, false, true, true>(p, st, ga)
                   : launch_replay_packed<ALGO, false, false, false, false, false, false, true>(p, st, ga);
    }
    if (packed && !lpf && !batch && !(comp && aux)) {
      return comp ? launch_replay_packed<ALGO, false, false, true, false, false, false, true>(p, st, ga)
                  : launch_replay_packed<ALGO, false, true, false, false, false, false, true>(p, st, ga);
    }
  }
  if constexpr (ALGO != WAHBA_PRECOMPUTED) {
    if (lpf) return comp ? launch_replay<ALGO, true, true, true, false, false, true, true>(p, use_tma, st, ga) : launch_replay<ALGO, true, true, false, false, false, true, true>(p, use_tma, st, ga);
  }
  return comp ? launch_replay<ALGO, false, true, true, false, false, true, true>(p, use_tma, st, ga) : launch_replay<ALGO, false, true, false, false, false, true, true>(p, use_tma, st, ga);
}

int launch_gated_algo(const ReplayParams& p, const GateArgs& ga, int algo, bool lpf, bool use_tma, bool packed, int innov_model,
                      cudaStream_t st) {
  if (algo == POSEKF_WAHBA_QR2) return launch_gated<WAHBA_QR2>(p, ga, lpf, use_tma, packed, innov_model, st);
  if (algo == POSEKF_WAHBA_PRECOMPUTED) return launch_gated<WAHBA_PRECOMPUTED>(p, ga, lpf, use_tma, packed, innov_model, st);
  if (algo == POSEKF_WAHBA_JACOBI) return launch_gated<WAHBA_JACOBI>(p, ga, lpf, use_tma, packed, innov_model, st);
  return POSEKF_EINVAL;
}

// Launches with general Q and R matrices (posekf_replay_general_f32): the scalar BATCH kernels with GEN, which step
// exactly as without BATCH when dt_cols and n_valid are null, with AUX (per-step outputs checked per pointer), on the
// launch's staging (the TMA kernel for a packed staging: the packed kernel has no GEN twin, its 124-168 registers leave
// no room for the 16 of Q and R at 3 CTAs per SM).  Plain variant only, no innovation sums, no gate.
template <int ALGO>
int launch_general(const ReplayParams& p, const GenQRArgs& gq, bool lpf, bool use_tma, cudaStream_t st) {
  if constexpr (ALGO != WAHBA_PRECOMPUTED) {
    if (lpf) return launch_replay<ALGO, true, true, false, false, false, true, false, true>(p, use_tma, st, gq);
  }
  return launch_replay<ALGO, false, true, false, false, false, true, false, true>(p, use_tma, st, gq);
}

int launch_general_algo(const ReplayParams& p, const GenQRArgs& gq, int algo, bool lpf, bool use_tma, cudaStream_t st) {
  if (algo == POSEKF_WAHBA_QR2) return launch_general<WAHBA_QR2>(p, gq, lpf, use_tma, st);
  if (algo == POSEKF_WAHBA_PRECOMPUTED) return launch_general<WAHBA_PRECOMPUTED>(p, gq, lpf, use_tma, st);
  if (algo == POSEKF_WAHBA_JACOBI) return launch_general<WAHBA_JACOBI>(p, gq, lpf, use_tma, st);
  return POSEKF_EINVAL;
}

// Launches with per-step innovation output (posekf_replay_innovation_steps_f32): the scalar BATCH kernels with INNOV
// (the statistic is needed whether or not the sums are) and AUX, gated or not, on the launch's staging.  A packed staging
// runs the scalar TMA kernel with the same bits (the packed kernel has no per-step-output twin; DESIGN.md section 5,
// f11).  ga: the pack's GateArgs (gated launches) and the InnovStepArgs.
template <int ALGO, bool TAN, bool GATE, typename... GA>
int launch_innov_steps(const ReplayParams& p, bool lpf, bool use_tma, cudaStream_t st, const GA&... ga) {
  const bool comp = p.state_x_lo != nullptr;
  if constexpr (ALGO != WAHBA_PRECOMPUTED) {
    if (lpf) return comp ? launch_replay<ALGO, true, true, true, true, TAN, true, GATE>(p, use_tma, st, ga...)
                         : launch_replay<ALGO, true, true, false, true, TAN, true, GATE>(p, use_tma, st, ga...);
  }
  return comp ? launch_replay<ALGO, false, true, true, true, TAN, true, GATE>(p, use_tma, st, ga...)
              : launch_replay<ALGO, false, true, false, true, TAN, true, GATE>(p, use_tma, st, ga...);
}

template <int ALGO>
int launch_innov_steps_model(const ReplayParams& p, const GateArgs* gate, const InnovStepArgs& ia, bool lpf, bool use_tma,
                             int innov_model, cudaStream_t st) {
  const bool tan = innov_model == POSEKF_INNOV_TANGENT;
  if (gate) return tan ? launch_innov_steps<ALGO, true, true>(p, lpf, use_tma, st, *gate, ia)
                       : launch_innov_steps<ALGO, false, true>(p, lpf, use_tma, st, *gate, ia);
  return tan ? launch_innov_steps<ALGO, true, false>(p, lpf, use_tma, st, ia) : launch_innov_steps<ALGO, false, false>(p, lpf, use_tma, st, ia);
}

int launch_innov_steps_algo(const ReplayParams& p, const GateArgs* gate, const InnovStepArgs& ia, int algo, bool lpf, bool use_tma,
                            int innov_model, cudaStream_t st) {
  if (algo == POSEKF_WAHBA_QR2) return launch_innov_steps_model<WAHBA_QR2>(p, gate, ia, lpf, use_tma, innov_model, st);
  if (algo == POSEKF_WAHBA_PRECOMPUTED) return launch_innov_steps_model<WAHBA_PRECOMPUTED>(p, gate, ia, lpf, use_tma, innov_model, st);
  if (algo == POSEKF_WAHBA_JACOBI) return launch_innov_steps_model<WAHBA_JACOBI>(p, gate, ia, lpf, use_tma, innov_model, st);
  return POSEKF_EINVAL;
}

// innov_model: POSEKF_INNOV_* of the sums in p.innov_acc (read only when it is set, or with steps).  gate: run the gated
// kernels with these arguments (null: the ungated ones).  gen: run the general-matrix kernels with these matrices.
// steps: run the innovation-steps kernels, which write the per-step terms there (with gen: the general-matrix kernels
// with the innovation terms, whose output there may be null).
int replay_dispatch(const ReplayParams& p, int algo, int staging, int innov_model, cudaStream_t st, const GateArgs* gate = nullptr,
                    const GenQRArgs* gen = nullptr, const InnovStepArgs* steps = nullptr) {
  const bool lpf = (p.alpha_acc >= 0.f) || (p.alpha_mag >= 0.f);
  bool use_tma, packed = false;
  if (staging == POSEKF_STAGE_LDG) use_tma = false;
  else if (staging == POSEKF_STAGE_TMA) { if (!tma_eligible(p)) return POSEKF_EALIGN; use_tma = true; }
  else if (staging == POSEKF_STAGE_TMA_PACKED) {
    if (!tma_eligible(p) || !packed_eligible(p) || algo == POSEKF_WAHBA_JACOBI) return POSEKF_EALIGN;
    use_tma = packed = true;
  } else if (staging == POSEKF_STAGE_AUTO) {
    use_tma = tma_eligible(p);
    packed = use_tma && kAutoPrefersPacked && algo != POSEKF_WAHBA_JACOBI && packed_eligible(p);
  } else return POSEKF_EINVAL;
  const bool batch = p.dt_cols != nullptr || p.n_valid != nullptr;
  int rc = gen ? (steps ? launch_general_innov_algo(p, *gen, gate, *steps, algo, lpf, use_tma, innov_model, st)
                        : launch_general_algo(p, *gen, algo, lpf, use_tma, st))
           : steps ? launch_innov_steps_algo(p, gate, *steps, algo, lpf, use_tma, innov_model, st)
           : gate ? launch_gated_algo(p, *gate, algo, lpf, use_tma, packed, innov_model, st)
                : batch ? launch_kernels<true>(p, algo, lpf, use_tma, packed, innov_model, st)
                        : launch_kernels<false>(p, algo, lpf, use_tma, packed, innov_model, st);
  // (held steps of a batched launch carry flip byte 0, which the fix-up leaves alone)
  if (rc == 0 && p.out_flip && p.T > 0 && algo == POSEKF_WAHBA_QR2 && !lpf) {
    // the flip-mask bytes the kernel marked as float32 ties of the reference's sign rule are settled in float64
    const FlipFixupParams fp{p.N, p.T, p.Ns, p.streams, p.acc_ref, p.mag_ref, p.out_flip};
    const int64_t words = (p.N * p.T + 3) / 4;
    flip_fixup_kernel<<<blocks_for(words, 256), 256, 0, st>>>(fp);
    rc = launch_status();
  }
  return rc;
}

// Entry points that take a device ordinal switch to it for their own work and put the caller's current device back on
// every exit path (the caller may be a torch process whose notion of "current device" must not change behind its back).
struct DeviceGuard {
  int prev = -1;
  cudaError_t status;
  explicit DeviceGuard(int device) {
    status = cudaGetDevice(&prev);
    if (status == cudaSuccess && prev != device) status = cudaSetDevice(device);
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

}  // namespace

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

const char* posekf_version(void) { return "posekf_b200 0.2 sm_100a"; }

}  // extern "C"

namespace {
// Validation and dispatch shared by posekf_replay_f32, posekf_replay_innovation(_ex)_f32, posekf_replay_batch_f32,
// posekf_replay_gated_f32 and posekf_replay_general_f32 (innov_acc null: the first; dt_cols and n_valid null: the first
// three; gate: the gated one; gen: the general one, whose q_scale and r_scale are null).
// innov_model: POSEKF_INNOV_FULL or POSEKF_INNOV_TANGENT (checked by the caller).
int replay_entry(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams, const float* dt,
                 int dt_per_step, const float* acc_ref, const float* mag_ref, const float* q_scale,
                 const float* r_scale, float lpf_alpha_acc, float lpf_alpha_mag, float* state_x, float* state_x_lo,
                 float* state_p, float* state_lpf, float* out_traj, uint8_t* out_flip, const float* truth, float* loss_acc,
                 float* innov_acc, int innov_model, int wahba_algo, int staging, int state_flags, void* stream,
                 const float* dt_cols = nullptr, const int32_t* n_valid = nullptr, bool gate = false, float gate_nis3 = 0.f,
                 int32_t* gate_count = nullptr, uint8_t* out_gated = nullptr, const GenQRArgs* gen = nullptr,
                 const InnovStepArgs* steps = nullptr) {
  if (dt_cols && !dt) { dt = dt_cols; dt_per_step = 0; }    // (the kernels read dt[0] unconditionally; it is unused then)
  if (n_filters < 0 || n_steps < 0 || n_streams <= 0 && n_filters > 0) return POSEKF_EINVAL;
  if (state_flags & ~(POSEKF_STATE_IN_FILTER_FRAME | POSEKF_STATE_OUT_FILTER_FRAME)) return POSEKF_EINVAL;
  if (n_filters == 0) return 0;
  if (n_steps == 0) {
    // nothing to replay; a launch is still needed when the state has to change frames
    const bool in_f = state_flags & POSEKF_STATE_IN_FILTER_FRAME, out_f = state_flags & POSEKF_STATE_OUT_FILTER_FRAME;
    if (in_f == out_f || wahba_algo == POSEKF_WAHBA_PRECOMPUTED) return 0;
    if (!acc_ref || !mag_ref || (!gen && (!q_scale || !r_scale)) || !state_x || !state_p) return POSEKF_EINVAL;
    if (n_streams > n_filters || (n_filters % n_streams) != 0) return POSEKF_EINVAL;
    staging = POSEKF_STAGE_LDG;
  } else if (!streams || !dt) return POSEKF_EINVAL;
  if (!acc_ref || !mag_ref || (!gen && (!q_scale || !r_scale)) || !state_x || !state_p) return POSEKF_EINVAL;
  if (n_streams > n_filters || (n_filters % n_streams) != 0) return POSEKF_EINVAL;
  const bool lpf = lpf_alpha_acc >= 0.f || lpf_alpha_mag >= 0.f;
  if (lpf && !state_lpf) return POSEKF_EINVAL;
  if (wahba_algo < POSEKF_WAHBA_QR2 || wahba_algo > POSEKF_WAHBA_PRECOMPUTED) return POSEKF_EINVAL;
  if (lpf && wahba_algo == POSEKF_WAHBA_PRECOMPUTED) return POSEKF_EINVAL;   // the low-pass belongs to the stream builder
  if ((n_filters + kThreads - 1) / kThreads > 0x7fffffffLL || n_steps > 0x7fffffffLL) return POSEKF_EINVAL;
  if (out_traj && (reinterpret_cast<uintptr_t>(out_traj) & 15) != 0) return POSEKF_EALIGN;
  if (truth && (!loss_acc || (reinterpret_cast<uintptr_t>(truth) & 15) != 0)) return truth && !loss_acc ? POSEKF_EINVAL : POSEKF_EALIGN;
  if ((reinterpret_cast<uintptr_t>(innov_acc) & 3) != 0) return POSEKF_EALIGN;
  if ((reinterpret_cast<uintptr_t>(dt_cols) & 3) != 0 || (reinterpret_cast<uintptr_t>(n_valid) & 3) != 0) return POSEKF_EALIGN;
  if ((reinterpret_cast<uintptr_t>(gate_count) & 3) != 0) return POSEKF_EALIGN;
  ReplayParams p;
  p.N = n_filters; p.T = n_steps; p.Ns = n_streams; p.streams = streams; p.dt = dt; p.dt_per_step = dt_per_step;
  p.acc_ref = acc_ref; p.mag_ref = mag_ref; p.q_scale = q_scale; p.r_scale = r_scale;
  p.alpha_acc = lpf_alpha_acc; p.alpha_mag = lpf_alpha_mag;
  p.state_x = state_x; p.state_x_lo = state_x_lo; p.state_p = state_p; p.state_lpf = state_lpf; p.out_traj = out_traj; p.out_flip = out_flip;
  p.truth = truth; p.loss_acc = loss_acc;
  p.innov_acc = n_steps > 0 ? innov_acc : nullptr;     // (a frame conversion has no step to add)
  p.state_flags = state_flags;
  p.dt_cols = n_steps > 0 ? dt_cols : nullptr;
  p.n_valid = n_steps > 0 ? n_valid : nullptr;
  const GateArgs ga{gate_nis3, gate_count, out_gated};
  return replay_dispatch(p, wahba_algo, staging, innov_model, (cudaStream_t)stream, gate && n_steps > 0 ? &ga : nullptr, gen,
                         n_steps > 0 ? steps : nullptr);
}
}  // namespace

extern "C" {

int posekf_replay_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams, const float* dt,
                      int dt_per_step, const float* acc_ref, const float* mag_ref, const float* q_scale,
                      const float* r_scale, float lpf_alpha_acc, float lpf_alpha_mag, float* state_x, float* state_x_lo,
                      float* state_p, float* state_lpf, float* out_traj, uint8_t* out_flip, const float* truth, float* loss_acc,
                      int wahba_algo, int staging, int state_flags, void* stream) {
  return replay_entry(n_filters, n_steps, streams, n_streams, dt, dt_per_step, acc_ref, mag_ref, q_scale, r_scale, lpf_alpha_acc,
                      lpf_alpha_mag, state_x, state_x_lo, state_p, state_lpf, out_traj, out_flip, truth, loss_acc, nullptr,
                      POSEKF_INNOV_FULL, wahba_algo, staging, state_flags, stream);
}

int posekf_replay_innovation_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams, const float* dt,
                                 int dt_per_step, const float* acc_ref, const float* mag_ref, const float* q_scale,
                                 const float* r_scale, float lpf_alpha_acc, float lpf_alpha_mag, float* state_x,
                                 float* state_x_lo, float* state_p, float* state_lpf, float* out_traj, uint8_t* out_flip,
                                 const float* truth, float* loss_acc, float* innov_acc, int wahba_algo, int staging,
                                 int state_flags, void* stream) {
  if (!innov_acc) return POSEKF_EINVAL;
  return replay_entry(n_filters, n_steps, streams, n_streams, dt, dt_per_step, acc_ref, mag_ref, q_scale, r_scale, lpf_alpha_acc,
                      lpf_alpha_mag, state_x, state_x_lo, state_p, state_lpf, out_traj, out_flip, truth, loss_acc, innov_acc,
                      POSEKF_INNOV_FULL, wahba_algo, staging, state_flags, stream);
}

int posekf_replay_innovation_ex_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams,
                                    const float* dt, int dt_per_step, const float* acc_ref, const float* mag_ref,
                                    const float* q_scale, const float* r_scale, float lpf_alpha_acc, float lpf_alpha_mag,
                                    float* state_x, float* state_x_lo, float* state_p, float* state_lpf, float* out_traj,
                                    uint8_t* out_flip, const float* truth, float* loss_acc, float* innov_acc, int innov_model,
                                    int wahba_algo, int staging, int state_flags, void* stream) {
  if (!innov_acc || (innov_model != POSEKF_INNOV_FULL && innov_model != POSEKF_INNOV_TANGENT)) return POSEKF_EINVAL;
  return replay_entry(n_filters, n_steps, streams, n_streams, dt, dt_per_step, acc_ref, mag_ref, q_scale, r_scale, lpf_alpha_acc,
                      lpf_alpha_mag, state_x, state_x_lo, state_p, state_lpf, out_traj, out_flip, truth, loss_acc, innov_acc,
                      innov_model, wahba_algo, staging, state_flags, stream);
}

int posekf_replay_batch_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams, const float* dt,
                            int dt_per_step, const float* acc_ref, const float* mag_ref, const float* q_scale,
                            const float* r_scale, float lpf_alpha_acc, float lpf_alpha_mag, float* state_x, float* state_x_lo,
                            float* state_p, float* state_lpf, float* out_traj, uint8_t* out_flip, const float* truth,
                            float* loss_acc, float* innov_acc, int innov_model, int wahba_algo, int staging, int state_flags,
                            void* stream, const float* dt_cols, const int32_t* n_valid) {
  if (innov_model != POSEKF_INNOV_FULL && innov_model != POSEKF_INNOV_TANGENT) return POSEKF_EINVAL;
  return replay_entry(n_filters, n_steps, streams, n_streams, dt, dt_per_step, acc_ref, mag_ref, q_scale, r_scale, lpf_alpha_acc,
                      lpf_alpha_mag, state_x, state_x_lo, state_p, state_lpf, out_traj, out_flip, truth, loss_acc, innov_acc,
                      innov_model, wahba_algo, staging, state_flags, stream, dt_cols, n_valid);
}

int posekf_replay_gated_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams, const float* dt,
                            int dt_per_step, const float* acc_ref, const float* mag_ref, const float* q_scale,
                            const float* r_scale, float lpf_alpha_acc, float lpf_alpha_mag, float* state_x, float* state_x_lo,
                            float* state_p, float* state_lpf, float* out_traj, uint8_t* out_flip, const float* truth,
                            float* loss_acc, float* innov_acc, int innov_model, int wahba_algo, int staging, int state_flags,
                            void* stream, const float* dt_cols, const int32_t* n_valid, float gate_nis3, int32_t* gate_count,
                            uint8_t* out_gated) {
  if (innov_model != POSEKF_INNOV_FULL && innov_model != POSEKF_INNOV_TANGENT) return POSEKF_EINVAL;
  if (gate_nis3 != gate_nis3) return POSEKF_EINVAL;      // NaN: no decision could ever be made with it
  return replay_entry(n_filters, n_steps, streams, n_streams, dt, dt_per_step, acc_ref, mag_ref, q_scale, r_scale, lpf_alpha_acc,
                      lpf_alpha_mag, state_x, state_x_lo, state_p, state_lpf, out_traj, out_flip, truth, loss_acc, innov_acc,
                      innov_model, wahba_algo, staging, state_flags, stream, dt_cols, n_valid, true, gate_nis3, gate_count,
                      out_gated);
}

int posekf_replay_innovation_steps_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams,
                                       const float* dt, int dt_per_step, const float* acc_ref, const float* mag_ref,
                                       const float* q_scale, const float* r_scale, float lpf_alpha_acc, float lpf_alpha_mag,
                                       float* state_x, float* state_x_lo, float* state_p, float* state_lpf, float* out_traj,
                                       uint8_t* out_flip, const float* truth, float* loss_acc, float* innov_acc,
                                       int innov_model, int wahba_algo, int staging, int state_flags, void* stream,
                                       const float* dt_cols, const int32_t* n_valid, float gate_nis3, int32_t* gate_count,
                                       uint8_t* out_gated, float* out_innov, int64_t innov_plane_stride) {
  if (innov_model != POSEKF_INNOV_FULL && innov_model != POSEKF_INNOV_TANGENT) return POSEKF_EINVAL;
  if (gate_nis3 != gate_nis3) return POSEKF_EINVAL;
  if (n_filters < 0 || n_steps < 0) return POSEKF_EINVAL;
  if (n_filters > 0 && n_steps > 0) {     // (an empty launch writes nothing: its buffer may be NULL, as torch's empty tensors are)
    if (!out_innov || n_steps > INT64_MAX / n_filters || innov_plane_stride < n_filters * n_steps) return POSEKF_EINVAL;
  }
  if ((reinterpret_cast<uintptr_t>(out_innov) & 3) != 0) return POSEKF_EALIGN;
  // +inf with no gate buffer decides nothing and records nothing: the ungated kernels (the same bits)
  const bool gate = !(gate_nis3 == INFINITY && !gate_count && !out_gated);
  const InnovStepArgs ia{out_innov, innov_plane_stride};
  return replay_entry(n_filters, n_steps, streams, n_streams, dt, dt_per_step, acc_ref, mag_ref, q_scale, r_scale, lpf_alpha_acc,
                      lpf_alpha_mag, state_x, state_x_lo, state_p, state_lpf, out_traj, out_flip, truth, loss_acc, innov_acc,
                      innov_model, wahba_algo, staging, state_flags, stream, dt_cols, n_valid, gate, gate_nis3, gate_count,
                      out_gated, nullptr, &ia);
}

int posekf_replay_general_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams, const float* dt,
                              int dt_per_step, const float* acc_ref, const float* mag_ref, const float* q_tri, int64_t nq,
                              const float* r_tri, int64_t nr, float lpf_alpha_acc, float lpf_alpha_mag, float* state_x,
                              float* state_x_lo, float* state_p, float* state_lpf, float* out_traj, uint8_t* out_flip,
                              const float* truth, float* loss_acc, float* innov_acc, int innov_model, int wahba_algo,
                              int staging, int state_flags, void* stream, const float* dt_cols, const int32_t* n_valid) {
  if (innov_model != POSEKF_INNOV_FULL && innov_model != POSEKF_INNOV_TANGENT) return POSEKF_EINVAL;
  if (innov_acc || state_x_lo) return POSEKF_EINVAL;     // no innovation sums, no precise variant with general matrices
  if (n_filters > 0 && (!q_tri || !r_tri || (nq != 1 && nq != n_filters) || (nr != 1 && nr != n_filters))) return POSEKF_EINVAL;
  if ((reinterpret_cast<uintptr_t>(q_tri) & 3) != 0 || (reinterpret_cast<uintptr_t>(r_tri) & 3) != 0) return POSEKF_EALIGN;
  const GenQRArgs gq{q_tri, nq, r_tri, nr};
  return replay_entry(n_filters, n_steps, streams, n_streams, dt, dt_per_step, acc_ref, mag_ref, nullptr, nullptr, lpf_alpha_acc,
                      lpf_alpha_mag, state_x, nullptr, state_p, state_lpf, out_traj, out_flip, truth, loss_acc, nullptr,
                      innov_model, wahba_algo, staging, state_flags, stream, dt_cols, n_valid, false, 0.f, nullptr, nullptr,
                      &gq);
}

int posekf_replay_general_innovation_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams,
                                         const float* dt, int dt_per_step, const float* acc_ref, const float* mag_ref,
                                         const float* q_tri, int64_t nq, const float* r_tri, int64_t nr, float lpf_alpha_acc,
                                         float lpf_alpha_mag, float* state_x, float* state_x_lo, float* state_p,
                                         float* state_lpf, float* out_traj, uint8_t* out_flip, const float* truth,
                                         float* loss_acc, float* innov_acc, int innov_model, int wahba_algo, int staging,
                                         int state_flags, void* stream, const float* dt_cols, const int32_t* n_valid,
                                         float gate_nis3, int32_t* gate_count, uint8_t* out_gated, float* out_innov,
                                         int64_t innov_plane_stride) {
  if (innov_model != POSEKF_INNOV_FULL && innov_model != POSEKF_INNOV_TANGENT) return POSEKF_EINVAL;
  if (gate_nis3 != gate_nis3) return POSEKF_EINVAL;
  if (state_x_lo) return POSEKF_EINVAL;                  // no precise variant with general matrices
  if (n_filters < 0 || n_steps < 0) return POSEKF_EINVAL;
  if (n_filters > 0 && (!q_tri || !r_tri || (nq != 1 && nq != n_filters) || (nr != 1 && nr != n_filters))) return POSEKF_EINVAL;
  if (out_innov && n_filters > 0 && n_steps > 0) {
    if (n_steps > INT64_MAX / n_filters || innov_plane_stride < n_filters * n_steps) return POSEKF_EINVAL;
  }
  if ((reinterpret_cast<uintptr_t>(q_tri) & 3) != 0 || (reinterpret_cast<uintptr_t>(r_tri) & 3) != 0) return POSEKF_EALIGN;
  if ((reinterpret_cast<uintptr_t>(out_innov) & 3) != 0) return POSEKF_EALIGN;
  const GenQRArgs gq{q_tri, nq, r_tri, nr};
  // +inf with no gate buffer decides nothing and records nothing: the ungated kernels (the same bits); a launch that
  // asks for no innovation output at all is the plain general replay
  const bool gate = !(gate_nis3 == INFINITY && !gate_count && !out_gated);
  const InnovStepArgs ia{out_innov, innov_plane_stride};
  const bool terms = innov_acc || out_innov || gate;
  return replay_entry(n_filters, n_steps, streams, n_streams, dt, dt_per_step, acc_ref, mag_ref, nullptr, nullptr, lpf_alpha_acc,
                      lpf_alpha_mag, state_x, nullptr, state_p, state_lpf, out_traj, out_flip, truth, loss_acc, innov_acc,
                      innov_model, wahba_algo, staging, state_flags, stream, dt_cols, n_valid, gate, gate_nis3, gate_count,
                      out_gated, &gq, terms ? &ia : nullptr);
}

// ---- host-buffer replay: workspace (device staging buffers, streams, events) ----------------------
struct HostWorkspace {
  int device = 0;
  int64_t N = 0, chunk_steps = 0;
  bool traj = false;
  cudaStream_t s_copy = nullptr, s_comp = nullptr, s_out = nullptr;
  cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr}, ev_traj[2] = {nullptr, nullptr},
              ev_tfree[2] = {nullptr, nullptr};
  float *d_in[2] = {nullptr, nullptr}, *d_traj[2] = {nullptr, nullptr};
  float *d_ref = nullptr, *d_qr = nullptr, *d_x = nullptr, *d_xlo = nullptr, *d_p = nullptr, *d_lpf = nullptr, *d_dt = nullptr;
};

static void host_ws_free(HostWorkspace* w) {
  if (!w) return;
  DeviceGuard guard(w->device);
  for (int i = 0; i < 2; ++i) {
    if (w->d_in[i]) cudaFree(w->d_in[i]);
    if (w->d_traj[i]) cudaFree(w->d_traj[i]);
    if (w->ev_in[i]) cudaEventDestroy(w->ev_in[i]);
    if (w->ev_free[i]) cudaEventDestroy(w->ev_free[i]);
    if (w->ev_traj[i]) cudaEventDestroy(w->ev_traj[i]);
    if (w->ev_tfree[i]) cudaEventDestroy(w->ev_tfree[i]);
  }
  float* ptrs[] = {w->d_ref, w->d_qr, w->d_x, w->d_xlo, w->d_p, w->d_lpf, w->d_dt};
  for (float* q : ptrs) if (q) cudaFree(q);
  if (w->s_copy) cudaStreamDestroy(w->s_copy);
  if (w->s_comp) cudaStreamDestroy(w->s_comp);
  if (w->s_out) cudaStreamDestroy(w->s_out);
  delete w;
}

int posekf_host_workspace_create(int device, int64_t n_filters, int64_t chunk_steps, int with_trajectory, void** out_ws) {
  if (!out_ws || n_filters <= 0) return POSEKF_EINVAL;
  *out_ws = nullptr;
  DeviceGuard guard(device);
  PKF_CUDA_TRY(guard.status);
  const int64_t N = n_filters;
  if (chunk_steps <= 0) {   // ~256 MiB per staging buffer: small enough that the first kernel starts after ~5 ms
    const int64_t bytes_per_step = (int64_t)kChannels * N * sizeof(float);
    chunk_steps = std::max<int64_t>(1, (int64_t)(256ll << 20) / bytes_per_step);
  }
  HostWorkspace* w = new HostWorkspace();
  w->device = device; w->N = N; w->chunk_steps = chunk_steps; w->traj = with_trajectory != 0;
#define WS_TRY(expr)                                                   \
  do {                                                                 \
    cudaError_t _e = (expr);                                           \
    if (_e != cudaSuccess) { host_ws_free(w); return (int)_e; }        \
  } while (0)
  WS_TRY(cudaStreamCreateWithFlags(&w->s_copy, cudaStreamNonBlocking));
  WS_TRY(cudaStreamCreateWithFlags(&w->s_comp, cudaStreamNonBlocking));
  WS_TRY(cudaStreamCreateWithFlags(&w->s_out, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) {
    WS_TRY(cudaEventCreateWithFlags(&w->ev_in[i], cudaEventDisableTiming));
    WS_TRY(cudaEventCreateWithFlags(&w->ev_free[i], cudaEventDisableTiming));
    WS_TRY(cudaEventCreateWithFlags(&w->ev_traj[i], cudaEventDisableTiming));
    WS_TRY(cudaEventCreateWithFlags(&w->ev_tfree[i], cudaEventDisableTiming));
    WS_TRY(cudaMalloc(&w->d_in[i], (size_t)chunk_steps * kChannels * N * sizeof(float)));
    if (w->traj) WS_TRY(cudaMalloc(&w->d_traj[i], (size_t)chunk_steps * 4 * N * sizeof(float)));
  }
  WS_TRY(cudaMalloc(&w->d_ref, (size_t)6 * N * sizeof(float)));
  WS_TRY(cudaMalloc(&w->d_qr, (size_t)2 * N * sizeof(float)));
  WS_TRY(cudaMalloc(&w->d_x, (size_t)4 * N * sizeof(float)));
  WS_TRY(cudaMalloc(&w->d_xlo, (size_t)4 * N * sizeof(float)));
  WS_TRY(cudaMalloc(&w->d_p, (size_t)10 * N * sizeof(float)));
  WS_TRY(cudaMalloc(&w->d_lpf, (size_t)6 * N * sizeof(float)));
  WS_TRY(cudaMalloc(&w->d_dt, sizeof(float)));
#undef WS_TRY
  *out_ws = w;
  return 0;
}

int posekf_host_workspace_destroy(void* ws) {
  host_ws_free(static_cast<HostWorkspace*>(ws));
  return 0;
}

int posekf_replay_host_f32(int64_t N, int64_t T, const float* streams_host, float dt, const float* acc_ref_host,
                           const float* mag_ref_host, const float* q_scale_host, const float* r_scale_host,
                           float lpf_alpha_acc, float lpf_alpha_mag, const float* x0_host, const float* p0_host,
                           float* out_x_host, float* out_p_host, float* out_traj_host, int64_t chunk_steps,
                           int wahba_algo, int precise, int device, void* workspace) {
  if (N <= 0 || T < 0 || !streams_host || !acc_ref_host || !mag_ref_host || !q_scale_host || !r_scale_host || !out_x_host)
    return POSEKF_EINVAL;
  // R = r I must be positive definite (the device state is P/r) and Q = q I positive semi-definite; NaN fails both tests
  for (int64_t n = 0; n < N; ++n)
    if (!(r_scale_host[n] > 0.f) || !(q_scale_host[n] >= 0.f)) return POSEKF_EINVAL;
  const bool traj = out_traj_host != nullptr;
  HostWorkspace* w = static_cast<HostWorkspace*>(workspace);
  bool own = false;
  if (w) {
    if (w->N != N || w->device != device || (traj && !w->traj)) return POSEKF_EINVAL;
  } else {
    void* tmp = nullptr;
    int rc0 = posekf_host_workspace_create(device, N, chunk_steps, traj ? 1 : 0, &tmp);
    if (rc0 != 0) return rc0;
    w = static_cast<HostWorkspace*>(tmp);
    own = true;
  }
  DeviceGuard guard(device);
  if (guard.status != cudaSuccess) { if (own) host_ws_free(w); return (int)guard.status; }
  chunk_steps = w->chunk_steps;
  const bool lpf = lpf_alpha_acc >= 0.f || lpf_alpha_mag >= 0.f;
  int rc = 0;
  cudaStream_t s_copy = w->s_copy, s_comp = w->s_comp, s_out = w->s_out;
  // on failure: nothing issued so far may still be reading the caller's host buffers when the call returns
  auto fail = [&](int code) {
    cudaStreamSynchronize(s_copy); cudaStreamSynchronize(s_comp); cudaStreamSynchronize(s_out);
    if (own) host_ws_free(w);
    return code;
  };
#define TRY(expr)                                          \
  do {                                                     \
    cudaError_t _e = (expr);                               \
    if (_e != cudaSuccess) return fail((int)_e);           \
  } while (0)
  float* d_ref = w->d_ref; float* d_qr = w->d_qr; float* d_x = w->d_x; float* d_p = w->d_p; float* d_dt = w->d_dt;
  float* d_lpf = lpf ? w->d_lpf : nullptr;
  float* d_xlo = precise ? w->d_xlo : nullptr;
  if (lpf) TRY(cudaMemsetAsync(d_lpf, 0, (size_t)6 * N * sizeof(float), s_comp));
  if (precise) TRY(cudaMemsetAsync(d_xlo, 0, (size_t)4 * N * sizeof(float), s_comp));
  TRY(cudaMemcpyAsync(d_ref, acc_ref_host, (size_t)3 * N * sizeof(float), cudaMemcpyHostToDevice, s_comp));
  TRY(cudaMemcpyAsync(d_ref + 3 * N, mag_ref_host, (size_t)3 * N * sizeof(float), cudaMemcpyHostToDevice, s_comp));
  TRY(cudaMemcpyAsync(d_qr, q_scale_host, (size_t)N * sizeof(float), cudaMemcpyHostToDevice, s_comp));
  TRY(cudaMemcpyAsync(d_qr + N, r_scale_host, (size_t)N * sizeof(float), cudaMemcpyHostToDevice, s_comp));
  // the first stream chunk is independent of the state set-up: start it right away
  const int64_t n_chunks = (T + chunk_steps - 1) / chunk_steps;
  auto issue_copy = [&](int64_t c) -> cudaError_t {
    const int b = (int)(c & 1);
    const int64_t t0 = c * chunk_steps, tc = std::min<int64_t>(chunk_steps, T - t0);
    cudaError_t e;
    if (c >= 2 && (e = cudaStreamWaitEvent(s_copy, w->ev_free[b], 0)) != cudaSuccess) return e;   // kernel of chunk c-2 done
    if ((e = cudaMemcpyAsync(w->d_in[b], streams_host + (size_t)t0 * kChannels * N, (size_t)tc * kChannels * N * sizeof(float),
                             cudaMemcpyHostToDevice, s_copy)) != cudaSuccess) return e;
    return cudaEventRecord(w->ev_in[b], s_copy);
  };
  if (n_chunks > 0) TRY(issue_copy(0));
  // initial state: X = [1,0,0,0], P = I4 (PKF/main_file.py:23,26) unless given; the device state holds P/r
  if (x0_host) TRY(cudaMemcpyAsync(d_x, x0_host, (size_t)4 * N * sizeof(float), cudaMemcpyHostToDevice, s_comp));
  if (p0_host) TRY(cudaMemcpyAsync(d_p, p0_host, (size_t)10 * N * sizeof(float), cudaMemcpyHostToDevice, s_comp));
  // (dt travels as a kernel argument: no asynchronous copy out of this function's stack frame)
  host_init_state_kernel<<<blocks_for(N, 256), 256, 0, s_comp>>>(N, x0_host != nullptr, p0_host != nullptr, d_qr + N, d_x, d_p, dt, d_dt);
  TRY(cudaPeekAtLastError());
  for (int64_t c = 0; c < n_chunks; ++c) {
    const int b = (int)(c & 1);
    const int64_t t0 = c * chunk_steps, tc = std::min<int64_t>(chunk_steps, T - t0);
    if (c + 1 < n_chunks) TRY(issue_copy(c + 1));                             // keep the copy engine one chunk ahead
    TRY(cudaStreamWaitEvent(s_comp, w->ev_in[b], 0));
    if (traj && c >= 2) TRY(cudaStreamWaitEvent(s_comp, w->ev_tfree[b], 0));  // D2H of chunk c-2 done with d_traj[b]
    // the state stays in the filter frame between chunks, so that chunking does not change a single bit
    const int frames = (c > 0 ? POSEKF_STATE_IN_FILTER_FRAME : 0) | (c + 1 < n_chunks ? POSEKF_STATE_OUT_FILTER_FRAME : 0);
    rc = posekf_replay_f32(N, tc, w->d_in[b], N, d_dt, 0, d_ref, d_ref + 3 * N, d_qr, d_qr + N, lpf_alpha_acc,
                           lpf_alpha_mag, d_x, d_xlo, d_p, d_lpf, traj ? w->d_traj[b] : nullptr, nullptr, nullptr, nullptr,
                           wahba_algo, POSEKF_STAGE_AUTO, frames, s_comp);
    if (rc != 0) return fail(rc);
    TRY(cudaEventRecord(w->ev_free[b], s_comp));
    if (traj) {
      TRY(cudaEventRecord(w->ev_traj[b], s_comp));
      TRY(cudaStreamWaitEvent(s_out, w->ev_traj[b], 0));
      TRY(cudaMemcpyAsync(out_traj_host + (size_t)t0 * 4 * N, w->d_traj[b], (size_t)tc * 4 * N * sizeof(float),
                          cudaMemcpyDeviceToHost, s_out));
      TRY(cudaEventRecord(w->ev_tfree[b], s_out));
    }
  }
  TRY(cudaMemcpyAsync(out_x_host, d_x, (size_t)4 * N * sizeof(float), cudaMemcpyDeviceToHost, s_comp));
  if (out_p_host) {
    host_unscale_p_kernel<<<blocks_for(N, 256), 256, 0, s_comp>>>(N, d_qr + N, d_p);     // P/r -> P
    TRY(cudaPeekAtLastError());
    TRY(cudaMemcpyAsync(out_p_host, d_p, (size_t)10 * N * sizeof(float), cudaMemcpyDeviceToHost, s_comp));
  }
  TRY(cudaStreamSynchronize(s_comp));
  TRY(cudaStreamSynchronize(s_out));
  TRY(cudaStreamSynchronize(s_copy));
#undef TRY
  if (own) host_ws_free(w);
  return 0;
}

#ifndef POSEKF_WAHBA2_WAVES
#define POSEKF_WAHBA2_WAVES 4
#endif
int posekf_wahba_f32(int64_t n, const float* acc_ref, const float* mag_ref, int ref_shared, const float* acc,
                     const float* mag, const float* k_acc, const float* k_mag, float k_acc_s, float k_mag_s,
                     int weights_from_acc, float* out_rot, float* out_quat, int wahba_algo, int jacobi_sweeps,
                     void* stream) {
  if (n < 0) return POSEKF_EINVAL;
  if (n == 0) return 0;
  if (!acc_ref || !mag_ref || !acc || !mag || (!out_rot && !out_quat) || ((k_acc == nullptr) != (k_mag == nullptr)))
    return POSEKF_EINVAL;
  WahbaParams p{n, acc_ref, mag_ref, ref_shared, acc, mag, k_acc, k_mag, k_acc_s, k_mag_s, weights_from_acc,
                out_rot, out_quat, jacobi_sweeps > 0 ? jacobi_sweeps : 6};
  cudaStream_t st = (cudaStream_t)stream;
  if (wahba_algo == POSEKF_WAHBA_QR2) {
    // two solves per thread (packed f32x2) when every [k][N] array can be read as float2
    bool packed = (n & 1) == 0;
    const void* ptrs[] = {acc, mag, k_acc, k_mag, out_rot, out_quat, ref_shared ? nullptr : acc_ref, ref_shared ? nullptr : mag_ref};
    for (const void* q : ptrs) packed = packed && (reinterpret_cast<uintptr_t>(q) & 7) == 0;
    if (packed) {
      // grid-stride loop with register prefetch inside: POSEKF_WAHBA2_WAVES x the CTAs that are resident at once
      // (4 waves measured best on B200: 145 G solves/s = 5.8 TB/s; one thread per pair was 128 G)
      int dev = 0, sms = 0, per_sm = 0;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wahba2_kernel, 256, 0);
      const int64_t need = blocks_for(n / 2, 256), resident = (int64_t)sms * (per_sm > 0 ? per_sm : 4) * POSEKF_WAHBA2_WAVES;
      wahba2_kernel<<<(unsigned)(need < resident ? need : resident), 256, 0, st>>>(p);
    }
    else wahba_kernel<WAHBA_QR2><<<blocks_for(n, 256), 256, 0, st>>>(p);
  }
  else if (wahba_algo == POSEKF_WAHBA_JACOBI) wahba_kernel<WAHBA_JACOBI><<<blocks_for(n, 256), 256, 0, st>>>(p);
  else return POSEKF_EINVAL;
  return launch_status();
}

int posekf_tracks_f32(int64_t n_filters, int64_t n_steps, const float* streams, int64_t n_streams, const float* dt,
                      int dt_per_step, const float* acc_ref, const float* mag_ref, float k_acc, float k_mag,
                      int weights_from_acc, float* gyro_state, float* out_gyro, float* out_wahba, int wahba_algo,
                      void* stream) {
  if (n_filters < 0 || n_steps < 0) return POSEKF_EINVAL;
  if (n_filters == 0 || n_steps == 0) return 0;
  if (!streams || !dt || n_streams <= 0 || n_streams > n_filters || (n_filters % n_streams) != 0) return POSEKF_EINVAL;
  if (!out_gyro && !out_wahba && !gyro_state) return POSEKF_EINVAL;
  if (out_wahba && (!acc_ref || !mag_ref)) return POSEKF_EINVAL;
  if (((reinterpret_cast<uintptr_t>(out_gyro) | reinterpret_cast<uintptr_t>(out_wahba)) & 15) != 0) return POSEKF_EALIGN;
  TracksParams p{n_filters, n_steps, n_streams, streams, dt, dt_per_step, acc_ref ? acc_ref : streams,
                 mag_ref ? mag_ref : streams, k_acc, k_mag, weights_from_acc, gyro_state, out_gyro, out_wahba};
  cudaStream_t st = (cudaStream_t)stream;
  // the Wahba-only track does not depend on its predecessors: with one stream per filter it runs packed (two filters
  // per thread), and the sequential kernel keeps the gyro-only track
  const bool packed_wahba = out_wahba && wahba_algo == POSEKF_WAHBA_QR2 && n_streams == n_filters && (n_filters & 1) == 0 &&
                            ((reinterpret_cast<uintptr_t>(streams) | reinterpret_cast<uintptr_t>(acc_ref) |
                              reinterpret_cast<uintptr_t>(mag_ref)) & 7) == 0;
  if (packed_wahba) {
    tracks_wahba2_kernel<<<blocks_for(n_filters / 2, 128), 128, 0, st>>>(p);
    if (int rc = launch_status()) return rc;
    if (!out_gyro && !gyro_state) return 0;
    p.out_wahba = nullptr;
  }
  if (wahba_algo == POSEKF_WAHBA_QR2) tracks_kernel<WAHBA_QR2><<<blocks_for(n_filters, 128), 128, 0, st>>>(p);
  else if (wahba_algo == POSEKF_WAHBA_JACOBI) tracks_kernel<WAHBA_JACOBI><<<blocks_for(n_filters, 128), 128, 0, st>>>(p);
  else return POSEKF_EINVAL;
  return launch_status();
}

int posekf_preprocess_f32(int64_t n_filters, int64_t n_steps, const float* gyro, const float* raw_prev,
                          const float* raw_next, const float* tspan, float lpf_alpha_acc, float lpf_alpha_mag,
                          float* lpf_state, float* out_streams, void* stream) {
  if (n_filters < 0 || n_steps < 0) return POSEKF_EINVAL;
  if (n_filters == 0 || n_steps == 0) return 0;
  if (!gyro || !raw_prev || !raw_next || !tspan || !out_streams) return POSEKF_EINVAL;
  if ((lpf_alpha_acc >= 0.f || lpf_alpha_mag >= 0.f) && !lpf_state) return POSEKF_EINVAL;
  PreprocessParams p{n_filters, n_steps, gyro, raw_prev, raw_next, tspan, lpf_alpha_acc, lpf_alpha_mag, lpf_state, out_streams};
  preprocess_kernel<<<blocks_for(n_filters, 256), 256, 0, (cudaStream_t)stream>>>(p);
  return launch_status();
}

int posekf_initial_values_f32(int64_t n_filters, int64_t n_samples, const float* samples, int normalize, float* out_mean,
                              float* out_var, void* stream) {
  if (n_filters < 0 || n_samples < 1) return POSEKF_EINVAL;
  if (n_filters == 0) return 0;
  if (!samples || !out_mean || (out_var && n_samples < 2)) return POSEKF_EINVAL;
  initial_values_kernel<<<blocks_for(n_filters, 256), 256, 0, (cudaStream_t)stream>>>(n_filters, n_samples, samples, normalize,
                                                                                        out_mean, out_var);
  return launch_status();
}

int posekf_align_events_f32(int64_t n_rec, int64_t k_init, const int64_t* gyro_t, const float* gyro_v, const int64_t* gyro_off,
                            const int64_t* acc_t, const float* acc_v, const int64_t* acc_off, const int64_t* mag_t,
                            const float* mag_v, const int64_t* mag_off, int64_t t_out, float* streams, float* dt_cols,
                            int32_t* lengths, float* acc_ref, float* mag_ref, void* stream) {
  if (n_rec < 0 || t_out < 0 || k_init < 1) return POSEKF_EINVAL;
  if (n_rec == 0) return 0;
  if (!gyro_t || !gyro_off || !acc_t || !acc_off || !mag_t || !mag_off || !lengths) return POSEKF_EINVAL;
  const bool query = streams == nullptr;
  if (!query && (!gyro_v || !acc_v || !mag_v || !dt_cols || !acc_ref || !mag_ref)) return POSEKF_EINVAL;
  const int64_t col_tiles = (n_rec + kAlignTile - 1) / kAlignTile, step_tiles = (t_out + kAlignTile - 1) / kAlignTile;
  if (blocks_for(n_rec, 256) > 0x7fffffffu || col_tiles * step_tiles > 0x7fffffffLL) return POSEKF_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  AlignParams p{n_rec, t_out, k_init, gyro_t, acc_t, mag_t, gyro_v, acc_v, mag_v, gyro_off, acc_off, mag_off, lengths, nullptr,
                acc_ref, mag_ref, streams, dt_cols};
  if (query) {
    align_bounds_kernel<<<blocks_for(n_rec, 256), 256, 0, st>>>(p);
    return launch_status();
  }
  // the step-0 gyro index and t_init of every recording, from the first kernel to the second (stream-ordered scratch)
  PKF_CUDA_TRY(cudaMallocAsync((void**)&p.bounds, (size_t)2 * n_rec * sizeof(int64_t), st));
  align_bounds_kernel<<<blocks_for(n_rec, 256), 256, 0, st>>>(p);
  int rc = launch_status();
  if (rc == 0 && t_out > 0) {
    align_events_kernel<<<(unsigned)(col_tiles * step_tiles), dim3(kAlignTile, kAlignWarps), 0, st>>>(p, col_tiles);
    rc = launch_status();
  }
  const cudaError_t e = cudaFreeAsync(p.bounds, st);
  return rc != 0 ? rc : (e == cudaSuccess ? 0 : (int)e);
}

int posekf_measurement_stream_f32(int64_t n_streams, int64_t n_steps, const float* streams, const float* acc_ref,
                                  const float* mag_ref, float lpf_alpha_acc, float lpf_alpha_mag, float* lpf_state,
                                  float* out_streams, int wahba_algo, void* stream) {
  if (n_streams < 0 || n_steps < 0) return POSEKF_EINVAL;
  if (n_streams == 0 || n_steps == 0) return 0;
  if (!streams || !acc_ref || !mag_ref || !out_streams) return POSEKF_EINVAL;
  if ((lpf_alpha_acc >= 0.f || lpf_alpha_mag >= 0.f) && !lpf_state) return POSEKF_EINVAL;
  MeasStreamParams p{n_streams, n_steps, streams, acc_ref, mag_ref, lpf_alpha_acc, lpf_alpha_mag, lpf_state, out_streams};
  cudaStream_t st = (cudaStream_t)stream;
  // time is split over gridDim.y when the samples are independent (no low-pass): aim at ~2 Mi threads
  const bool sequential = lpf_alpha_acc >= 0.f || lpf_alpha_mag >= 0.f;
  int64_t ty = sequential ? 1 : ((int64_t)2 << 20) / (blocks_for(n_streams, 128) * (int64_t)128);
  ty = ty < 1 ? 1 : (ty > n_steps ? n_steps : (ty > 65535 ? 65535 : ty));
  const dim3 grid(blocks_for(n_streams, 128), (unsigned)ty);
  if (wahba_algo == POSEKF_WAHBA_QR2) measurement_stream_kernel<WAHBA_QR2><<<grid, 128, 0, st>>>(p);
  else if (wahba_algo == POSEKF_WAHBA_JACOBI) measurement_stream_kernel<WAHBA_JACOBI><<<grid, 128, 0, st>>>(p);
  else return POSEKF_EINVAL;
  if (int rc = launch_status()) return rc;
  if (!sequential && streams != out_streams) {     // float32 ties of the reference's sign rule, re-decided in float64
    meas_fixup_kernel<<<blocks_for(n_streams * n_steps, 256), 256, 0, st>>>(p);
  }
  return launch_status();
}

int posekf_traj2rpy_f32(int64_t m, const float* traj, float* out_rpy_deg, void* stream) {
  if (m < 0) return POSEKF_EINVAL;
  if (m == 0) return 0;
  if (!traj || !out_rpy_deg) return POSEKF_EINVAL;
  if ((reinterpret_cast<uintptr_t>(traj) & 15) != 0) return POSEKF_EALIGN;
  traj2rpy_kernel<<<blocks_for(m, 256), 256, 0, (cudaStream_t)stream>>>(m, reinterpret_cast<const float4*>(traj), out_rpy_deg);
  return launch_status();
}

int posekf_rot2quat_f32(int64_t n, const float* rot, float* out_quat, void* stream) {
  if (n < 0) return POSEKF_EINVAL;
  if (n == 0) return 0;
  if (!rot || !out_quat) return POSEKF_EINVAL;
  rot2quat_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(n, rot, out_quat);
  return launch_status();
}

int posekf_predict_f32(int64_t n, const float* gyro, const float* dt, int dt_shared, const float* x, const float* p,
                       const float* q_mat, const float* r_mat, const float* q_scale, const float* r_scale, float* out_z,
                       float* out_p, float* out_k, void* stream) {
  if (n < 0) return POSEKF_EINVAL;
  if (n == 0) return 0;
  if (!gyro || !dt || !x || !p || !q_mat || !r_mat || !out_z || !out_p || !out_k) return POSEKF_EINVAL;
  PredictParams a{n, gyro, dt, dt_shared, x, p, q_mat, r_mat, q_scale, r_scale, out_z, out_p, out_k};
  predict_kernel<<<blocks_for(n, 128), 128, 0, (cudaStream_t)stream>>>(a);
  return launch_status();
}

int posekf_correct_f32(int64_t n, const float* mag, const float* acc, const float* acc_ref, const float* mag_ref,
                       int ref_shared, const float* z, const float* p, const float* k, float* out_x, float* out_p,
                       uint8_t* out_flip, float* out_meas, int wahba_algo, void* stream) {
  if (n < 0) return POSEKF_EINVAL;
  if (n == 0) return 0;
  if (!mag || !acc || !acc_ref || !mag_ref || !z || !p || !k || !out_x || !out_p) return POSEKF_EINVAL;
  CorrectParams a{n, mag, acc, acc_ref, mag_ref, ref_shared, z, p, k, out_x, out_p, out_flip, out_meas};
  cudaStream_t st = (cudaStream_t)stream;
  if (wahba_algo == POSEKF_WAHBA_QR2) correct_kernel<WAHBA_QR2><<<blocks_for(n, 128), 128, 0, st>>>(a);
  else if (wahba_algo == POSEKF_WAHBA_JACOBI) correct_kernel<WAHBA_JACOBI><<<blocks_for(n, 128), 128, 0, st>>>(a);
  else return POSEKF_EINVAL;
  return launch_status();
}

int posekf_rk4_f32(int64_t n, const float* q, const float* dt, int dt_shared, const float* w, float* out_q, void* stream) {
  if (n < 0) return POSEKF_EINVAL;
  if (n == 0) return 0;
  if (!q || !dt || !w || !out_q) return POSEKF_EINVAL;
  rk4_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(n, q, dt, dt_shared, w, out_q);
  return launch_status();
}

int posekf_jacobians_f32(int64_t n, const float* w, float* out_a, const float* q, float* out_b, void* stream) {
  if (n < 0) return POSEKF_EINVAL;
  if (n == 0) return 0;
  if (!((w && out_a) || (q && out_b))) return POSEKF_EINVAL;
  jacobians_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(n, w, out_a, q, out_b);
  return launch_status();
}

int posekf_comparator_f32(int64_t n, const float* q1, const float* q2, float* out, void* stream) {
  if (n < 0) return POSEKF_EINVAL;
  if (n == 0) return 0;
  if (!q1 || !q2 || !out) return POSEKF_EINVAL;
  comparator_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(n, q1, q2, out);
  return launch_status();
}

int posekf_lowpass_f32(int64_t n, int64_t n_steps, const float* x, float alpha, float* state, float* out, void* stream) {
  if (n < 0 || n_steps < 0) return POSEKF_EINVAL;
  if (n == 0 || n_steps == 0) return 0;
  if (!x || !state || !out) return POSEKF_EINVAL;
  lowpass_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(n, n_steps, x, alpha, state, out);
  return launch_status();
}

int posekf_quat2rpy_f32(int64_t n, const float* q, float* out_rpy_deg, void* stream) {
  if (n < 0) return POSEKF_EINVAL;
  if (n == 0) return 0;
  if (!q || !out_rpy_deg) return POSEKF_EINVAL;
  quat2rpy_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(n, q, out_rpy_deg);
  return launch_status();
}

int posekf_norm_f32(int64_t n, int k, const float* v, float* out, void* stream) {
  if (n < 0 || k < 0) return POSEKF_EINVAL;
  if (n == 0) return 0;
  if (!v || !out) return POSEKF_EINVAL;
  norm_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(n, k, v, out);
  return launch_status();
}

int posekf_copy_async(void* dst, const void* src, int64_t bytes, int to_device, void* stream) {
  if (bytes < 0 || (bytes > 0 && (!dst || !src))) return POSEKF_EINVAL;
  if (bytes == 0) return 0;
  PKF_CUDA_TRY(cudaMemcpyAsync(dst, src, (size_t)bytes, to_device ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost,
                               (cudaStream_t)stream));
  return 0;
}

int posekf_stream_sync(void* stream) {
  PKF_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  return 0;
}

int posekf_fp32_peak_tflops(int device, double* out_tflops, double* out_ms) {
  if (!out_tflops) return POSEKF_EINVAL;
  DeviceGuard guard(device);
  PKF_CUDA_TRY(guard.status);
  cudaDeviceProp prop;
  PKF_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  const int blocks = prop.multiProcessorCount * 8;
  float* out = nullptr;
  PKF_CUDA_TRY(cudaMalloc(&out, (size_t)blocks * 256 * sizeof(float)));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int w = 0; w < 3; ++w) fp32_probe_kernel<<<blocks, 256>>>(out, 1.0001f, 1e-4f);
  cudaDeviceSynchronize();
  float best = 1e30f;
  for (int r = 0; r < 5; ++r) {
    cudaEventRecord(e0);
    fp32_probe_kernel<<<blocks, 256>>>(out, 1.0001f, 1e-4f);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms;
    cudaEventElapsedTime(&ms, e0, e1);
    best = std::min(best, ms);
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(out);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  const double flops = 2.0 * kProbeIters * kProbeAcc * (double)blocks * 256;
  *out_tflops = flops / (best * 1e-3) / 1e12;
  if (out_ms) *out_ms = best;
  return 0;
}

}  // extern "C"
