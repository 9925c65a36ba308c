// replay_kernels.cuh -- the fused replay kernels (T Prediction+Correction steps for N filters per launch):
//   replay_ldg_kernel   one filter per thread, coalesced LDG with a one-step register prefetch
//   replay_tma_kernel   one filter per thread, TMA/mbarrier ring of [steps][9][128] tiles
//   replay_tma2_kernel  TWO filters per thread in packed f32x2 lanes (FFMA2), same ring  -- the default
// Replaces the loop body of "Python Kalman Filter/main_file.py":38-47 (see include/posekf.h).
#pragma once
#include <type_traits>
#include "device_util.cuh"

namespace pkf_dev {

struct ReplayParams {
  int64_t N, T, Ns;
  const float* streams;
  const float* dt;
  int dt_per_step;
  const float* acc_ref;
  const float* mag_ref;
  const float* q_scale;
  const float* r_scale;
  float alpha_acc, alpha_mag;
  float* state_x;
  float* state_x_lo;    // [4][N] low-order part of the two-float state (compensated variant), or null
  float* state_p;
  float* state_lpf;
  float* out_traj;
  uint8_t* out_flip;
  const float* truth;   // [T][Ns][4] reference track for the tuning objective, or null
  float* loss_acc;      // [N] in/out: sum over steps of 1 - (x . truth)^2
  int state_flags;      // POSEKF_STATE_IN_FILTER_FRAME | POSEKF_STATE_OUT_FILTER_FRAME (include/posekf.h)
  float* innov_acc;     // [2][N] in/out innovation likelihood sums (NIS, ln det S; TAN kernels: of the tangent-space
                        // model), or null; read by INNOV kernels only
  // batched recordings (read by BATCH kernels only; filter n uses column n % Ns of both):
  const float* dt_cols;     // [T][Ns] per-stream time steps (overrides dt / dt_per_step), or null
  const int32_t* n_valid;   // [Ns] steps of this launch that stream n % Ns has (0..T); later steps hold the filter, or null
                            // (last: the parameter offsets of the other kernels are unchanged)
};
constexpr int kStateInFilterFrame = 1, kStateOutFilterFrame = 2;

struct FilterRegs {
  Quat<float> x;
  Quat<float> xlo;      // used by the compensated variant only
  Sym4<float> P;
  FilterConst<float> fc;
  Vec3<float> la, lm;   // low-pass state
  InnovAcc<float> in;   // innovation likelihood sums (INNOV kernels only)
};

template <int ALGO, bool LPF, bool COMP, bool INNOV = false, bool TAN = false>
__device__ __forceinline__ void load_filter(const ReplayParams& p, int64_t n, int64_t col, FilterRegs& f) {
  const int64_t N = p.N, Ns = p.Ns;
  Vec3<float> ra = {p.acc_ref[col], p.acc_ref[Ns + col], p.acc_ref[2 * Ns + col]};
  Vec3<float> rm = {p.mag_ref[col], p.mag_ref[Ns + col], p.mag_ref[2 * Ns + col]};
  f.fc = make_filter_const<float>(ra, rm, p.q_scale[n], p.r_scale[n]);
  if (INNOV) f.in = make_innov_acc<float, TAN>(p.innov_acc[n], p.innov_acc[N + n], p.r_scale[n]);
  f.x = {p.state_x[n], p.state_x[N + n], p.state_x[2 * N + n], p.state_x[3 * N + n]};
  f.xlo = {0.f, 0.f, 0.f, 0.f};
  if (COMP) f.xlo = {p.state_x_lo[n], p.state_x_lo[N + n], p.state_x_lo[2 * N + n], p.state_x_lo[3 * N + n]};
  const float* sp = p.state_p + n;   // P/r: the step works in units of r (see ekf_step), so does the state buffer
  f.P = {sp[0], sp[N], sp[2 * N], sp[3 * N], sp[4 * N], sp[5 * N], sp[6 * N], sp[7 * N], sp[8 * N], sp[9 * N]};
  if (LPF) {
    const float* sl = p.state_lpf + n;
    f.la = {sl[0], sl[N], sl[2 * N]};
    f.lm = {sl[3 * N], sl[4 * N], sl[5 * N]};
  }
  // the step runs in the filter frame (ekf_math.cuh); the state buffers hold the reference frame unless flagged
  adopt_state(f.fc, f.x, f.xlo);
  if (uses_filter_frame<ALGO>() && !(p.state_flags & kStateInFilterFrame)) enter_filter_frame(f.fc, f.x, f.xlo, f.P, COMP);
}

template <int ALGO, bool LPF, bool COMP, bool INNOV = false, bool TAN = false>
__device__ __forceinline__ void store_filter(const ReplayParams& p, int64_t n, FilterRegs& f) {
  const int64_t N = p.N;
  if (uses_filter_frame<ALGO>() && !(p.state_flags & kStateOutFilterFrame)) leave_filter_frame(f.fc, f.x, f.xlo, f.P, COMP);
  p.state_x[n] = f.x.w; p.state_x[N + n] = f.x.x; p.state_x[2 * N + n] = f.x.y; p.state_x[3 * N + n] = f.x.z;
  if (COMP) {
    p.state_x_lo[n] = f.xlo.w; p.state_x_lo[N + n] = f.xlo.x; p.state_x_lo[2 * N + n] = f.xlo.y; p.state_x_lo[3 * N + n] = f.xlo.z;
  }
  float* sp = p.state_p + n;
  sp[0] = f.P.a00; sp[N] = f.P.a01; sp[2 * N] = f.P.a02; sp[3 * N] = f.P.a03; sp[4 * N] = f.P.a11;
  sp[5 * N] = f.P.a12; sp[6 * N] = f.P.a13; sp[7 * N] = f.P.a22; sp[8 * N] = f.P.a23; sp[9 * N] = f.P.a33;
  if (LPF) {
    float* sl = p.state_lpf + n;
    sl[0] = f.la.x; sl[N] = f.la.y; sl[2 * N] = f.la.z; sl[3 * N] = f.lm.x; sl[4 * N] = f.lm.y; sl[5 * N] = f.lm.z;
  }
  if (INNOV) { p.innov_acc[n] = f.in.nis; p.innov_acc[N + n] = f.in.logdet; }
}

// One filter step + optional outputs.  AUX = the launch has a trajectory and/or flip output.
struct AuxPtrs {
  float4* traj;          // this filter's slot in out_traj, advanced by N per step
  uint8_t* flips;
  const float4* truth;   // this filter's column in the reference track, advanced by Ns per step
  float loss;
};

template <bool AUX> __device__ __forceinline__ AuxPtrs make_aux(const ReplayParams& p, int64_t n, int64_t col, bool valid) {
  AuxPtrs a = {nullptr, nullptr, nullptr, 0.f};
  if (AUX && valid) {
    if (p.out_traj) a.traj = reinterpret_cast<float4*>(p.out_traj) + n;
    if (p.out_flip) a.flips = p.out_flip + n;
    if (p.truth) { a.truth = reinterpret_cast<const float4*>(p.truth) + col; a.loss = p.loss_acc[n]; }
  }
  return a;
}

template <int ALGO, bool LPF, bool AUX, bool COMP, bool INNOV = false, bool TAN = false>
__device__ __forceinline__ void filter_step(const ReplayParams& p, FilterRegs& f, const float (&s)[kChannels], float h,
                                            AuxPtrs& aux) {
  Vec3<float> w = {s[0], s[1], s[2]}, a = {s[3], s[4], s[5]}, m = {s[6], s[7], s[8]};
  if (LPF) {   // SRV/KalmanFilter.cpp:285,298 -- filtered values feed Wahba, not renormalised
    if (p.alpha_acc >= 0.f) { lowpass<float>(f.la, a, p.alpha_acc, 1.f - p.alpha_acc); a = f.la; }
    if (p.alpha_mag >= 0.f) { lowpass<float>(f.lm, m, p.alpha_mag, 1.f - p.alpha_mag); m = f.lm; }
  }
  bool flip;
  // flip-mask byte: the float32 decision, plus the tie marker and per-branch alternatives that flip_fixup_kernel settles
  // in float64 after the launch (raw samples only: a low-passed sample is not in the stream any more)
  unsigned code = 0;
  ekf_step<float, ALGO, AUX, COMP, INNOV, TAN>(f.x, f.xlo, f.P, f.fc, w, a, m, StepH<float>(h), flip, aux.flips != nullptr,
                                               (AUX && !LPF && ALGO == WAHBA_QR2) ? &code : nullptr, INNOV ? &f.in : nullptr);
  if (!(AUX && !LPF && ALGO == WAHBA_QR2)) code = flip ? 1u : 0u;
  if (AUX) {
    // per-step outputs are in the reference frame (the reference's X_k)
    Quat<float> xr = f.x;
    if (uses_filter_frame<ALGO>() && (aux.traj || aux.truth)) xr = state_in_reference_frame(f.fc, f.x);
    if (aux.traj) {   // [T][N][4]: one 16-byte store per filter-step, consecutive filters consecutive
      asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(aux.traj), "f"(xr.w), "f"(xr.x), "f"(xr.y),
                   "f"(xr.z)
                   : "memory");
      aux.traj += p.N;
    }
    if (aux.flips) { *aux.flips = (uint8_t)code; aux.flips += p.N; }
    if (aux.truth) {  // tuning objective: sin^2 of the angle between the estimate and the reference track
      const float4 qt = __ldg(aux.truth);
      aux.truth += p.Ns;
      // sin^2 of the angle as the squared 4-D wedge product |X ^ q_ref|^2 = |X|^2 |q_ref|^2 - (X.q_ref)^2
      // (Lagrange identity): the six 2x2 minors are small numbers computed without the 1 - d^2
      // cancellation and without sensitivity to the 1e-7 norm error of either quaternion.
      const float xw = xr.w, xx = xr.x, xy = xr.y, xz = xr.z, qw = qt.x, qx = qt.y, qy = qt.z, qz = qt.w;
      const float m01 = fmaf(xw, qx, -(xx * qw)), m02 = fmaf(xw, qy, -(xy * qw)), m03 = fmaf(xw, qz, -(xz * qw));
      const float m12 = fmaf(xx, qy, -(xy * qx)), m13 = fmaf(xx, qz, -(xz * qx)), m23 = fmaf(xy, qz, -(xz * qy));
      aux.loss += fmaf(m23, m23, fmaf(m13, m13, fmaf(m12, m12, fmaf(m03, m03, fmaf(m02, m02, m01 * m01)))));
    }
  }
}

// A step at or past the length of the filter's stream (BATCH kernels): the filter is left as it is, the trajectory slot
// gets the held state, the flip byte is 0 (unmarked: flip_fixup_kernel leaves it alone) and the objectives add nothing.
// The step's sample and dt are not read.
template <int ALGO, bool AUX>
__device__ __forceinline__ void hold_step(const ReplayParams& p, const FilterRegs& f, AuxPtrs& aux) {
  if (AUX) {
    if (aux.traj) {
      Quat<float> xr = f.x;
      if (uses_filter_frame<ALGO>()) xr = state_in_reference_frame(f.fc, f.x);
      stg_stream4(aux.traj, xr.w, xr.x, xr.y, xr.z);
      aux.traj += p.N;
    }
    if (aux.flips) { *aux.flips = 0; aux.flips += p.N; }
    if (aux.truth) aux.truth += p.Ns;
  }
}

// ---------------------------------------------------------------------------------------------
// Replay, LDG staging: coalesced loads straight to registers, next step prefetched while the
// current one is computed.
// ---------------------------------------------------------------------------------------------
// (INNOV: the innovation likelihood, TAN: its tangent-space form; their instantiations always have AUX and are built for
//  3 CTAs per SM, <= 168 registers.  BATCH: per-stream dt columns and lengths, ReplayParams::dt_cols / n_valid)
template <int ALGO, bool LPF, bool AUX, bool COMP, bool INNOV = false, bool TAN = false, bool BATCH = false>
__global__ void __launch_bounds__(kThreads, INNOV ? 3 : ((ALGO == WAHBA_JACOBI || (COMP && LPF && AUX)) ? 4 : ((COMP || LPF) ? (kMinCtasPerSm > 5 ? 5 : kMinCtasPerSm) : kMinCtasPerSm)))
    replay_ldg_kernel(const ReplayParams p) {
  const int64_t n = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (n >= p.N) return;
  const int64_t Ns = p.Ns;
  const int64_t col = (Ns == p.N) ? n : (n % Ns);
  FilterRegs f;
  load_filter<ALGO, LPF, COMP, INNOV, TAN>(p, n, col, f);
  AuxPtrs aux = make_aux<AUX>(p, n, col, true);
  const float* s = p.streams + col;
  const int64_t step_stride = kChannels * Ns;
  float cur[kChannels], nxt[kChannels];
  const int T = (int)p.T;     // T == 0: a frame conversion of the state only (no stream is read)
  // BATCH: this stream's length and time-step column (prefetched with the samples)
  const int nv = (BATCH && p.n_valid) ? p.n_valid[col] : T;
  const float* dc = (BATCH && p.dt_cols) ? p.dt_cols + col : nullptr;
  float hcur = 0.f, hnxt = 0.f;
#pragma unroll
  for (int c = 0; c < kChannels; ++c) cur[c] = T > 0 ? ldg_stream(s + c * Ns) : 0.f;
  if (BATCH && dc && T > 0) hcur = ldg_stream(dc);
  const float dt0 = T > 0 ? p.dt[0] : 0.f;
  for (int t = 0; t < T; ++t) {
    if (t + 1 < T) s += step_stride;
#pragma unroll
    for (int c = 0; c < kChannels; ++c) nxt[c] = ldg_stream(s + c * Ns);
    if (BATCH && dc) hnxt = ldg_stream(dc + (int64_t)(t + 1 < T ? t + 1 : t) * Ns);
    const float h = (BATCH && dc) ? hcur : (p.dt_per_step ? __ldg(p.dt + t) : dt0);
    if (!BATCH || t < nv) filter_step<ALGO, LPF, AUX, COMP, INNOV, TAN>(p, f, cur, h, aux);
    else hold_step<ALGO, AUX>(p, f, aux);
#pragma unroll
    for (int c = 0; c < kChannels; ++c) cur[c] = nxt[c];
    if (BATCH) hcur = hnxt;
  }
  store_filter<ALGO, LPF, COMP, INNOV, TAN>(p, n, f);
  if (AUX && aux.truth) p.loss_acc[n] = aux.loss;
}

// BATCH kernels: the stream length(s) of the thread's filter(s) and the per-step dt of the current and the next tile
// (registers; the next tile's are loaded one tile ahead, like the samples)
template <bool BATCH, typename V, int S> struct BatchRegs {};
template <typename V, int S> struct BatchRegs<true, V, S> {
  int nv, nv1, min_nv;
  const float* dc;
  V cur[S], next[S];
};

// dt of the S steps of tile k (0 past T): a column of dt_cols, or the launch's dt / dt[T]
template <int S>
__device__ __forceinline__ void load_dt_tile(float (&h)[S], const ReplayParams& p, const float* dc, int k, int T, float dt0) {
#pragma unroll
  for (int tt = 0; tt < S; ++tt) {
    const int t = k * S + tt;
    h[tt] = t >= T ? 0.f : (dc ? ldg_stream(dc + (int64_t)t * p.Ns) : (p.dt_per_step ? __ldg(p.dt + t) : dt0));
  }
}
template <int S>
__device__ __forceinline__ void load_dt_tile(f32x2 (&h)[S], const ReplayParams& p, const float* dc, int k, int T, float dt0) {
#pragma unroll
  for (int tt = 0; tt < S; ++tt) {
    const int t = k * S + tt;
    h[tt] = t >= T ? f32x2(0.f) : (dc ? ldg2_stream(dc + (int64_t)t * p.Ns) : f32x2(p.dt_per_step ? __ldg(p.dt + t) : dt0));
  }
}

// ---------------------------------------------------------------------------------------------
// Replay, TMA staging: a ring of kTmaStages tiles [kTmaSteps][9][128] in shared memory, each filled
// by ONE cp.async.bulk.tensor.3d issued by thread 0 and signalled through an mbarrier; consumers
// release a tile with one mbarrier arrive per warp.  Out-of-range columns/steps are zero-filled by
// the TMA unit, so ragged N and T need no special casing on the load side.
// ---------------------------------------------------------------------------------------------
struct __align__(128) TmaSmem {
  float tile[kTmaStages][kTmaSteps][kChannels][kThreads];
  uint64_t full[kTmaStages];
  uint64_t empty[kTmaStages];
};
constexpr uint32_t kTileBytes = kTmaSteps * kChannels * kThreads * sizeof(float);

template <int ALGO, bool LPF, bool AUX, bool COMP, bool INNOV = false, bool TAN = false, bool BATCH = false>
__global__ void __launch_bounds__(kThreads, INNOV ? 3 : (ALGO == WAHBA_JACOBI ? 4 : ((COMP && (LPF || AUX)) ? (kMinCtasPerSm > 5 ? 5 : kMinCtasPerSm) : kMinCtasPerSm)))
    replay_tma_kernel(const ReplayParams p, const __grid_constant__ CUtensorMap tmap) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  TmaSmem& sm = *reinterpret_cast<TmaSmem*>(smem_raw);
  const int tid = threadIdx.x;
  const int64_t n0 = (int64_t)blockIdx.x * kThreads;
  const int64_t n = n0 + tid;
  const bool valid = n < p.N;
  const int col0 = (int)((p.Ns == p.N) ? n0 : (n0 % p.Ns));
  const int T = (int)p.T;
  const int n_chunks = (T + kTmaSteps - 1) / kTmaSteps;

  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < kTmaStages; ++s) { mbar_init(&sm.full[s], 1); mbar_init(&sm.empty[s], kThreads / 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (tid == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
#pragma unroll
    for (int s = 0; s < kTmaStages; ++s) {
      if (s < n_chunks) {
        mbar_expect_tx(&sm.full[s], kTileBytes);
        tma_load_3d(&sm.tile[s][0][0][0], &tmap, &sm.full[s], col0, 0, s * kTmaSteps);
      }
    }
  }

  FilterRegs f;
  if (valid) load_filter<ALGO, LPF, COMP, INNOV, TAN>(p, n, (int64_t)col0 + tid, f);
  AuxPtrs aux = make_aux<AUX>(p, n, (int64_t)col0 + tid, valid);
  const float dt0 = p.dt[0];
  // BATCH: this stream's length, and the time steps of the next tile held in registers (loaded one tile ahead: the
  // shared-memory ring has no room left at this kernel's occupancy)
  [[maybe_unused]] BatchRegs<BATCH, float, kTmaSteps> bt;
  if constexpr (BATCH) {
    bt.nv = (valid && p.n_valid) ? p.n_valid[col0 + tid] : T;
    bt.dc = p.dt_cols ? p.dt_cols + col0 + tid : nullptr;
    if (valid) load_dt_tile(bt.next, p, bt.dc, 0, T, dt0);
  }

  int stage = 0;
  uint32_t parity = 0;
  for (int k = 0; k < n_chunks; ++k) {
    // producer: refill the tile that every warp released in the previous iteration
    if (tid == 0 && k >= 1 && (k - 1 + kTmaStages) < n_chunks) {
      const int ps = (stage == 0) ? kTmaStages - 1 : stage - 1;
      const uint32_t pp = (stage == 0) ? (parity ^ 1u) : parity;     // parity of iteration k-1
      mbar_wait(&sm.empty[ps], pp);
      mbar_expect_tx(&sm.full[ps], kTileBytes);
      tma_load_3d(&sm.tile[ps][0][0][0], &tmap, &sm.full[ps], col0, 0, (k - 1 + kTmaStages) * kTmaSteps);
    }
    if constexpr (BATCH) {
#pragma unroll
      for (int tt = 0; tt < kTmaSteps; ++tt) bt.cur[tt] = bt.next[tt];
      if (valid && k + 1 < n_chunks) load_dt_tile(bt.next, p, bt.dc, k + 1, T, dt0);
    }
    mbar_wait(&sm.full[stage], parity);
    if (valid) {
      const int steps = min(kTmaSteps, T - k * kTmaSteps);     // < kTmaSteps only in the last chunk
#pragma unroll
      for (int tt = 0; tt < kTmaSteps; ++tt) {
        if (tt < steps) {
          if constexpr (BATCH) {
            if (k * kTmaSteps + tt >= bt.nv) { hold_step<ALGO, AUX>(p, f, aux); continue; }
          }
          float s[kChannels];
#pragma unroll
          for (int c = 0; c < kChannels; ++c) s[c] = sm.tile[stage][tt][c][tid];
          if constexpr (BATCH) {
            filter_step<ALGO, LPF, AUX, COMP, INNOV, TAN>(p, f, s, bt.cur[tt], aux);
          } else {
            const float h = p.dt_per_step ? __ldg(p.dt + k * kTmaSteps + tt) : dt0;
            filter_step<ALGO, LPF, AUX, COMP, INNOV, TAN>(p, f, s, h, aux);
          }
        }
      }
    }
    __syncwarp();
    if ((tid & 31) == 0) mbar_arrive(&sm.empty[stage]);
    if (++stage == kTmaStages) { stage = 0; parity ^= 1; }
  }
  if (valid) store_filter<ALGO, LPF, COMP, INNOV, TAN>(p, n, f);
  if (AUX && valid && aux.truth) p.loss_acc[n] = aux.loss;
}

// ---------------------------------------------------------------------------------------------
// Replay, TMA staging, PACKED: each thread advances TWO filters in the lanes of f32x2 values, so
// every FP32 operation of the step is one FFMA2 / FMUL2 / FADD2.  Same tiles, same barriers and
// the same arithmetic per filter as replay_tma_kernel (results are bit-identical); kThreads2 = 128 threads own a
// tile of 256 filters, 3 CTAs (12 warps) per SM.  A complete tile whose samples all have |a_z| <= 1 (and a constant
// dt) runs as ONE basic block of kTma2Steps steps.  ALGO is WAHBA_QR2 or WAHBA_PRECOMPUTED (the Jacobi variant uses
// the scalar kernel).
// ---------------------------------------------------------------------------------------------
struct __align__(128) Tma2Smem {
  float tile[kTma2Stages][kTma2Steps][kChannels][kTile2];
  uint64_t full[kTma2Stages];
  uint64_t empty[kTma2Stages];
};
constexpr uint32_t kTile2Bytes = kTma2Steps * kChannels * kTile2 * sizeof(float);
constexpr uint32_t kBatchSmem2 = (kThreads2 / 32) * sizeof(int);     // BATCH: per-warp minima of the stream lengths

struct FilterRegs2 {
  Quat<f32x2> x, xlo;
  Sym4<f32x2> P;
  FilterConst<f32x2> fc;
  Vec3<f32x2> la, lm;
  InnovAcc<f32x2> in;
};

template <bool HOLD> struct HeldLanes {};
template <> struct HeldLanes<true> { mask2 live; FilterRegs2 f0; f32x2 loss0; };

// BATCH: the lanes that were past their stream's length (live false) get back the values they had before the step
template <bool LPF, bool COMP, bool INNOV>
__device__ __forceinline__ void hold_lanes(mask2 live, FilterRegs2& f, const FilterRegs2& f0) {
  f.x = {sel_(live, f.x.w, f0.x.w), sel_(live, f.x.x, f0.x.x), sel_(live, f.x.y, f0.x.y), sel_(live, f.x.z, f0.x.z)};
  if (COMP) f.xlo = {sel_(live, f.xlo.w, f0.xlo.w), sel_(live, f.xlo.x, f0.xlo.x), sel_(live, f.xlo.y, f0.xlo.y), sel_(live, f.xlo.z, f0.xlo.z)};
  f.P = {sel_(live, f.P.a00, f0.P.a00), sel_(live, f.P.a01, f0.P.a01), sel_(live, f.P.a02, f0.P.a02), sel_(live, f.P.a03, f0.P.a03),
         sel_(live, f.P.a11, f0.P.a11), sel_(live, f.P.a12, f0.P.a12), sel_(live, f.P.a13, f0.P.a13), sel_(live, f.P.a22, f0.P.a22),
         sel_(live, f.P.a23, f0.P.a23), sel_(live, f.P.a33, f0.P.a33)};
  if (LPF) {
    f.la = {sel_(live, f.la.x, f0.la.x), sel_(live, f.la.y, f0.la.y), sel_(live, f.la.z, f0.la.z)};
    f.lm = {sel_(live, f.lm.x, f0.lm.x), sel_(live, f.lm.y, f0.lm.y), sel_(live, f.lm.z, f0.lm.z)};
  }
  if (INNOV) { f.in.nis = sel_(live, f.in.nis, f0.in.nis); f.in.logdet = sel_(live, f.in.logdet, f0.in.logdet); }
}

// (the precise variant with per-step outputs needs ~190 registers: 8 warps per SM instead of 12.  INNOV: the innovation
//  likelihood (TAN: tangent-space form), instantiated without per-step outputs and low-pass -- the sweep path;
//  replay_dispatch routes the rest.  BATCH: per-stream dt columns and lengths; a tile runs as the one-block fast tile
//  when every filter of the CTA is live for all of its steps, and otherwise steps both lanes and keeps the old values of
//  a lane past its length)
template <int ALGO, bool LPF, bool AUX, bool COMP, bool INNOV = false, bool TAN = false, bool BATCH = false>
__global__ void __launch_bounds__(kThreads2, (AUX && COMP) ? ((256 / kThreads2) < PKF_MIN_CTAS2 ? (256 / kThreads2) : PKF_MIN_CTAS2) : PKF_MIN_CTAS2)
    replay_tma2_kernel(const ReplayParams p, const __grid_constant__ CUtensorMap tmap) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Tma2Smem& sm = *reinterpret_cast<Tma2Smem*>(smem_raw);
  const int tid = threadIdx.x;
  const int64_t n0 = (int64_t)blockIdx.x * kTile2;
  const int64_t n = n0 + 2 * tid;                  // this thread owns filters n and n + 1 (N is even)
  const bool valid = n < p.N;
  const int col0 = (int)((p.Ns == p.N) ? n0 : (n0 % p.Ns));
  const int T = (int)p.T;
  const int n_chunks = (T + kTma2Steps - 1) / kTma2Steps;
  const int64_t N = p.N, Ns = p.Ns;
  // BATCH: the lengths of this thread's two streams and their minimum over the CTA (reduced once, here)
  [[maybe_unused]] BatchRegs<BATCH, f32x2, kTma2Steps> bt;
  if constexpr (BATCH) {
    int* warp_min = reinterpret_cast<int*>(smem_raw + sizeof(Tma2Smem));     // kBatchSmem2 bytes past the ring
    bt.nv = bt.nv1 = bt.min_nv = T;
    if (valid && p.n_valid) { bt.nv = p.n_valid[col0 + 2 * tid]; bt.nv1 = p.n_valid[col0 + 2 * tid + 1]; }
    const int m = __reduce_min_sync(0xffffffffu, valid ? min(bt.nv, bt.nv1) : T);
    if ((tid & 31) == 0) warp_min[tid >> 5] = m;
  }

  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < kTma2Stages; ++s) { mbar_init(&sm.full[s], 1); mbar_init(&sm.empty[s], kThreads2 / 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if constexpr (BATCH) {
    const int* warp_min = reinterpret_cast<const int*>(smem_raw + sizeof(Tma2Smem));
#pragma unroll
    for (int w = 0; w < kThreads2 / 32; ++w) bt.min_nv = min(bt.min_nv, warp_min[w]);
  }
  if (tid == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
#pragma unroll
    for (int s = 0; s < kTma2Stages; ++s) {
      if (s < n_chunks) {
        mbar_expect_tx(&sm.full[s], kTile2Bytes);
        tma_load_3d(&sm.tile[s][0][0][0], &tmap, &sm.full[s], col0, 0, s * kTma2Steps);
      }
    }
  }

  FilterRegs2 f;
  if (valid) {
    const int64_t col = (int64_t)col0 + 2 * tid;
    Vec3<f32x2> ra = {ld2(p.acc_ref + col), ld2(p.acc_ref + Ns + col), ld2(p.acc_ref + 2 * Ns + col)};
    Vec3<f32x2> rm = {ld2(p.mag_ref + col), ld2(p.mag_ref + Ns + col), ld2(p.mag_ref + 2 * Ns + col)};
    f.fc = make_filter_const<f32x2>(ra, rm, ld2(p.q_scale + n), ld2(p.r_scale + n));
    if (INNOV) f.in = make_innov_acc<f32x2, TAN>(ld2(p.innov_acc + n), ld2(p.innov_acc + N + n), ld2(p.r_scale + n));
    f.x = {ld2(p.state_x + n), ld2(p.state_x + N + n), ld2(p.state_x + 2 * N + n), ld2(p.state_x + 3 * N + n)};
    f.xlo = {f32x2(0.f), f32x2(0.f), f32x2(0.f), f32x2(0.f)};
    if (COMP) f.xlo = {ld2(p.state_x_lo + n), ld2(p.state_x_lo + N + n), ld2(p.state_x_lo + 2 * N + n), ld2(p.state_x_lo + 3 * N + n)};
    const float* sp = p.state_p + n;
    f.P = {ld2(sp), ld2(sp + N), ld2(sp + 2 * N), ld2(sp + 3 * N), ld2(sp + 4 * N), ld2(sp + 5 * N), ld2(sp + 6 * N),
           ld2(sp + 7 * N), ld2(sp + 8 * N), ld2(sp + 9 * N)};
    if (LPF) {
      const float* sl = p.state_lpf + n;
      f.la = {ld2(sl), ld2(sl + N), ld2(sl + 2 * N)};
      f.lm = {ld2(sl + 3 * N), ld2(sl + 4 * N), ld2(sl + 5 * N)};
    }
    adopt_state(f.fc, f.x, f.xlo);
    if (uses_filter_frame<ALGO>() && !(p.state_flags & kStateInFilterFrame)) enter_filter_frame(f.fc, f.x, f.xlo, f.P, COMP);
  }
  const float dt0 = p.dt[0];
  const StepH<f32x2> sh0{f32x2(dt0), f32x2(dt0 * dt0), f32x2(dt0 * (-1.f / 6.f))};
  // auxiliary outputs: this thread's pair of adjacent slots
  float4* traj = nullptr;
  uint8_t* flips = nullptr;
  const float4* truth = nullptr;
  f32x2 loss(0.f);
  if (AUX && valid) {
    if (p.out_traj) traj = reinterpret_cast<float4*>(p.out_traj) + n;
    if (p.out_flip) flips = p.out_flip + n;
    if (p.truth) { truth = reinterpret_cast<const float4*>(p.truth) + ((int64_t)col0 + 2 * tid); loss = ld2(p.loss_acc + n); }
  }
  // BATCH: the per-lane time steps of the next tile, held in registers (loaded one tile ahead: the shared-memory ring has
  // no room left for them at 3 CTAs per SM)
  if constexpr (BATCH) {
    bt.dc = p.dt_cols ? p.dt_cols + col0 + 2 * tid : nullptr;
    if (valid) load_dt_tile(bt.next, p, bt.dc, 0, T, dt0);
  }

  int stage = 0;
  uint32_t parity = 0;
  for (int k = 0; k < n_chunks; ++k) {
    if (tid == 0 && k >= 1 && (k - 1 + kTma2Stages) < n_chunks) {
      const int ps = (stage == 0) ? kTma2Stages - 1 : stage - 1;
      const uint32_t pp = (stage == 0) ? (parity ^ 1u) : parity;
      mbar_wait(&sm.empty[ps], pp);
      mbar_expect_tx(&sm.full[ps], kTile2Bytes);
      tma_load_3d(&sm.tile[ps][0][0][0], &tmap, &sm.full[ps], col0, 0, (k - 1 + kTma2Stages) * kTma2Steps);
    }
#if PKF_L2_PREFETCH > 0
    if (tid == 0 && (k + kTma2Stages - 1 + PKF_L2_PREFETCH) < n_chunks)
      tma_prefetch_l2_3d(&tmap, col0, 0, (k + kTma2Stages - 1 + PKF_L2_PREFETCH) * kTma2Steps);
#endif
    if constexpr (BATCH) {
#pragma unroll
      for (int tt = 0; tt < kTma2Steps; ++tt) bt.cur[tt] = bt.next[tt];
      if (valid && k + 1 < n_chunks) load_dt_tile(bt.next, p, bt.dc, k + 1, T, dt0);
    }
    mbar_wait(&sm.full[stage], parity);
    if (valid) {
      const int steps = min(kTma2Steps, T - k * kTma2Steps);
      // One packed step on the samples of slot tt of the current tile.  FAST: the tile is complete and none of its
      // samples takes the rare reflected-Wahba path (|a_z| > 1), so the whole tile is ONE basic block for the
      // scheduler (the measurement of step t+1 does not depend on the state and overlaps the update of step t).
      auto one_step = [&](int tt, auto fast_tag) {
        constexpr bool FAST = decltype(fast_tag)::value;
        f32x2 s[kChannels];
#pragma unroll
        for (int c = 0; c < kChannels; ++c) s[c] = ld2(&sm.tile[stage][tt][c][2 * tid]);
        StepH<f32x2> sh = sh0;                         // launch constant (the fast path runs only then) ...
        if constexpr (BATCH) sh = StepH<f32x2>(bt.cur[tt]);     // (per lane: rounds as the scalar StepH<float> of each lane)
        else if (!FAST && p.dt_per_step) sh = StepH<f32x2>(f32x2(__ldg(p.dt + k * kTma2Steps + tt)));     // ... unless dt comes per step
        // BATCH, general path: the lanes past their stream's length get their values from before the step back
        [[maybe_unused]] HeldLanes<BATCH && !FAST> held;
        if constexpr (BATCH) {
          if constexpr (!FAST) {
            const int t = k * kTma2Steps + tt;
            held.live = mask2{t < bt.nv, t < bt.nv1};
            held.f0 = f;
            held.loss0 = loss;
          }
        }
        Vec3<f32x2> w = {s[0], s[1], s[2]}, a = {s[3], s[4], s[5]}, m = {s[6], s[7], s[8]};
        if (LPF) {
          if (p.alpha_acc >= 0.f) { lowpass<f32x2>(f.la, a, f32x2(p.alpha_acc), f32x2(1.f - p.alpha_acc)); a = f.la; }
          if (p.alpha_mag >= 0.f) { lowpass<f32x2>(f.lm, m, f32x2(p.alpha_mag), f32x2(1.f - p.alpha_mag)); m = f.lm; }
        }
        mask2 flip;
        constexpr bool kTieCode = AUX && !LPF && ALGO == WAHBA_QR2;     // see filter_step
        FlipCode2 code = {0u, 0u};
        if constexpr (FAST && ALGO == WAHBA_QR2) ekf_step_plain_measured<f32x2, AUX, COMP, INNOV, TAN>(f.x, f.xlo, f.P, f.fc, w, a, m, sh, flip, flips != nullptr,
                                                                                                        kTieCode ? &code : nullptr, INNOV ? &f.in : nullptr);
        else ekf_step<f32x2, ALGO, AUX, COMP, INNOV, TAN>(f.x, f.xlo, f.P, f.fc, w, a, m, sh, flip, flips != nullptr, kTieCode ? &code : nullptr,
                                                          INNOV ? &f.in : nullptr);
        if (!kTieCode) code = FlipCode2{flip.x ? 1u : 0u, flip.y ? 1u : 0u};
        if constexpr (BATCH && !FAST) {
          if (!(held.live.x && held.live.y)) {
            hold_lanes<LPF, COMP, INNOV>(held.live, f, held.f0);
            code = FlipCode2{held.live.x ? code.x : 0u, held.live.y ? code.y : 0u};
          }
        }
        if (AUX) {
          Quat<f32x2> xr = f.x;     // per-step outputs are in the reference frame
          if (uses_filter_frame<ALGO>() && (traj || truth)) xr = state_in_reference_frame(f.fc, f.x);
          if (traj) {   // [T][N][4]: two adjacent 16-byte quaternions
            asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(traj), "f"(xr.w.x), "f"(xr.x.x), "f"(xr.y.x),
                         "f"(xr.z.x) : "memory");
            asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(traj + 1), "f"(xr.w.y), "f"(xr.x.y),
                         "f"(xr.y.y), "f"(xr.z.y) : "memory");
            traj += N;
          }
          if (flips) { *reinterpret_cast<uchar2*>(flips) = make_uchar2((unsigned char)code.x, (unsigned char)code.y); flips += N; }
          if (truth) {  // squared wedge product |X ^ q_ref|^2 per lane (see the scalar kernel)
            const float4 t0 = __ldg(truth), t1 = __ldg(truth + 1);
            truth += Ns;
            const f32x2 qw(t0.x, t1.x), qx(t0.y, t1.y), qy(t0.z, t1.z), qz(t0.w, t1.w);
            const f32x2 xw = xr.w, xx = xr.x, xy = xr.y, xz = xr.z;
            const f32x2 m01 = fma_(xw, qx, -(xx * qw)), m02 = fma_(xw, qy, -(xy * qw)), m03 = fma_(xw, qz, -(xz * qw));
            const f32x2 m12 = fma_(xx, qy, -(xy * qx)), m13 = fma_(xx, qz, -(xz * qx)), m23 = fma_(xy, qz, -(xz * qy));
            loss = loss + fma_(m23, m23, fma_(m13, m13, fma_(m12, m12, fma_(m03, m03, fma_(m02, m02, m01 * m01)))));
            if constexpr (BATCH && !FAST) loss = sel_(held.live, loss, held.loss0);
          }
        }
      };
      bool fast = false;
      // (BATCH: the time steps come per lane from registers; every filter of the CTA is live for the whole tile)
      bool whole;
      if constexpr (BATCH) whole = k * kTma2Steps + kTma2Steps <= bt.min_nv;
      else whole = !p.dt_per_step;
      if constexpr (ALGO == WAHBA_PRECOMPUTED && PKF_FAST_TILE) fast = steps == kTma2Steps && whole;   // no branch in that step at all
      if constexpr (ALGO == WAHBA_QR2 && !LPF && PKF_FAST_TILE) {
        if (steps == kTma2Steps && whole) {
          // |a_z| <= 1 for every sample of the tile (both lanes): the accelerometer weight 1 - |a_z| is non-negative
          float az = 0.f;
#pragma unroll
          for (int tt = 0; tt < kTma2Steps; ++tt) {
            const float2 v = *reinterpret_cast<const float2*>(&sm.tile[stage][tt][5][2 * tid]);
            az = fmaxf(az, fmaxf(fabsf(v.x), fabsf(v.y)));
          }
          fast = az <= 1.f;
        }
      }
      if (fast) {
#pragma unroll
        for (int tt = 0; tt < kTma2Steps; ++tt) one_step(tt, std::true_type{});
      } else {
#pragma unroll
        for (int tt = 0; tt < kTma2Steps; ++tt) {
          if (tt < steps) one_step(tt, std::false_type{});
        }
      }
    }
    __syncwarp();
    if ((tid & 31) == 0) mbar_arrive(&sm.empty[stage]);
    if (++stage == kTma2Stages) { stage = 0; parity ^= 1; }
  }
  if (valid) {
    if (uses_filter_frame<ALGO>() && !(p.state_flags & kStateOutFilterFrame)) leave_filter_frame(f.fc, f.x, f.xlo, f.P, COMP);
    st2(p.state_x + n, f.x.w); st2(p.state_x + N + n, f.x.x); st2(p.state_x + 2 * N + n, f.x.y); st2(p.state_x + 3 * N + n, f.x.z);
    if (COMP) {
      st2(p.state_x_lo + n, f.xlo.w); st2(p.state_x_lo + N + n, f.xlo.x); st2(p.state_x_lo + 2 * N + n, f.xlo.y);
      st2(p.state_x_lo + 3 * N + n, f.xlo.z);
    }
    float* sp = p.state_p + n;
    st2(sp, f.P.a00); st2(sp + N, f.P.a01); st2(sp + 2 * N, f.P.a02); st2(sp + 3 * N, f.P.a03); st2(sp + 4 * N, f.P.a11);
    st2(sp + 5 * N, f.P.a12); st2(sp + 6 * N, f.P.a13); st2(sp + 7 * N, f.P.a22); st2(sp + 8 * N, f.P.a23); st2(sp + 9 * N, f.P.a33);
    if (LPF) {
      float* sl = p.state_lpf + n;
      st2(sl, f.la.x); st2(sl + N, f.la.y); st2(sl + 2 * N, f.la.z); st2(sl + 3 * N, f.lm.x); st2(sl + 4 * N, f.lm.y); st2(sl + 5 * N, f.lm.z);
    }
    if (AUX && p.truth) st2(p.loss_acc + n, loss);
    if (INNOV) { st2(p.innov_acc + n, f.in.nis); st2(p.innov_acc + N + n, f.in.logdet); }
  }
}

}  // namespace pkf_dev
