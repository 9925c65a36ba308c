// ops_kernels.cuh -- stand-alone operators with the reference's per-function semantics (Wahba, rot2quat,
// Prediction, Correction, RK4, Jacobians, Comparator, low-pass, RPY, norm), the comparison tracks,
// the raw-sensor pre-processing, and the measurement / host-replay helper kernels.
#pragma once
#include "device_util.cuh"

namespace pkf_dev {

// ---------------------------------------------------------------------------------------------
// Stand-alone Wahba (config "Wahba-only batched 3x3 SVD + R->quat").
// The Jacobi variant runs sweeps until every lane of the warp has converged (warp vote), at most
// `max_sweeps`.
// ---------------------------------------------------------------------------------------------
struct WahbaParams {
  int64_t N;
  const float *acc_ref, *mag_ref;
  int ref_shared;
  const float *acc, *mag, *k_acc, *k_mag;
  float k_acc_s, k_mag_s;
  int weights_from_acc;
  float *out_rot, *out_quat;
  int max_sweeps;
};

template <int ALGO> __global__ void __launch_bounds__(256) wahba_kernel(const WahbaParams p) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = n < p.N;
  const int64_t i = valid ? n : 0;   // tail lanes recompute element 0 so the warp vote stays full
  const int64_t N = p.N;
  Vec3<float> ra, rm;
  if (p.ref_shared) {
    ra = {__ldg(p.acc_ref), __ldg(p.acc_ref + 1), __ldg(p.acc_ref + 2)};
    rm = {__ldg(p.mag_ref), __ldg(p.mag_ref + 1), __ldg(p.mag_ref + 2)};
  } else {
    ra = {ldg_stream(p.acc_ref + i), ldg_stream(p.acc_ref + N + i), ldg_stream(p.acc_ref + 2 * N + i)};
    rm = {ldg_stream(p.mag_ref + i), ldg_stream(p.mag_ref + N + i), ldg_stream(p.mag_ref + 2 * N + i)};
  }
  Vec3<float> a = {ldg_stream(p.acc + i), ldg_stream(p.acc + N + i), ldg_stream(p.acc + 2 * N + i)};
  Vec3<float> m = {ldg_stream(p.mag + i), ldg_stream(p.mag + N + i), ldg_stream(p.mag + 2 * N + i)};
  float ka, km;
  if (p.k_acc) { ka = ldg_stream(p.k_acc + i); km = ldg_stream(p.k_mag + i); }
  else if (p.weights_from_acc) { ka = fabsf(a.z); km = 1.f - ka; }           // PKF/ExtendedKalmanFilter.py:71
  else { ka = p.k_acc_s; km = p.k_mag_s; }
  Mat3<float> R;
  if (ALGO == WAHBA_QR2) R = wahba_qr2<float>(frame_from_pair<float>(ra, rm), a, m, ka, km);
  else R = wahba_jacobi<float>(ra, rm, a, m, ka, km, p.max_sweeps);
  if (!valid) return;
  if (p.out_rot) {
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) stg_stream(p.out_rot + (3 * r + c) * N + n, R.m[r][c]);
  }
  if (p.out_quat) {
    Quat<float> q = rotation_to_quat_ref<float>(R);
    stg_stream(p.out_quat + n, q.w); stg_stream(p.out_quat + N + n, q.x);
    stg_stream(p.out_quat + 2 * N + n, q.y); stg_stream(p.out_quat + 3 * N + n, q.z);
  }
}

// ---------------------------------------------------------------------------------------------
// Comparison tracks of the tuning workflow (what Results/*.png overlays): the gyro-only attitude
// (RK4 without correction: SRV/KalmanFilter.cpp:149, `Quarternion_Gyro_pure`) and the Wahba-only
// attitude per sample (PKF/main_file.py:40: getQuarternion(acc, mag, .5, .5), raw sign convention).
// ---------------------------------------------------------------------------------------------
struct TracksParams {
  int64_t N, T, Ns;
  const float *streams, *dt;
  int dt_per_step;
  const float *acc_ref, *mag_ref;
  float k_acc, k_mag;
  int weights_from_acc;
  float* gyro_state;   // [4][N] in/out, or null
  float* out_gyro;     // [T][N][4] or null
  float* out_wahba;    // [T][N][4] or null
};

template <int ALGO> __global__ void __launch_bounds__(128) tracks_kernel(const TracksParams p) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= p.N) return;
  const int64_t N = p.N, Ns = p.Ns, col = (Ns == N) ? n : (n % Ns);
  Vec3<float> ra = {p.acc_ref[col], p.acc_ref[Ns + col], p.acc_ref[2 * Ns + col]};
  Vec3<float> rm = {p.mag_ref[col], p.mag_ref[Ns + col], p.mag_ref[2 * Ns + col]};
  const RefFrame<float> E = frame_from_pair<float>(ra, rm);
  Quat<float> g = {1.f, 0.f, 0.f, 0.f};
  if (p.gyro_state) g = {p.gyro_state[n], p.gyro_state[N + n], p.gyro_state[2 * N + n], p.gyro_state[3 * N + n]};
  const float* s = p.streams + col;
  float4* og = p.out_gyro ? reinterpret_cast<float4*>(p.out_gyro) + n : nullptr;
  float4* ow = p.out_wahba ? reinterpret_cast<float4*>(p.out_wahba) + n : nullptr;
  const float dt0 = p.dt[0];
  // the next step's channels are requested before the current step is computed and stored (one thread walks one
  // filter through time, so without this every step would expose a full memory latency)
  const bool need_gyro = og || p.gyro_state;
  float cur[kChannels], nxt[kChannels];
  auto load_step = [&](float (&v)[kChannels], const float* q) {
#pragma unroll
    for (int c = 0; c < kChannels; ++c) v[c] = ((c < 3) ? need_gyro : (ow != nullptr)) ? ldg_stream(q + c * Ns) : 0.f;
  };
  if (p.T > 0) load_step(cur, s);
  for (int64_t t = 0; t < p.T; ++t, s += kChannels * Ns) {
    if (t + 1 < p.T) load_step(nxt, s + kChannels * Ns);
    const float h = p.dt_per_step ? __ldg(p.dt + t) : dt0;
    if (need_gyro) {
      Vec3<float> hw = {0.5f * cur[0], 0.5f * cur[1], 0.5f * cur[2]};
      g = rk4_step<float>(g, hw, h);
      if (og) { stg_stream4(og, g.w, g.x, g.y, g.z); og += N; }
    }
    if (ow) {
      Vec3<float> a = {cur[3], cur[4], cur[5]};
      Vec3<float> m = {cur[6], cur[7], cur[8]};
      float ka = p.k_acc, km = p.k_mag;
      if (p.weights_from_acc) { ka = fabsf(a.z); km = 1.f - ka; }
      Mat3<float> R = (ALGO == WAHBA_QR2) ? wahba_qr2<float>(E, a, m, ka, km) : wahba_jacobi<float>(ra, rm, a, m, ka, km, 6);
      Quat<float> q = rotation_to_quat_ref<float>(R);
      stg_stream4(ow, q.w, q.x, q.y, q.z);
      ow += N;
    }
#pragma unroll
    for (int c = 0; c < kChannels; ++c) cur[c] = nxt[c];
  }
  if (p.gyro_state) { p.gyro_state[n] = g.w; p.gyro_state[N + n] = g.x; p.gyro_state[2 * N + n] = g.y; p.gyro_state[3 * N + n] = g.z; }
}

// ---------------------------------------------------------------------------------------------
// Raw-sensor pre-processing of the online pipeline (the step in front of the filter): linear
// interpolation of the accel / mag samples that bracket the gyro timestamp, normalisation, and the
// optional alpha low-pass -- SRV/Parser.cpp:229-267 (ExecuteKalmanFilter, LinearInterpolationSensor),
// :221-228 (NormalizeValues), SRV/KalmanFilter.cpp:279-303 (low-pass inside Set*Measurements).
// Writes the [T][9][N] stream the replay kernel consumes.
// ---------------------------------------------------------------------------------------------
// ExecuteKalmanFilter's sequence for one sensor (Parser.cpp:232-242): interpolate the bracketing samples y1, y2 to the
// gyro timestamp, y = (y2 - y1)/(t2 - t1)*(t3 - t1) + y1 (:264), then normalise (:223-227), in that operation order.
// preprocess_kernel and align_events_kernel both call it, so that the two cannot round differently.
__device__ __forceinline__ Vec3<float> interpolate_normalise(const float* y1, const float* y2, float t21, float t31) {
  float v[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) v[c] = (y2[c] - y1[c]) / t21 * t31 + y1[c];
  const float den = sqrtf(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
  return {v[0] / den, v[1] / den, v[2] / den};
}

struct PreprocessParams {
  int64_t N, T;
  const float* gyro;        // [T][3][N]
  const float* raw_prev;    // [T][6][N]  acc xyz, mag xyz : sample before the gyro timestamp (y1)
  const float* raw_next;    // [T][6][N]  sample after (y2)
  const float* tspan;       // [T][4][N]  seconds: acc (t2-t1), acc (t3-t1), mag (t2-t1), mag (t3-t1)
  float alpha_acc, alpha_mag;
  float* lpf_state;         // [6][N] in/out or null
  float* out_streams;       // [T][9][N]
};

__global__ void __launch_bounds__(256) preprocess_kernel(const PreprocessParams p) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= p.N) return;
  const int64_t N = p.N;
  const bool lpa = p.alpha_acc >= 0.f, lpm = p.alpha_mag >= 0.f;
  Vec3<float> la = {0.f, 0.f, 0.f}, lm = {0.f, 0.f, 0.f};
  if (p.lpf_state) {
    la = {p.lpf_state[n], p.lpf_state[N + n], p.lpf_state[2 * N + n]};
    lm = {p.lpf_state[3 * N + n], p.lpf_state[4 * N + n], p.lpf_state[5 * N + n]};
  }
  // one step's inputs: 3 gyro + 6 + 6 bracketing samples + 4 time spans; the next step's are requested before the
  // current step is computed and stored (see tracks_kernel)
  struct Step { float g[3], y1[6], y2[6], ts[4]; };
  auto load_step = [&](Step& v, int64_t t) {
    const float* y1 = p.raw_prev + t * 6 * N + n;
    const float* y2 = p.raw_next + t * 6 * N + n;
    const float* ts = p.tspan + t * 4 * N + n;
    const float* g = p.gyro + t * 3 * N + n;
#pragma unroll
    for (int c = 0; c < 3; ++c) v.g[c] = ldg_stream(g + c * N);
#pragma unroll
    for (int c = 0; c < 6; ++c) { v.y1[c] = ldg_stream(y1 + c * N); v.y2[c] = ldg_stream(y2 + c * N); }
#pragma unroll
    for (int c = 0; c < 4; ++c) v.ts[c] = ldg_stream(ts + c * N);
  };
  Step cur, nxt;
  if (p.T > 0) load_step(cur, 0);
  for (int64_t t = 0; t < p.T; ++t) {
    if (t + 1 < p.T) load_step(nxt, t + 1);
    float* o = p.out_streams + t * 9 * N + n;
    o[0] = cur.g[0]; o[N] = cur.g[1]; o[2 * N] = cur.g[2];
#pragma unroll
    for (int s = 0; s < 2; ++s) {                      // s = 0 accel, 1 mag
      Vec3<float> u = interpolate_normalise(cur.y1 + 3 * s, cur.y2 + 3 * s, cur.ts[2 * s], cur.ts[2 * s + 1]);
      if (s == 0 && lpa) { lowpass<float>(la, u, p.alpha_acc, 1.f - p.alpha_acc); u = la; }
      if (s == 1 && lpm) { lowpass<float>(lm, u, p.alpha_mag, 1.f - p.alpha_mag); u = lm; }
      o[(3 + 3 * s) * N] = u.x; o[(4 + 3 * s) * N] = u.y; o[(5 + 3 * s) * N] = u.z;
    }
    cur = nxt;
  }
  if (p.lpf_state) {
    p.lpf_state[n] = la.x; p.lpf_state[N + n] = la.y; p.lpf_state[2 * N + n] = la.z;
    p.lpf_state[3 * N + n] = lm.x; p.lpf_state[4 * N + n] = lm.y; p.lpf_state[5 * N + n] = lm.z;
  }
}

// Mean of K samples of one sensor, sample k's component j at x[k * k_stride + first + j * c_stride].  float64 accumulators, the
// reference's own precision and order (InitialValues.cpp:22-29,48-62): this runs once per recording over K = 100
// samples, and a float32 running sum would cost sqrt(K) ulps of the reference vectors.  Shared by initial_values_kernel
// and align_bounds_kernel.
__device__ __forceinline__ void initial_mean(const float* x, int64_t k_stride, int64_t first, int64_t c_stride, int64_t K,
                                             double& m0, double& m1, double& m2) {
  double s0 = 0.0, s1 = 0.0, s2 = 0.0;
  for (int64_t k = 0; k < K; ++k) {
    const float* p = x + k * k_stride + first;
    s0 += (double)ldg_stream(p); s1 += (double)ldg_stream(p + c_stride); s2 += (double)ldg_stream(p + 2 * c_stride);
  }
  m0 = s0 / (double)K; m1 = s1 / (double)K; m2 = s2 / (double)K;
}
// NormalizeValues in float64 (Parser.cpp:223-227), how acc_0 / mag_0 are made from the means (Parser.cpp:46-49)
__device__ __forceinline__ void normalise_f64(double& m0, double& m1, double& m2) {
  const double den = sqrt((m0 * m0) + (m1 * m1) + (m2 * m2));
  m0 = m0 / den; m1 = m1 / den; m2 = m2 / den;
}

// Initial reference vectors of the online pipeline: mean (and unbiased variance) of the first K samples of a
// sensor, the mean optionally normalised -- SRV/InitialValues.cpp:19-66 (running sum, two-pass variance with
// K-1), SRV/Parser.cpp:46-49 (acc0 / mag0 = normalised means).  samples [K][3][N] -> mean [3][N], var [3][N].
__global__ void __launch_bounds__(256)
    initial_values_kernel(int64_t N, int64_t K, const float* __restrict__ x, int normalize, float* __restrict__ mean,
                          float* __restrict__ var) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  double m0, m1, m2;
  initial_mean(x, 3 * N, n, N, K, m0, m1, m2);
  if (var) {
    double v0 = 0.0, v1 = 0.0, v2 = 0.0;
    for (int64_t k = 0; k < K; ++k) {
      const float* p = x + k * 3 * N + n;
      const double d0 = (double)__ldg(p) - m0, d1 = (double)__ldg(p + N) - m1, d2 = (double)__ldg(p + 2 * N) - m2;
      v0 += d0 * d0; v1 += d1 * d1; v2 += d2 * d2;
    }
    const double k1 = (double)(K - 1);
    var[n] = (float)(v0 / k1); var[N + n] = (float)(v1 / k1); var[2 * N + n] = (float)(v2 / k1);
  }
  double o0 = m0, o1 = m1, o2 = m2;
  if (normalize) normalise_f64(o0, o1, o2);
  mean[n] = (float)o0; mean[N + n] = (float)o1; mean[2 * N + n] = (float)o2;
}

// ---------------------------------------------------------------------------------------------
// Alignment of raw event recordings to the gyro clock (posekf_align_events_f32, DESIGN section 5 f10): the steps of
// recording c are its gyro events after t_init[c] (the later of the K-th acc and mag timestamps) that both sensors
// bracket; each step interpolates the last acc / mag event at or before the gyro timestamp and the first one after it.
// Timestamps are int64 ns and strictly increasing within a stream; every difference is formed in int64 and only then
// converted to float seconds (ns since an epoch do not fit in float32).  Streams are concatenated CSR style:
// recording c owns events off[c] .. off[c+1]-1, values are [3][M] with M = off[Ns].
// ---------------------------------------------------------------------------------------------
struct AlignParams {
  int64_t Ns, T, K;
  const int64_t *g_t, *a_t, *m_t;          // [M_s] ns
  const float *g_v, *a_v, *m_v;            // [3][M_s]
  const int64_t *g_off, *a_off, *m_off;    // [Ns+1]
  int32_t* lengths;                        // [Ns]
  int64_t* bounds;                         // [2][Ns]: gyro index of step 0, t_init (null: lengths only)
  float *acc_ref, *mag_ref;                // [3][Ns]
  float *streams, *dt;                     // [T][9][Ns], [T][Ns]
};

// first index in [lo, hi) whose timestamp is > key (hi if none); t strictly increasing
__device__ __forceinline__ int64_t upper_bound_ns(const int64_t* t, int64_t lo, int64_t hi, int64_t key) {
  while (lo < hi) {
    const int64_t mid = lo + ((hi - lo) >> 1);
    if (__ldg(t + mid) <= key) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

__device__ __forceinline__ float ns_to_seconds(int64_t d) { return (float)((double)d * 1e-9); }

// One thread per recording: t_init, the first and one-past-last bracketed gyro events (binary searches), the lengths,
// and the reference vectors from the first K events of each sensor (initial_values_kernel's arithmetic).  A recording
// with fewer than K events of either sensor has length 0 and stack_logs' padding reference vectors.
__global__ void __launch_bounds__(256) align_bounds_kernel(const AlignParams p) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= p.Ns) return;
  const int64_t Ns = p.Ns, K = p.K;
  const int64_t g0 = p.g_off[c], g1 = p.g_off[c + 1], a0 = p.a_off[c], a1 = p.a_off[c + 1], m0 = p.m_off[c], m1 = p.m_off[c + 1];
  const bool enough = a1 - a0 >= K && m1 - m0 >= K;
  int64_t first = g0, len = 0, t_init = 0;
  if (enough) {
    t_init = max(__ldg(p.a_t + a0 + K - 1), __ldg(p.m_t + m0 + K - 1));
    const int64_t t_end = min(__ldg(p.a_t + a1 - 1), __ldg(p.m_t + m1 - 1));     // a step needs an event after it
    first = upper_bound_ns(p.g_t, g0, g1, t_init);
    len = upper_bound_ns(p.g_t, first, g1, t_end - 1) - first;                  // gyro events in (t_init, t_end)
  }
  p.lengths[c] = (int32_t)len;
  if (!p.bounds) return;
  p.bounds[c] = first;
  p.bounds[Ns + c] = t_init;
  double ra[3] = {0.0, 0.0, 1.0}, rm[3] = {1.0, 0.0, 0.0};
  if (enough) {
    initial_mean(p.a_v, 1, a0, p.a_off[Ns], K, ra[0], ra[1], ra[2]);
    initial_mean(p.m_v, 1, m0, p.m_off[Ns], K, rm[0], rm[1], rm[2]);
    normalise_f64(ra[0], ra[1], ra[2]);
    normalise_f64(rm[0], rm[1], rm[2]);
  }
#pragma unroll
  for (int j = 0; j < 3; ++j) { p.acc_ref[j * Ns + c] = (float)ra[j]; p.mag_ref[j * Ns + c] = (float)rm[j]; }
}

// One thread per (step, recording) over tiles of 32 steps x 32 recordings.  A warp computes 32 consecutive steps of one
// recording, so its reads of the gyro events and of the bracketing acc / mag events are coalesced and its binary searches
// walk the same cache lines; the tile is transposed through shared memory so that every row of streams [T][9][Ns] and
// dt [T][Ns] is written 32 recordings at a time.  Steps at or past a recording's length repeat its last step with dt = 0;
// a recording of length 0 has gyro 0 and its reference vectors as acc / mag (stack_logs' padding).
constexpr int kAlignTile = 32, kAlignWarps = 8, kAlignRows = kChannels + 1;
__global__ void __launch_bounds__(kAlignTile * kAlignWarps) align_events_kernel(const AlignParams p, int64_t n_col_tiles) {
  __shared__ float tile[kAlignRows][kAlignTile][kAlignTile + 1];
  const int64_t bt = (int64_t)blockIdx.x / n_col_tiles, bc = (int64_t)blockIdx.x - bt * n_col_tiles;
  const int64_t i0 = bt * kAlignTile, c0 = bc * kAlignTile, Ns = p.Ns;
  const int lane = threadIdx.x, warp = threadIdx.y;
  const int64_t Mg = p.g_off[Ns], Ma = p.a_off[Ns], Mm = p.m_off[Ns];
  for (int cl = warp; cl < kAlignTile && c0 + cl < Ns; cl += kAlignWarps) {
    const int64_t c = c0 + cl, L = p.lengths[c], i = i0 + lane;
    float o[kAlignRows];
    if (L == 0) {
#pragma unroll
      for (int j = 0; j < 3; ++j) { o[j] = 0.f; o[3 + j] = p.acc_ref[j * Ns + c]; o[6 + j] = p.mag_ref[j * Ns + c]; }
      o[9] = 0.f;
    } else {
      const int64_t s = i < L ? i : L - 1;
      const int64_t g = p.bounds[c] + s, tg = __ldg(p.g_t + g);
      const int64_t t_prev = s == 0 ? p.bounds[Ns + c] : __ldg(p.g_t + g - 1);
      o[9] = i < L ? ns_to_seconds(tg - t_prev) : 0.f;
#pragma unroll
      for (int j = 0; j < 3; ++j) o[j] = __ldg(p.g_v + j * Mg + g);
#pragma unroll
      for (int sn = 0; sn < 2; ++sn) {                 // 0 accel, 1 mag
        const int64_t* t = sn ? p.m_t : p.a_t;
        const float* v = sn ? p.m_v : p.a_v;
        const int64_t M = sn ? Mm : Ma, e0 = sn ? p.m_off[c] : p.a_off[c], e1 = sn ? p.m_off[c + 1] : p.a_off[c + 1];
        // the K-th event is at or before t_init < tg, and the last one is after tg
        const int64_t j1 = upper_bound_ns(t, e0 + p.K - 1, e1, tg) - 1;
        const int64_t t1 = __ldg(t + j1);
        const float y1[3] = {__ldg(v + j1), __ldg(v + M + j1), __ldg(v + 2 * M + j1)};
        const float y2[3] = {__ldg(v + j1 + 1), __ldg(v + M + j1 + 1), __ldg(v + 2 * M + j1 + 1)};
        const Vec3<float> u = interpolate_normalise(y1, y2, ns_to_seconds(__ldg(t + j1 + 1) - t1), ns_to_seconds(tg - t1));
        o[3 + 3 * sn] = u.x; o[4 + 3 * sn] = u.y; o[5 + 3 * sn] = u.z;
      }
    }
#pragma unroll
    for (int r = 0; r < kAlignRows; ++r) tile[r][lane][cl] = o[r];
  }
  __syncthreads();
  for (int q = warp; q < kAlignRows * kAlignTile; q += kAlignWarps) {
    const int il = q / kAlignRows, r = q - il * kAlignRows;
    const int64_t i = i0 + il, c = c0 + lane;
    if (i >= p.T || c >= Ns) continue;
    const float v = tile[r][il][lane];
    if (r < kChannels) p.streams[(i * kChannels + r) * Ns + c] = v;
    else p.dt[i * Ns + c] = v;
  }
}

// Measurement stream for POSEKF_WAHBA_PRECOMPUTED: solves the Wahba problem of every (stream, step) ONCE --
// getQuarternion(acc, mag, |acc_z|, 1-|acc_z|) with the reference's sign convention, after the optional
// low-pass -- and writes a stream of the same [T][9][Ns] shape: rows 0-2 gyro, rows 3-6 the quaternion
// (w,x,y,z), rows 7-8 zero.  A (Q,R) sweep then replays it N/Ns times without redoing the solve.
struct MeasStreamParams {
  int64_t Ns, T;
  const float *streams, *acc_ref, *mag_ref;
  float alpha_acc, alpha_mag;
  float* lpf_state;    // [6][Ns] in/out or null
  float* out;          // [T][9][Ns]
};

template <int ALGO> __global__ void __launch_bounds__(128) measurement_stream_kernel(const MeasStreamParams p) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= p.Ns) return;
  const int64_t Ns = p.Ns;
  Vec3<float> ra = {p.acc_ref[n], p.acc_ref[Ns + n], p.acc_ref[2 * Ns + n]};
  Vec3<float> rm = {p.mag_ref[n], p.mag_ref[Ns + n], p.mag_ref[2 * Ns + n]};
  const RefFrame<float> E = frame_from_pair<float>(ra, rm);
  Vec3<float> la = {0.f, 0.f, 0.f}, lm = {0.f, 0.f, 0.f};
  if (p.lpf_state) {
    la = {p.lpf_state[n], p.lpf_state[Ns + n], p.lpf_state[2 * Ns + n]};
    lm = {p.lpf_state[3 * Ns + n], p.lpf_state[4 * Ns + n], p.lpf_state[5 * Ns + n]};
  }
  // Without the low-pass a sample's solution does not depend on its predecessors, so time is split over blockIdx.y
  // (thread (n, y) solves t = y, y + gridDim.y, ...): a sweep has few streams (256) and many steps (5000), and one
  // thread per stream walking all of them would leave the GPU empty.  With the low-pass gridDim.y is 1.
  // The next step's channels are requested before the current step is solved and stored (see tracks_kernel).
  const int64_t t0 = blockIdx.y, dt_ = gridDim.y;
  float cur[kChannels], nxt[kChannels];
  auto load_step = [&](float (&v)[kChannels], int64_t t) {
    const float* s = p.streams + t * kChannels * Ns + n;
#pragma unroll
    for (int c = 0; c < kChannels; ++c) v[c] = ldg_stream(s + c * Ns);
  };
  if (t0 < p.T) load_step(cur, t0);
  for (int64_t t = t0; t < p.T; t += dt_) {
    if (t + dt_ < p.T) load_step(nxt, t + dt_);
    float* o = p.out + t * kChannels * Ns + n;
    o[0] = cur[0]; o[Ns] = cur[1]; o[2 * Ns] = cur[2];      // plain stores: a sweep re-reads this stream from L2
    Vec3<float> a = {cur[3], cur[4], cur[5]};
    Vec3<float> m = {cur[6], cur[7], cur[8]};
    if (p.alpha_acc >= 0.f) { lowpass<float>(la, a, p.alpha_acc, 1.f - p.alpha_acc); a = la; }
    if (p.alpha_mag >= 0.f) { lowpass<float>(lm, m, p.alpha_mag, 1.f - p.alpha_mag); m = lm; }
    const float ka = fabsf(a.z), km = 1.f - ka;                                // PKF/ExtendedKalmanFilter.py:71
    Mat3<float> R = (ALGO == WAHBA_QR2) ? wahba_qr2<float>(E, a, m, ka, km) : wahba_jacobi<float>(ra, rm, a, m, ka, km, 6);
    const Quat<float> q = rotation_to_quat_ref<float>(R);
    // row 7 marks the samples whose sign rule sits on a float32 tie (raw samples only): meas_fixup_kernel re-decides
    // them in float64 and clears the mark, so that the replay's comparator sees the reference's own sign
    const bool raw = p.alpha_acc < 0.f && p.alpha_mag < 0.f && p.streams != p.out;     // (the fix-up reads the raw sample)
    const float tie = (raw && near_tie_(q.x * q.x, q.y * q.y, q.z * q.z, 1.f)) ? 1.f : 0.f;
    o[3 * Ns] = q.w; o[4 * Ns] = q.x; o[5 * Ns] = q.y; o[6 * Ns] = q.z; o[7 * Ns] = tie; o[8 * Ns] = 0.f;
#pragma unroll
    for (int c = 0; c < kChannels; ++c) cur[c] = nxt[c];
  }
  if (p.lpf_state && blockIdx.y == 0) {
    p.lpf_state[n] = la.x; p.lpf_state[Ns + n] = la.y; p.lpf_state[2 * Ns + n] = la.z;
    p.lpf_state[3 * Ns + n] = lm.x; p.lpf_state[4 * Ns + n] = lm.y; p.lpf_state[5 * Ns + n] = lm.z;
  }
}

// trajectory [M][4] -> roll/pitch/yaw degrees [M][3]   (PKF/UtilityFunctions.py:3-14 per row)
__global__ void __launch_bounds__(256) traj2rpy_kernel(int64_t M, const float4* __restrict__ q, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  const float4 v = q[i];
  const float w = v.x, x = v.y, y = v.z, z = v.w, k = 57.29577951308232f;
  // products that feed a sum or difference go through one FMA (one rounding instead of two where the terms cancel)
  out[3 * i] = atan2f(2.f * fmaf(w, x, y * z), fmaf(-2.f, fmaf(x, x, y * y), 1.f)) * k;
  out[3 * i + 1] = asinf(2.f * fmaf(w, y, -(z * x))) * k;
  out[3 * i + 2] = atan2f(2.f * fmaf(w, z, x * y), fmaf(-2.f, fmaf(y, y, z * z), 1.f)) * k;
}

// Packed form of the rank-2 Wahba kernel: two solves per thread in f32x2 lanes (N even, per-pair or
// shared references).  Same arithmetic per solve as wahba_kernel<WAHBA_QR2>.
// The kernel is memory-bound (40 B per solve against ~250 FP32 operations), so it is written as a
// grid-stride loop over a resident grid with the NEXT pair's six 8-byte loads issued before the current
// pair is solved and stored: every thread always has 48-96 B of reads in flight instead of alternating
// between a load phase and a compute/store phase.  With shared references the frame of (acc_0, mag_0) is
// built once per thread, outside the loop.
struct Wahba2Inputs { Vec3<f32x2> a, m; f32x2 ka, km; };
__device__ __forceinline__ f32x2 ld2_stream(const float* q) {
  float2 v;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(q));
  return f32x2(v.x, v.y);
}
__device__ __forceinline__ void st2_stream(float* q, const f32x2& v) {
  asm volatile("st.global.cs.v2.f32 [%0], {%1, %2};" ::"l"(q), "f"(v.x), "f"(v.y) : "memory");
}
__device__ __forceinline__ Wahba2Inputs wahba2_load(const WahbaParams& p, int64_t n) {
  const int64_t N = p.N;
  Wahba2Inputs in;
  in.a = {ld2_stream(p.acc + n), ld2_stream(p.acc + N + n), ld2_stream(p.acc + 2 * N + n)};
  in.m = {ld2_stream(p.mag + n), ld2_stream(p.mag + N + n), ld2_stream(p.mag + 2 * N + n)};
  if (p.k_acc) { in.ka = ld2_stream(p.k_acc + n); in.km = ld2_stream(p.k_mag + n); }
  else { in.ka = f32x2(p.k_acc_s); in.km = f32x2(p.k_mag_s); }
  return in;
}
#ifndef PKF_WAHBA2_MIN_CTAS
#define PKF_WAHBA2_MIN_CTAS 3
#endif
__global__ void __launch_bounds__(256, PKF_WAHBA2_MIN_CTAS) wahba2_kernel(const WahbaParams p) {
  const int64_t N = p.N;
  const int64_t stride = 2 * (int64_t)gridDim.x * blockDim.x;
  int64_t n = 2 * ((int64_t)blockIdx.x * blockDim.x + threadIdx.x);
  if (n >= N) return;
  RefFrame<f32x2> E;
  if (p.ref_shared) {
    const Vec3<f32x2> ra = {f32x2(__ldg(p.acc_ref)), f32x2(__ldg(p.acc_ref + 1)), f32x2(__ldg(p.acc_ref + 2))};
    const Vec3<f32x2> rm = {f32x2(__ldg(p.mag_ref)), f32x2(__ldg(p.mag_ref + 1)), f32x2(__ldg(p.mag_ref + 2))};
    E = frame_from_pair<f32x2>(ra, rm);
  }
  Wahba2Inputs cur = wahba2_load(p, n);
  while (true) {
    const int64_t nn = n + stride;
    const bool more = nn < N;
    Wahba2Inputs nxt = cur;
    if (more) nxt = wahba2_load(p, nn);              // in flight while the current pair is solved
    if (!p.ref_shared) {
      const Vec3<f32x2> ra = {ld2(p.acc_ref + n), ld2(p.acc_ref + N + n), ld2(p.acc_ref + 2 * N + n)};
      const Vec3<f32x2> rm = {ld2(p.mag_ref + n), ld2(p.mag_ref + N + n), ld2(p.mag_ref + 2 * N + n)};
      E = frame_from_pair<f32x2>(ra, rm);
    }
    f32x2 ka = cur.ka, km = cur.km;
    if (!p.k_acc && p.weights_from_acc) { ka = abs_<f32x2>(cur.a.z); km = f32x2(1.f) - ka; }   // PKF/ExtendedKalmanFilter.py:71
    const Mat3<f32x2> R = wahba_qr2<f32x2>(E, cur.a, cur.m, ka, km);
    if (p.out_rot) {
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) st2_stream(p.out_rot + (3 * r + c) * N + n, R.m[r][c]);
    }
    if (p.out_quat) {
      const Quat<f32x2> q = rotation_to_quat_ref<f32x2>(R);
      st2_stream(p.out_quat + n, q.w); st2_stream(p.out_quat + N + n, q.x);
      st2_stream(p.out_quat + 2 * N + n, q.y); st2_stream(p.out_quat + 3 * N + n, q.z);
    }
    if (!more) break;
    cur = nxt; n = nn;
  }
}

// Packed form of the Wahba-only comparison track (tracks_kernel's second output): two filters per thread in f32x2
// lanes, one thread walks its pair of filters through time with the next step's six 8-byte loads in flight while the
// current pair of samples is solved and stored as two float4 quaternions.  Same arithmetic per sample as
// tracks_kernel<WAHBA_QR2> (bit-identical results); needs N even, Ns == N and 8-byte aligned rows.
__global__ void __launch_bounds__(128) tracks_wahba2_kernel(const TracksParams p) {
  const int64_t n = 2 * ((int64_t)blockIdx.x * blockDim.x + threadIdx.x);
  if (n >= p.N) return;
  const int64_t N = p.N;
  const Vec3<f32x2> ra = {ld2(p.acc_ref + n), ld2(p.acc_ref + N + n), ld2(p.acc_ref + 2 * N + n)};
  const Vec3<f32x2> rm = {ld2(p.mag_ref + n), ld2(p.mag_ref + N + n), ld2(p.mag_ref + 2 * N + n)};
  const RefFrame<f32x2> E = frame_from_pair<f32x2>(ra, rm);
  float4* ow = reinterpret_cast<float4*>(p.out_wahba) + n;
  const float* s = p.streams + n;
  // TWO steps ahead in flight (96 B per thread): one thread walks its filters through time, so the memory-level
  // parallelism has to come from the depth of its own prefetch
  f32x2 cur[6], nx1[6], nx2[6];
  auto load_step = [&](f32x2 (&v)[6], const float* q) {
#pragma unroll
    for (int c = 0; c < 6; ++c) v[c] = ld2_stream(q + (3 + c) * N);
  };
  const int64_t step = kChannels * N;
  if (p.T > 0) load_step(cur, s);
  if (p.T > 1) load_step(nx1, s + step);
  for (int64_t t = 0; t < p.T; ++t, s += step) {
    if (t + 2 < p.T) load_step(nx2, s + 2 * step);
    const Vec3<f32x2> a = {cur[0], cur[1], cur[2]}, m = {cur[3], cur[4], cur[5]};
    f32x2 ka(p.k_acc), km(p.k_mag);
    if (p.weights_from_acc) { ka = abs_<f32x2>(a.z); km = f32x2(1.f) - ka; }
    const Quat<f32x2> q = rotation_to_quat_ref<f32x2>(wahba_qr2<f32x2>(E, a, m, ka, km));
    stg_stream4(ow, q.w.x, q.x.x, q.y.x, q.z.x);
    stg_stream4(ow + 1, q.w.y, q.x.y, q.y.y, q.z.y);
    ow += N;
#pragma unroll
    for (int c = 0; c < 6; ++c) { cur[c] = nx1[c]; nx1[c] = nx2[c]; }
  }
}

__global__ void __launch_bounds__(256) rot2quat_kernel(int64_t N, const float* __restrict__ rot, float* __restrict__ out) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  Mat3<float> R;
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) R.m[r][c] = rot[(3 * r + c) * N + n];
  // The stand-alone operator accepts ANY 3x3 the reference accepts.  A rotation (M^T M = I to 1e-3: every matrix the
  // Wahba stage produces) goes through rotation_to_quat_ref: the best-conditioned Shepperd candidate with the
  // reference's sign rule -- the reference's own formula divides by S = 2 sqrt(tr_i) -> 0 near the identity, which
  // float64 survives and a float32 INPUT matrix does not (its 1e-7 rounding would come out as 1e-5).  Anything else
  // (scaled, sheared) evaluates the reference's three branches literally, in float64 on the float32 inputs
  // (PKF/Wahba.py:20-47): the reference's un-normalised vector to the rounding of the float32 output.
  float ortho = 0.f;
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = i; j < 3; ++j) {
      const float d = R.m[0][i] * R.m[0][j] + R.m[1][i] * R.m[1][j] + R.m[2][i] * R.m[2][j] - (i == j ? 1.f : 0.f);
      ortho = fmaxf(ortho, fabsf(d));
    }
  if (ortho < 1e-3f) {
    const Quat<float> q = rotation_to_quat_ref<float>(R);
    out[n] = q.w; out[N + n] = q.x; out[2 * N + n] = q.y; out[3 * N + n] = q.z;
    return;
  }
  const double m00 = R.m[0][0], m01 = R.m[0][1], m02 = R.m[0][2], m10 = R.m[1][0], m11 = R.m[1][1], m12 = R.m[1][2],
               m20 = R.m[2][0], m21 = R.m[2][1], m22 = R.m[2][2];
  const double tr1 = 1.0 + m00 - m11 - m22, tr2 = 1.0 - m00 + m11 - m22, tr3 = 1.0 - m00 - m11 + m22;
  double qw, qx, qy, qz;
  if (tr1 > tr2 && tr1 > tr3) {
    const double S = sqrt(tr1) * 2.0;
    qw = (m21 - m12) / S; qx = 0.25 * S; qy = (m01 + m10) / S; qz = (m02 + m20) / S;
  } else if (tr2 > tr1 && tr2 > tr3) {
    const double S = sqrt(tr2) * 2.0;
    qw = (m02 - m20) / S; qx = (m01 + m10) / S; qy = 0.25 * S; qz = (m12 + m21) / S;
  } else {
    const double S = sqrt(tr3) * 2.0;
    qw = (m10 - m01) / S; qx = (m02 + m20) / S; qy = (m12 + m21) / S; qz = 0.25 * S;
  }
  out[n] = (float)qw; out[N + n] = (float)qx; out[2 * N + n] = (float)qy; out[3 * N + n] = (float)qz;
}

// ---------------------------------------------------------------------------------------------
// General Prediction / Correction (full matrices, exactly the reference's operations).
// ---------------------------------------------------------------------------------------------
struct PredictParams {
  int64_t N;
  const float *gyro, *dt;
  int dt_shared;
  const float *x, *p, *q_mat, *r_mat, *q_scale, *r_scale;
  float *out_z, *out_p, *out_k;
};

__global__ void __launch_bounds__(128) predict_kernel(const PredictParams a) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= a.N) return;
  const int64_t N = a.N;
  Vec3<float> w = {a.gyro[n], a.gyro[N + n], a.gyro[2 * N + n]};
  Quat<float> x = {a.x[n], a.x[N + n], a.x[2 * N + n], a.x[3 * N + n]};
  Mat4<float> P, A, AP, S, Si;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) P.m[i][j] = a.p[(4 * i + j) * N + n];
  half_omega<float>(w, A);                                      // GetJacobian_A  :43-48
  // GetJacobian_B(x)  :51-56
  const float B[4][3] = {{-0.5f * x.x, -0.5f * x.y, -0.5f * x.z},
                         {0.5f * x.w, 0.5f * x.z, -0.5f * x.y},
                         {-0.5f * x.z, 0.5f * x.w, 0.5f * x.x},
                         {0.5f * x.y, -0.5f * x.x, 0.5f * x.w}};
  const float qs = a.q_scale ? a.q_scale[n] : 1.f, rs = a.r_scale ? a.r_scale[n] : 1.f;
  float BQ[4][3];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      float acc = 0.f;
#pragma unroll
      for (int k = 0; k < 3; ++k) acc = fmaf(B[i][k], qs * __ldg(a.q_mat + 3 * k + j), acc);
      BQ[i][j] = acc;
    }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float acc = 0.f;
#pragma unroll
      for (int k = 0; k < 4; ++k) acc = fmaf(A.m[i][k], P.m[k][j], acc);
      AP.m[i][j] = acc;
    }
  Mat4<float> Pn;                                               // P = A P A^T + B Q B^T   :61
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float acc = 0.f;
#pragma unroll
      for (int k = 0; k < 4; ++k) acc = fmaf(AP.m[i][k], A.m[j][k], acc);
#pragma unroll
      for (int k = 0; k < 3; ++k) acc = fmaf(BQ[i][k], B[j][k], acc);
      Pn.m[i][j] = acc;
      S.m[i][j] = acc + rs * __ldg(a.r_mat + 4 * i + j);        // S = P + R   :63
    }
  const float h = a.dt_shared ? a.dt[0] : a.dt[n];
  Vec3<float> hw = {0.5f * w.x, 0.5f * w.y, 0.5f * w.z};
  Quat<float> z = rk4_step<float>(x, hw, h);                    // :62
  inverse4<float>(S, Si);                                       // :65
  a.out_z[n] = z.w; a.out_z[N + n] = z.x; a.out_z[2 * N + n] = z.y; a.out_z[3 * N + n] = z.z;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float acc = 0.f;                                          // K = P S^-1   :66
#pragma unroll
      for (int k = 0; k < 4; ++k) acc = fmaf(Pn.m[i][k], Si.m[k][j], acc);
      a.out_k[(4 * i + j) * N + n] = acc;
      a.out_p[(4 * i + j) * N + n] = Pn.m[i][j];
    }
}

struct CorrectParams {
  int64_t N;
  const float *mag, *acc, *acc_ref, *mag_ref;
  int ref_shared;
  const float *z, *p, *k;
  float *out_x, *out_p;
  uint8_t* out_flip;
  float* out_meas;
};

template <int ALGO> __global__ void __launch_bounds__(128) correct_kernel(const CorrectParams a) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= a.N) return;
  const int64_t N = a.N;
  Vec3<float> ra, rm;
  if (a.ref_shared) {
    ra = {a.acc_ref[0], a.acc_ref[1], a.acc_ref[2]};
    rm = {a.mag_ref[0], a.mag_ref[1], a.mag_ref[2]};
  } else {
    ra = {a.acc_ref[n], a.acc_ref[N + n], a.acc_ref[2 * N + n]};
    rm = {a.mag_ref[n], a.mag_ref[N + n], a.mag_ref[2 * N + n]};
  }
  Vec3<float> ac = {a.acc[n], a.acc[N + n], a.acc[2 * N + n]};
  Vec3<float> mg = {a.mag[n], a.mag[N + n], a.mag[2 * N + n]};
  Quat<float> z = {a.z[n], a.z[N + n], a.z[2 * N + n], a.z[3 * N + n]};
  const float ka = fabsf(ac.z), km = 1.f - ka;                                     // :71
  Mat3<float> R = (ALGO == WAHBA_QR2) ? wahba_qr2<float>(frame_from_pair<float>(ra, rm), ac, mg, ka, km)
                                      : wahba_jacobi<float>(ra, rm, ac, mg, ka, km, 6);
  Quat<float> y = rotation_to_quat_ref<float>(R);
  const bool flip = dot4(y, z) < 0.f;                                              // :73-74 (Comparator[0] == dot)
  if (flip) { y.w = -y.w; y.x = -y.x; y.y = -y.y; y.z = -y.z; }
  const float e[4] = {y.w - z.w, y.x - z.x, y.y - z.y, y.z - z.z};                 // :76
  float K[4][4], P[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) { K[i][j] = a.k[(4 * i + j) * N + n]; P[i][j] = a.p[(4 * i + j) * N + n]; }
  const float zz[4] = {z.w, z.x, z.y, z.z};
  float X[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float acc = zz[i];                                                             // X = z + K e   :77
#pragma unroll
    for (int j = 0; j < 4; ++j) acc = fmaf(K[i][j], e[j], acc);
    X[i] = acc;
  }
  const float inv = rsqrtf(fmaf(X[3], X[3], fmaf(X[2], X[2], fmaf(X[1], X[1], X[0] * X[0]))));
#pragma unroll
  for (int i = 0; i < 4; ++i) a.out_x[i * N + n] = X[i] * inv;                     // :79
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float acc = P[i][j];                                                         // P = P - K P   :78
#pragma unroll
      for (int k = 0; k < 4; ++k) acc = fmaf(-K[i][k], P[k][j], acc);
      a.out_p[(4 * i + j) * N + n] = acc;
    }
  if (a.out_flip) a.out_flip[n] = flip ? 1 : 0;
  if (a.out_meas) { a.out_meas[n] = y.w; a.out_meas[N + n] = y.x; a.out_meas[2 * N + n] = y.y; a.out_meas[3 * N + n] = y.z; }
}

__global__ void __launch_bounds__(256)
    rk4_kernel(int64_t N, const float* q, const float* dt, int dt_shared, const float* w, float* out) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  Quat<float> x = {q[n], q[N + n], q[2 * N + n], q[3 * N + n]};
  Vec3<float> hw = {0.5f * w[n], 0.5f * w[N + n], 0.5f * w[2 * N + n]};
  Quat<float> z = rk4_step<float>(x, hw, dt_shared ? dt[0] : dt[n]);
  out[n] = z.w; out[N + n] = z.x; out[2 * N + n] = z.y; out[3 * N + n] = z.z;
}

__global__ void __launch_bounds__(256)
    jacobians_kernel(int64_t N, const float* w, float* out_a, const float* q, float* out_b) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  if (w && out_a) {
    Mat4<float> A;
    half_omega<float>({w[n], w[N + n], w[2 * N + n]}, A);
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) out_a[(4 * i + j) * N + n] = A.m[i][j];
  }
  if (q && out_b) {
    const float q0 = 0.5f * q[n], q1 = 0.5f * q[N + n], q2 = 0.5f * q[2 * N + n], q3 = 0.5f * q[3 * N + n];
    const float B[12] = {-q1, -q2, -q3, q0, q3, -q2, -q3, q0, q1, q2, -q1, q0};
#pragma unroll
    for (int i = 0; i < 12; ++i) out_b[i * N + n] = B[i];
  }
}

__global__ void __launch_bounds__(256) comparator_kernel(int64_t N, const float* q1, const float* q2, float* out) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  // conj(q1) (x) q2, written as the reference's 4x4 mat-vec (PKF/ExtendedKalmanFilter.py:17-23)
  const float c0 = q1[n], c1 = -q1[N + n], c2 = -q1[2 * N + n], c3 = -q1[3 * N + n];
  const float b0 = q2[n], b1 = q2[N + n], b2 = q2[2 * N + n], b3 = q2[3 * N + n];
  out[n] = fmaf(-c3, b3, fmaf(-c2, b2, fmaf(-c1, b1, c0 * b0)));
  out[N + n] = fmaf(c2, b3, fmaf(-c3, b2, fmaf(c0, b1, c1 * b0)));
  out[2 * N + n] = fmaf(-c1, b3, fmaf(c0, b2, fmaf(c3, b1, c2 * b0)));
  out[3 * N + n] = fmaf(c0, b3, fmaf(c1, b2, fmaf(-c2, b1, c3 * b0)));
}

__global__ void __launch_bounds__(256)
    lowpass_kernel(int64_t N, int64_t T, const float* x, float alpha, float* state, float* out) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  Vec3<float> y = {state[n], state[N + n], state[2 * N + n]};
  const float oma = 1.f - alpha;
  for (int64_t t = 0; t < T; ++t) {
    const float* xi = x + t * 3 * N + n;
    Vec3<float> v = {ldg_stream(xi), ldg_stream(xi + N), ldg_stream(xi + 2 * N)};
    lowpass<float>(y, v, alpha, oma);
    float* o = out + t * 3 * N + n;
    o[0] = y.x; o[N] = y.y; o[2 * N] = y.z;
  }
  state[n] = y.x; state[N + n] = y.y; state[2 * N + n] = y.z;
}

__global__ void __launch_bounds__(256) quat2rpy_kernel(int64_t N, const float* q, float* out) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  // The stand-alone operator evaluates the reference's float64 expressions (PKF/UtilityFunctions.py:3-14) in float64
  // on the float32 inputs: the result is the reference's value to the rounding of the float32 output (~1e-5 deg).
  // (The streaming form over a stored trajectory, traj2rpy_kernel, stays in float32.)
  const double w = q[n], x = q[N + n], y = q[2 * N + n], z = q[3 * N + n];
  const double k = 57.29577951308232;
  out[n] = (float)(atan2(2.0 * (w * x + y * z), 1.0 - 2.0 * (x * x + y * y)) * k);
  out[N + n] = (float)(asin(2.0 * (w * y - z * x)) * k);
  out[2 * N + n] = (float)(atan2(2.0 * (w * z + x * y), 1.0 - 2.0 * (y * y + z * z)) * k);
}

__global__ void __launch_bounds__(256) norm_kernel(int64_t N, int k, const float* v, float* out) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float acc = 0.f;
  for (int i = 0; i < k; ++i) { const float e = v[(int64_t)i * N + n]; acc = fmaf(e, e, acc); }   // left to right, :18-19
  out[n] = sqrtf(acc);
}

// Sign fix-up of a measurement stream (see measurement_stream_kernel): one thread per (step, stream).
__global__ void __launch_bounds__(256) meas_fixup_kernel(const MeasStreamParams p) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.Ns * p.T) return;
  const int64_t t = i / p.Ns, n = i - t * p.Ns, Ns = p.Ns;
  float* o = p.out + t * kChannels * Ns + n;
  if (o[7 * Ns] == 0.f) return;
  const float* s = p.streams + t * kChannels * Ns + n;
  const float az = s[5 * Ns], ka = fabsf(az);
  const int branch = reference_branch_exact(p.acc_ref[n], p.acc_ref[Ns + n], p.acc_ref[2 * Ns + n], p.mag_ref[n], p.mag_ref[Ns + n],
                                            p.mag_ref[2 * Ns + n], s[3 * Ns], s[4 * Ns], az, s[6 * Ns], s[7 * Ns], s[8 * Ns], ka, 1.f - ka);
  if (o[(4 + branch) * Ns] < 0.f) {       // the reference's quaternion has component `branch` >= 0 (PKF/Wahba.py:28,35,41)
#pragma unroll
    for (int c = 3; c < 7; ++c) o[c * Ns] = -o[c * Ns];
  }
  o[7 * Ns] = 0.f;
}

// ---------------------------------------------------------------------------------------------
// Flip-mask fix-up: the replay kernels mark the (few per 1e5) steps where the reference's 3-branch sign rule
// (PKF/Wahba.py:26-47) sits on a float32 tie of two squared components -- byte = 0x80 | alternatives << 1 | float32
// decision, see reference_flip_quat -- and this pass settles them in float64 from the raw sample and reference vectors,
// the values the float64 reference itself consumes: the stored mask is then IDENTICAL to ExtendedKalmanFilter.py:73-75.
// One thread per four mask bytes; unmarked bytes are not rewritten.
// ---------------------------------------------------------------------------------------------
struct FlipFixupParams {
  int64_t N, T, Ns;
  const float* streams;      // [T][9][Ns]
  const float *acc_ref, *mag_ref;
  uint8_t* flips;            // [T][N]
};
__global__ void __launch_bounds__(256) flip_fixup_kernel(const FlipFixupParams p) {
  const int64_t total = p.N * p.T;
  const int64_t i0 = 4 * ((int64_t)blockIdx.x * blockDim.x + threadIdx.x);
  if (i0 >= total) return;
  unsigned word = 0;
  const bool aligned4 = (reinterpret_cast<uintptr_t>(p.flips) & 3) == 0 && i0 + 4 <= total;
  if (aligned4) word = *reinterpret_cast<const unsigned*>(p.flips + i0);
  else for (int k = 0; k < 4 && i0 + k < total; ++k) word |= (unsigned)p.flips[i0 + k] << (8 * k);
  if ((word & 0x80808080u) == 0u) return;
  for (int k = 0; k < 4; ++k) {
    const unsigned b = (word >> (8 * k)) & 0xffu;
    if (!(b & 0x80u)) continue;
    const int64_t i = i0 + k, t = i / p.N, n = i - t * p.N, col = (p.Ns == p.N) ? n : (n % p.Ns);
    const float* s = p.streams + t * kChannels * p.Ns + col;
    const float az = s[5 * p.Ns], ka = fabsf(az);                       // PKF/ExtendedKalmanFilter.py:71
    const int branch = reference_branch_exact(p.acc_ref[col], p.acc_ref[p.Ns + col], p.acc_ref[2 * p.Ns + col], p.mag_ref[col],
                                              p.mag_ref[p.Ns + col], p.mag_ref[2 * p.Ns + col], s[3 * p.Ns], s[4 * p.Ns], az,
                                              s[6 * p.Ns], s[7 * p.Ns], s[8 * p.Ns], ka, 1.f - ka);
    p.flips[i] = (uint8_t)((b >> (1 + branch)) & 1u);
  }
}

// host-replay helpers: initial state and P <-> P/r conversion on the device
__global__ void __launch_bounds__(256)
    host_init_state_kernel(int64_t N, int have_x0, int have_p0, const float* __restrict__ r, float* x, float* p, float dt,
                           float* dt_out) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  if (n == 0) *dt_out = dt;
  if (!have_x0) { x[n] = 1.f; x[N + n] = 0.f; x[2 * N + n] = 0.f; x[3 * N + n] = 0.f; }     // PKF/main_file.py:26
  const float ir = 1.f / r[n];
#pragma unroll
  for (int k = 0; k < 10; ++k) {
    const bool diag = (k == 0 || k == 4 || k == 7 || k == 9);
    const float p0 = have_p0 ? p[k * N + n] : (diag ? 1.f : 0.f);                            // PKF/main_file.py:23
    p[k * N + n] = p0 * ir;
  }
}
__global__ void __launch_bounds__(256) host_unscale_p_kernel(int64_t N, const float* __restrict__ r, float* p) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const float rr = r[n];
#pragma unroll
  for (int k = 0; k < 10; ++k) p[k * N + n] *= rr;
}

// FP32 peak probe: 16 independent FFMA chains per thread, all SMs full.
constexpr int kProbeIters = 8192, kProbeAcc = 16;
__global__ void __launch_bounds__(256) fp32_probe_kernel(float* out, float b, float c) {
  float a[kProbeAcc];
#pragma unroll
  for (int i = 0; i < kProbeAcc; ++i) a[i] = threadIdx.x * 1e-3f + i;
  for (int it = 0; it < kProbeIters; ++it) {
#pragma unroll
    for (int i = 0; i < kProbeAcc; ++i) a[i] = fmaf(a[i], b, c);
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < kProbeAcc; ++i) s += a[i];
  out[(int64_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// ---------------------------------------------------------------------------------------------
}  // namespace pkf_dev
