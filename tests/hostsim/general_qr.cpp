// general_qr.cpp -- CPU build of the general-matrix step of poseestimationkf_b200/csrc/ekf_math.cuh (GEN).
//
// TEST TOOL ONLY (like gating.cpp beside it): the replay the GEN kernels run, computed by the same header in float32
// and float64, plus the isotropic step of the same build for comparison, for the `-m "not gpu"` tests.
// Compiled by tests/hostsim/general_qr.py.
#include <cstdint>
#include <cstddef>
#include "../../poseestimationkf_b200/csrc/ekf_math.cuh"

using namespace pkf;

// One launch from the reference's initial state (X = [1,0,0,0], P = I), as the kernels run it: filter frame in, out.
// GEN: q_tri [6][N] and r_tri [10][N] (upper triangles); otherwise the isotropic step with q = q_tri[0], r = r_tri[0]
// (P carried in units of r, converted back on output).
template <typename F, int ALGO, bool GEN>
static void replay_t(int64_t N, int64_t T, const float* streams, const double* dt, int dt_per_step, const float* acc_ref,
                     const float* mag_ref, const float* q_tri, const float* r_tri, double* traj, uint8_t* flips,
                     double* x_out, double* p_out) {
  for (int64_t n = 0; n < N; ++n) {
    Vec3<F> ra = {(F)acc_ref[n], (F)acc_ref[N + n], (F)acc_ref[2 * N + n]};
    Vec3<F> rm = {(F)mag_ref[n], (F)mag_ref[N + n], (F)mag_ref[2 * N + n]};
    const F rr = GEN ? F(1) : (F)r_tri[n];
    FilterConst<F> fc = make_filter_const<F>(ra, rm, GEN ? F(4) : (F)q_tri[n], rr);
    F q6[6], r10[10];
    for (int k = 0; k < 6; ++k) q6[k] = (F)q_tri[k * N + n];
    for (int k = 0; k < 10; ++k) r10[k] = (F)r_tri[k * N + n];
    Quat<F> x = {F(1), F(0), F(0), F(0)}, xlo = {F(0), F(0), F(0), F(0)};
    const F ir = F(1) / rr;
    Sym4<F> P = {ir, F(0), F(0), F(0), ir, F(0), F(0), ir, F(0), ir};
    adopt_state(fc, x, xlo);
    const bool frame = uses_filter_frame<ALGO>();
    if (frame) enter_filter_frame(fc, x, xlo, P, false);
    const GenQR<F> gq = make_gen_qr<F>(fc, q6, r10, frame);
    for (int64_t t = 0; t < T; ++t) {
      const float* s = streams + (size_t)t * 9 * N;
      Vec3<F> w = {(F)s[n], (F)s[N + n], (F)s[2 * N + n]};
      Vec3<F> a = {(F)s[3 * N + n], (F)s[4 * N + n], (F)s[5 * N + n]};
      Vec3<F> m = {(F)s[6 * N + n], (F)s[7 * N + n], (F)s[8 * N + n]};
      const F h = F((float)(dt_per_step ? dt[t] : dt[0]));
      bool flip;
      ekf_step<F, ALGO, true, false, false, false, false, GEN>(x, xlo, P, fc, w, a, m, StepH<F>(h), flip, true, nullptr,
                                                               nullptr, nullptr, (bool*)nullptr, GEN ? &gq : nullptr);
      flips[(size_t)t * N + n] = flip ? 1 : 0;
      const Quat<F> xr = frame ? state_in_reference_frame(fc, x) : x;
      double* row = traj + ((size_t)t * N + n) * 4;
      row[0] = xr.w; row[1] = xr.x; row[2] = xr.y; row[3] = xr.z;
    }
    if (frame) leave_filter_frame(fc, x, xlo, P, false);
    x_out[n] = x.w; x_out[N + n] = x.x; x_out[2 * N + n] = x.y; x_out[3 * N + n] = x.z;
    const F pv[10] = {P.a00, P.a01, P.a02, P.a03, P.a11, P.a12, P.a13, P.a22, P.a23, P.a33};
    for (int k = 0; k < 10; ++k) p_out[k * N + n] = (double)pv[k] * (double)rr;
  }
}

extern "C" {

// precision: 0 = float32, 1 = float64; algo: 0 = QR2, 1 = Jacobi, 2 = precomputed (stream rows 3-6 hold the Wahba
// quaternion); general: 1 = the GEN step with q_tri [6][N], r_tri [10][N], 0 = the isotropic step with q_tri [N],
// r_tri [N].  traj [T][N][4] reference frame, flips [T][N], x [4][N] and p [10][N] (unscaled) after the last step.
int hostsim_general_qr(int precision, int algo, int general, int64_t N, int64_t T, const float* streams, const double* dt,
                       int dt_per_step, const float* acc_ref, const float* mag_ref, const float* q_tri, const float* r_tri,
                       double* traj, uint8_t* flips, double* x, double* p) {
#define GO(F, A) do { if (general) replay_t<F, A, true>(N, T, streams, dt, dt_per_step, acc_ref, mag_ref, q_tri, r_tri, traj, flips, x, p); \
                      else replay_t<F, A, false>(N, T, streams, dt, dt_per_step, acc_ref, mag_ref, q_tri, r_tri, traj, flips, x, p); } while (0)
#define ALG(F) do { if (algo == 0) GO(F, WAHBA_QR2); else if (algo == 1) GO(F, WAHBA_JACOBI); else GO(F, WAHBA_PRECOMPUTED); } while (0)
  if (algo < 0 || algo > 2) return 1;
  if (precision == 0) ALG(float);
  else if (precision == 1) ALG(double);
  else return 1;
#undef ALG
#undef GO
  return 0;
}

}  // extern "C"
