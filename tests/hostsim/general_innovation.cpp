// general_innovation.cpp -- CPU build of the innovation terms and the gate of the general-matrix step of
// poseestimationkf_b200/csrc/ekf_math.cuh (GEN with INNOV / GATE).
//
// TEST TOOL ONLY (like general_qr.cpp beside it): the replay the GEN innovation kernels run, computed by the same header
// in float32 and float64, with the per-step terms, the gate decisions and the running sums of the same build, for the
// `-m "not gpu"` tests.  Compiled by tests/hostsim/general_innovation.py.
#include <cmath>
#include <cstdint>
#include <cstddef>
#include "../../poseestimationkf_b200/csrc/ekf_math.cuh"

using namespace pkf;

// One launch from the reference's initial state (X = [1,0,0,0], P = I), as the kernels run it: filter frame in, out.
// q_tri [6][N], r_tri [10][N] (upper triangles).  terms [2][T][N] (NIS_t, ln det S_t of the model), gated [T][N],
// innov [2][N] the running sums, traj [T][N][4] reference frame.
template <typename F, int ALGO, bool TAN, bool GATE>
static void replay_t(int64_t N, int64_t T, const float* streams, const double* dt, int dt_per_step, const float* acc_ref,
                     const float* mag_ref, const float* q_tri, const float* r_tri, float gamma, double* terms,
                     uint8_t* gated_out, double* innov, double* traj) {
  for (int64_t n = 0; n < N; ++n) {
    Vec3<F> ra = {(F)acc_ref[n], (F)acc_ref[N + n], (F)acc_ref[2 * N + n]};
    Vec3<F> rm = {(F)mag_ref[n], (F)mag_ref[N + n], (F)mag_ref[2 * N + n]};
    FilterConst<F> fc = make_filter_const<F>(ra, rm, F(4), F(1));
    F q6[6], r10[10];
    for (int k = 0; k < 6; ++k) q6[k] = (F)q_tri[k * N + n];
    for (int k = 0; k < 10; ++k) r10[k] = (F)r_tri[k * N + n];
    Quat<F> x = {F(1), F(0), F(0), F(0)}, xlo = {F(0), F(0), F(0), F(0)};
    Sym4<F> P = {F(1), F(0), F(0), F(0), F(1), F(0), F(0), F(1), F(0), F(1)};
    adopt_state(fc, x, xlo);
    const bool frame = uses_filter_frame<ALGO>();
    if (frame) enter_filter_frame(fc, x, xlo, P, false);
    const GenQR<F> gq = make_gen_qr<F>(fc, q6, r10, frame);
    InnovAcc<F> acc = make_innov_acc<F, TAN>(F(0), F(0), F(1));
    const GateParams<F> gp = make_gate_params<F>(F(1), gamma);
    for (int64_t t = 0; t < T; ++t) {
      const float* s = streams + (size_t)t * 9 * N;
      Vec3<F> w = {(F)s[n], (F)s[N + n], (F)s[2 * N + n]};
      Vec3<F> a = {(F)s[3 * N + n], (F)s[4 * N + n], (F)s[5 * N + n]};
      Vec3<F> m = {(F)s[6 * N + n], (F)s[7 * N + n], (F)s[8 * N + n]};
      const F h = F((float)(dt_per_step ? dt[t] : dt[0]));
      bool flip, gated = false;
      InnovTerms<F> it;
      ekf_step<F, ALGO, true, false, true, TAN, GATE, true>(x, xlo, P, fc, w, a, m, StepH<F>(h), flip, true, nullptr, &acc,
                                                           GATE ? &gp : nullptr, &gated, &gq, &it);
      terms[(size_t)t * N + n] = (double)it.nis;
      terms[(size_t)(T + t) * N + n] = (double)it.logdet;
      gated_out[(size_t)t * N + n] = gated ? 1 : 0;
      const Quat<F> xr = frame ? state_in_reference_frame(fc, x) : x;
      double* row = traj + ((size_t)t * N + n) * 4;
      row[0] = xr.w; row[1] = xr.x; row[2] = xr.y; row[3] = xr.z;
    }
    innov[n] = (double)acc.nis;
    innov[N + n] = (double)acc.logdet;
  }
}

extern "C" {

// precision: 0 = float32, 1 = float64; algo: 0 = QR2, 1 = Jacobi, 2 = precomputed; model: 0 = full, 1 = tangent;
// gate: 1 = gated at gamma.
int hostsim_general_innovation(int precision, int algo, int model, int gate, float gamma, int64_t N, int64_t T,
                               const float* streams, const double* dt, int dt_per_step, const float* acc_ref,
                               const float* mag_ref, const float* q_tri, const float* r_tri, double* terms, uint8_t* gated,
                               double* innov, double* traj) {
#define GO(F, A, TAN, G) replay_t<F, A, TAN, G>(N, T, streams, dt, dt_per_step, acc_ref, mag_ref, q_tri, r_tri, gamma, terms, gated, innov, traj)
#define GATED(F, A, TAN) do { if (gate) GO(F, A, TAN, true); else GO(F, A, TAN, false); } while (0)
#define MODEL(F, A) do { if (model) GATED(F, A, true); else GATED(F, A, false); } while (0)
#define ALG(F) do { if (algo == 0) MODEL(F, WAHBA_QR2); else if (algo == 1) MODEL(F, WAHBA_JACOBI); else MODEL(F, WAHBA_PRECOMPUTED); } while (0)
  if (algo < 0 || algo > 2 || model < 0 || model > 1) return 1;
  if (precision == 0) ALG(float);
  else if (precision == 1) ALG(double);
  else return 1;
#undef ALG
#undef MODEL
#undef GATED
#undef GO
  return 0;
}

}  // extern "C"
