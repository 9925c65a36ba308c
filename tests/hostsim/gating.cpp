// gating.cpp -- CPU build of the innovation gate of poseestimationkf_b200/csrc/ekf_math.cuh (GATE).
//
// TEST TOOL ONLY (like innovation_tangent.cpp beside it): the replay the GATE kernels run, computed by the same header
// in float32, float64 and the packed f32x2 lanes, with and without the gate, for the `-m "not gpu"` tests.
// Compiled by tests/hostsim/gating.py.
#include <cstdint>
#include <cstddef>
#include "../../poseestimationkf_b200/csrc/ekf_math.cuh"

using namespace pkf;

template <typename F> static F lanes_(const float* v, int64_t n) { return (F)v[n]; }
template <> f32x2 lanes_<f32x2>(const float* v, int64_t n) { return f32x2(v[n], v[n + 1]); }
template <typename F> static void put_(double* o, int64_t n, const F& v) { o[n] = v; }
template <> void put_<f32x2>(double* o, int64_t n, const f32x2& v) { o[n] = v.x; o[n + 1] = v.y; }
static void putm_(uint8_t* o, int64_t n, bool g) { o[n] = g ? 1 : 0; }
static void putm_(uint8_t* o, int64_t n, mask2 g) { o[n] = g.x ? 1 : 0; o[n + 1] = g.y ? 1 : 0; }

// One launch from the reference's initial state (X = [1,0,0,0], P = I), as the kernels run it: filter frame in, out.
// IM: 0 no innovation sums, 1 the 4-D ones, 2 the tangent-space ones.  GATE false: the ungated step of the same build.
template <typename F, int ALGO, bool COMP, bool GATE, int IM>
static void gated_t(int64_t N, int64_t T, const float* streams, const double* dt, int dt_per_step, const float* acc_ref,
                    const float* mag_ref, const float* q, const float* r, float gamma, double* traj, uint8_t* gated_out,
                    double* x_out, double* p_out, double* innov_out) {
  const int64_t L = Lanes<F>::n;
  for (int64_t n = 0; n < N; n += L) {
    Vec3<F> ra = {lanes_<F>(acc_ref, n), lanes_<F>(acc_ref, N + n), lanes_<F>(acc_ref, 2 * N + n)};
    Vec3<F> rm = {lanes_<F>(mag_ref, n), lanes_<F>(mag_ref, N + n), lanes_<F>(mag_ref, 2 * N + n)};
    const F rr = lanes_<F>(r, n);
    FilterConst<F> fc = make_filter_const<F>(ra, rm, lanes_<F>(q, n), rr);
    InnovAcc<F> acc = make_innov_acc<F, IM == 2>(F(0), F(0), rr);
    const GateParams<F> gp = make_gate_params<F>(rr, gamma);
    Quat<F> x = {F(1), F(0), F(0), F(0)}, xlo = {F(0), F(0), F(0), F(0)};
    const F ir = F(1) / rr;
    Sym4<F> P = {ir, F(0), F(0), F(0), ir, F(0), F(0), ir, F(0), ir};
    adopt_state(fc, x, xlo);
    enter_filter_frame(fc, x, xlo, P, COMP);
    for (int64_t t = 0; t < T; ++t) {
      const float* s = streams + (size_t)t * 9 * N;
      Vec3<F> w = {lanes_<F>(s, n), lanes_<F>(s, N + n), lanes_<F>(s, 2 * N + n)};
      Vec3<F> a = {lanes_<F>(s, 3 * N + n), lanes_<F>(s, 4 * N + n), lanes_<F>(s, 5 * N + n)};
      Vec3<F> m = {lanes_<F>(s, 6 * N + n), lanes_<F>(s, 7 * N + n), lanes_<F>(s, 8 * N + n)};
      const F h = F((float)(dt_per_step ? dt[t] : dt[0]));
      decltype(F(0) < F(0)) flip, g = decltype(F(0) < F(0))();
      ekf_step<F, ALGO, false, COMP, IM != 0, IM == 2, GATE>(x, xlo, P, fc, w, a, m, StepH<F>(h), flip, false, nullptr,
                                                             IM != 0 ? &acc : nullptr, GATE ? &gp : nullptr, GATE ? &g : nullptr);
      putm_(gated_out + (size_t)t * N, n, g);
      const Quat<F> xr = state_in_reference_frame(fc, x);
      double* row = traj + (size_t)t * N * 4;
      for (int64_t l = 0; l < L; ++l) {
        row[4 * (n + l) + 0] = lane_(xr.w, (int)l); row[4 * (n + l) + 1] = lane_(xr.x, (int)l);
        row[4 * (n + l) + 2] = lane_(xr.y, (int)l); row[4 * (n + l) + 3] = lane_(xr.z, (int)l);
      }
    }
    leave_filter_frame(fc, x, xlo, P, COMP);
    put_<F>(x_out, n, x.w); put_<F>(x_out, N + n, x.x); put_<F>(x_out, 2 * N + n, x.y); put_<F>(x_out, 3 * N + n, x.z);
    const F pv[10] = {P.a00, P.a01, P.a02, P.a03, P.a11, P.a12, P.a13, P.a22, P.a23, P.a33};
    for (int k = 0; k < 10; ++k) put_<F>(p_out, k * N + n, pv[k]);
    put_<F>(innov_out, n, acc.nis);
    put_<F>(innov_out, N + n, acc.logdet);
  }
}

template <typename F, int ALGO, bool COMP>
static void dispatch_(int gate, int im, int64_t N, int64_t T, const float* streams, const double* dt, int dt_per_step,
                      const float* acc_ref, const float* mag_ref, const float* q, const float* r, float gamma, double* traj,
                      uint8_t* gated, double* x, double* p, double* innov) {
#define GO(G, I) gated_t<F, ALGO, COMP, G, I>(N, T, streams, dt, dt_per_step, acc_ref, mag_ref, q, r, gamma, traj, gated, x, p, innov)
  if (gate) { if (im == 0) GO(true, 0); else if (im == 1) GO(true, 1); else GO(true, 2); }
  else { if (im == 0) GO(false, 0); else if (im == 1) GO(false, 1); else GO(false, 2); }
#undef GO
}

extern "C" {

// precision: 0 = float32, 1 = float64, 2 = packed float32 (f32x2); algo: 0 = QR2, 1 = Jacobi (not packed);
// gate: 0 = the ungated step, 1 = the gated one (threshold gamma); innov_model: 0 none, 1 4-D, 2 tangent.
// traj [T][N][4] reference frame, gated [T][N], x [4][N] and p [10][N] (P/r) after the last step, innov [2][N].
int hostsim_gating(int precision, int algo, int comp, int gate, int innov_model, float gamma, int64_t N, int64_t T,
                   const float* streams, const double* dt, int dt_per_step, const float* acc_ref, const float* mag_ref,
                   const float* q, const float* r, double* traj, uint8_t* gated, double* x, double* p, double* innov) {
  if (innov_model < 0 || innov_model > 2) return 1;
#define GO(F, A) if (comp) dispatch_<F, A, true>(gate, innov_model, N, T, streams, dt, dt_per_step, acc_ref, mag_ref, q, r, gamma, traj, gated, x, p, innov); \
                 else dispatch_<F, A, false>(gate, innov_model, N, T, streams, dt, dt_per_step, acc_ref, mag_ref, q, r, gamma, traj, gated, x, p, innov)
  if (precision == 0 && algo == 0) GO(float, WAHBA_QR2);
  else if (precision == 0 && algo == 1) GO(float, WAHBA_JACOBI);
  else if (precision == 1 && algo == 0) GO(double, WAHBA_QR2);
  else if (precision == 1 && algo == 1) GO(double, WAHBA_JACOBI);
  else if (precision == 2 && algo == 0 && N % 2 == 0) GO(f32x2, WAHBA_QR2);
  else return 1;
#undef GO
  return 0;
}

}  // extern "C"
