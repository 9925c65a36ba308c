// innovation_steps.cpp -- CPU build of the per-step innovation terms of poseestimationkf_b200/csrc/ekf_math.cuh
// (the InnovTerms that ekf_step hands to the innovation-steps kernels).
//
// TEST TOOL ONLY (like gating.cpp beside it): the terms each step adds to the innovation sums, computed by the same
// header in float32, float64 and the packed f32x2 lanes, with the sums the same build accumulates, for the
// `-m "not gpu"` tests.  Compiled by tests/hostsim/innovation_steps.py.
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

// One launch from the reference's initial state (X = [1,0,0,0], P = I), filter frame in and out, as the kernels run it.
// TAN: the tangent-space model.  GATE: the innovation gate at gamma.
template <typename F, int ALGO, bool COMP, bool TAN, bool GATE>
static void steps_t(int64_t N, int64_t T, const float* streams, const double* dt, int dt_per_step, const float* acc_ref,
                    const float* mag_ref, const float* q, const float* r, float gamma, double* terms, uint8_t* gated_out,
                    double* innov_out) {
  const int64_t L = Lanes<F>::n;
  for (int64_t n = 0; n < N; n += L) {
    Vec3<F> ra = {lanes_<F>(acc_ref, n), lanes_<F>(acc_ref, N + n), lanes_<F>(acc_ref, 2 * N + n)};
    Vec3<F> rm = {lanes_<F>(mag_ref, n), lanes_<F>(mag_ref, N + n), lanes_<F>(mag_ref, 2 * N + n)};
    const F rr = lanes_<F>(r, n);
    FilterConst<F> fc = make_filter_const<F>(ra, rm, lanes_<F>(q, n), rr);
    InnovAcc<F> acc = make_innov_acc<F, TAN>(F(0), F(0), rr);
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
      InnovTerms<F> it;
      ekf_step<F, ALGO, false, COMP, true, TAN, GATE>(x, xlo, P, fc, w, a, m, StepH<F>(h), flip, false, nullptr, &acc,
                                                      GATE ? &gp : nullptr, GATE ? &g : nullptr, nullptr, &it);
      putm_(gated_out + (size_t)t * N, n, g);
      put_<F>(terms, (size_t)t * N + n, it.nis);
      put_<F>(terms, (size_t)(T + t) * N + n, it.logdet);
    }
    put_<F>(innov_out, n, acc.nis);
    put_<F>(innov_out, N + n, acc.logdet);
  }
}

template <typename F, int ALGO>
static int dispatch_(int comp, int tan, int gate, int64_t N, int64_t T, const float* streams, const double* dt, int dt_per_step,
                     const float* acc_ref, const float* mag_ref, const float* q, const float* r, float gamma, double* terms,
                     uint8_t* gated, double* innov) {
#define GO(C, M, G) steps_t<F, ALGO, C, M, G>(N, T, streams, dt, dt_per_step, acc_ref, mag_ref, q, r, gamma, terms, gated, innov)
  const int k = (comp ? 4 : 0) | (tan ? 2 : 0) | (gate ? 1 : 0);
  switch (k) {
    case 0: GO(false, false, false); break;
    case 1: GO(false, false, true); break;
    case 2: GO(false, true, false); break;
    case 3: GO(false, true, true); break;
    case 4: GO(true, false, false); break;
    case 5: GO(true, false, true); break;
    case 6: GO(true, true, false); break;
    default: GO(true, true, true); break;
  }
#undef GO
  return 0;
}

extern "C" {

// precision: 0 = float32, 1 = float64, 2 = packed float32 (f32x2, N even); algo: 0 = QR2, 1 = Jacobi (not packed);
// tangent: the model; gate: the gated step at gamma.  terms [2][T][N] (NIS_t, ln det S_t), gated [T][N], innov [2][N]
// (the sums the same build accumulates).
int hostsim_innovation_steps(int precision, int algo, int comp, int tangent, int gate, float gamma, int64_t N, int64_t T,
                             const float* streams, const double* dt, int dt_per_step, const float* acc_ref,
                             const float* mag_ref, const float* q, const float* r, double* terms, uint8_t* gated,
                             double* innov) {
#define GO(F, A) return dispatch_<F, A>(comp, tangent, gate, N, T, streams, dt, dt_per_step, acc_ref, mag_ref, q, r, gamma, terms, gated, innov)
  if (precision == 0 && algo == 0) GO(float, WAHBA_QR2);
  if (precision == 0 && algo == 1) GO(float, WAHBA_JACOBI);
  if (precision == 1 && algo == 0) GO(double, WAHBA_QR2);
  if (precision == 1 && algo == 1) GO(double, WAHBA_JACOBI);
  if (precision == 2 && algo == 0 && N % 2 == 0) GO(f32x2, WAHBA_QR2);
#undef GO
  return 1;
}

}  // extern "C"
