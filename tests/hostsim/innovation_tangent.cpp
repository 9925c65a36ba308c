// innovation_tangent.cpp -- CPU build of the tangent-space innovation statistic of poseestimationkf_b200/csrc/ekf_math.cuh.
//
// TEST TOOL ONLY (like innovation.cpp beside it, which builds the 4-D statistic): the sums the TAN replay kernels
// accumulate, computed by the same header in float32, float64 and the packed f32x2 lanes, for the `-m "not gpu"` tests.
// Compiled by tests/hostsim/innovation_tangent.py.
#include <cstdint>
#include <cstddef>
#include "../../poseestimationkf_b200/csrc/ekf_math.cuh"

using namespace pkf;

// Tangent-space innovation likelihood sums of a replay (sum_t NIS3_t, sum_t ln det S3_t per filter), accumulated in F
// like the kernels (launch constants from make_innov_acc<F, true>, one launch from the reference's initial state).
// F = f32x2 runs two filters per "thread" as the packed kernel does; N must then be even.
template <typename F> static F lanes_(const float* v, int64_t n) { return (F)v[n]; }
template <> f32x2 lanes_<f32x2>(const float* v, int64_t n) { return f32x2(v[n], v[n + 1]); }
template <typename F> static void put_(double* o, int64_t n, const F& v) { o[n] = v; }
template <> void put_<f32x2>(double* o, int64_t n, const f32x2& v) { o[n] = v.x; o[n + 1] = v.y; }

template <typename F, int ALGO, bool COMP>
static void tangent_t(int64_t N, int64_t T, const float* streams, const double* dt, int dt_per_step, const float* acc_ref,
                      const float* mag_ref, const float* q, const float* r, double* out) {
  const int64_t L = Lanes<F>::n;
  for (int64_t n = 0; n < N; n += L) {
    Vec3<F> ra = {lanes_<F>(acc_ref, n), lanes_<F>(acc_ref, N + n), lanes_<F>(acc_ref, 2 * N + n)};
    Vec3<F> rm = {lanes_<F>(mag_ref, n), lanes_<F>(mag_ref, N + n), lanes_<F>(mag_ref, 2 * N + n)};
    const F rr = lanes_<F>(r, n);
    FilterConst<F> fc = make_filter_const<F>(ra, rm, lanes_<F>(q, n), rr);
    InnovAcc<F> acc = make_innov_acc<F, true>(F(0), F(0), rr);
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
      decltype(F(0) < F(0)) flip;
      ekf_step<F, ALGO, false, COMP, true, true>(x, xlo, P, fc, w, a, m, StepH<F>(h), flip, false, nullptr, &acc);
    }
    put_<F>(out, n, acc.nis);
    put_<F>(out, N + n, acc.logdet);
  }
}

extern "C" {

// precision: 0 = float32, 1 = float64, 2 = packed float32 (f32x2); algo: 0 = QR2, 1 = Jacobi (not packed).
// out [2][N]: sum_t NIS3_t, sum_t ln det S3_t.
int hostsim_innovation_tangent(int precision, int algo, int comp, int64_t N, int64_t T, const float* streams, const double* dt,
                               int dt_per_step, const float* acc_ref, const float* mag_ref, const float* q, const float* r,
                               double* out) {
#define GO(F, A) if (comp) tangent_t<F, A, true>(N, T, streams, dt, dt_per_step, acc_ref, mag_ref, q, r, out); else tangent_t<F, A, false>(N, T, streams, dt, dt_per_step, acc_ref, mag_ref, q, r, out)
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
