// ekf_math.cuh -- per-filter arithmetic of the quaternion EKF step, register resident.
//
// Everything here is a __host__ __device__ template over the scalar type F so that the *same*
// source is (a) instantiated with F=float inside the sm_100a kernels (replay_kernels.cuh, ops_kernels.cuh) and
// (b) compiled by g++ with F=float / F=double in tests/hostsim (a CPU-only numerics probe used while
// developing without a GPU; it is a test tool, never a product path).
//
// Reference behaviour being reproduced (file:line relative to the reference repository,
// PKF = "Python Kalman Filter"):
//   RK4 of q' = 0.5*Omega(w) q + normalise ........ PKF/ExtendedKalmanFilter.py:25-41
//   A = 0.5*Omega(w), B(q) ......................... PKF/ExtendedKalmanFilter.py:43-56
//   P = A P A^T + B Q B^T, S = P + R, K = P S^-1 ... PKF/ExtendedKalmanFilter.py:58-68
//   Wahba: B = ka r_a b_a^T + km r_m b_m^T, SVD, det fix, R = U M V^T ... PKF/Wahba.py:8-17
//   rotation matrix -> quaternion (3 branch) ....... PKF/Wahba.py:20-47
//   q/-q comparator, X = z + K(y - z), P = P - K P, normalise ... PKF/ExtendedKalmanFilter.py:70-80
//   low-pass y = a x + (1-a) y ..................... PKF/Test.py:27-33 ; C++ twin KalmanFilter.cpp:21-24
//
// Algebraic restructurings (exact in real arithmetic; they change rounding only, see DESIGN.md):
//   * RK4 on a linear constant-coefficient ODE is the degree-4 Taylor polynomial of exp(hA); with
//     A^2 = -(|w|^2/4) I it collapses to  z = c0 x + c1 (A x).
//   * With Q = q I3:  B Q B^T = (q/4)(|x|^2 I - x x^T).
//   * With R = r I4:  K = P S^-1 = I - r S^-1 (symmetric) and  P - K P = r K  (see kalman_gain).
//   * P is kept as its upper triangle (10 values).
//   * rank(B_wahba) = 2 always (two observations), so the SVD is taken on the 2x2 core of a QR
//     factorisation of both vector pairs (see wahba_qr2) -- this is also what makes fp32 safe when
//     the reference's weights ka=|a_z|, km=1-|a_z| drive B towards rank 1.  The fused step goes one step
//     further and evaluates the two-observation optimum directly as a quaternion (wahba_quat2_local).
//   * A = 0.5*Omega(w) is a right quaternion multiplication: in the (1 + 3x3) split of symmetric 4x4 matrices
//     A P A^T touches the 3x3 block only (propagate_cov).
//   * The recursion is equivariant under a fixed left rotation of the state, so the fused step runs in the
//     coordinates of the reference frame built from (acc_0, mag_0) ("filter frame").
#pragma once

#include <math.h>

#if defined(__CUDACC__)
#define PKF_HD __host__ __device__ __forceinline__
#define PKF_HD_RARE __host__ __device__ __noinline__ inline   // rare paths: kept out of line so they cost the hot code no registers
#else
#define PKF_HD inline
#define PKF_HD_RARE inline
#endif

namespace pkf {

// ------------------------------------------------------------------------------------------
// scalar primitives
// ------------------------------------------------------------------------------------------
template <typename F> PKF_HD F fma_(F a, F b, F c) { return a * b + c; }
template <typename F> PKF_HD F abs_(F a) { return a < F(0) ? -a : a; }
template <typename F> PKF_HD F sqrt_(F a) { return (F)sqrt((double)a); }
template <typename F> PKF_HD F rcp_(F a) { return F(1) / a; }
template <typename F> PKF_HD F rsqrt_(F a) { return F(1) / (F)sqrt((double)a); }

#if defined(__CUDA_ARCH__)
template <> __device__ __forceinline__ float fma_<float>(float a, float b, float c) { return __fmaf_rn(a, b, c); }
template <> __device__ __forceinline__ float abs_<float>(float a) { return fabsf(a); }
template <> __device__ __forceinline__ float sqrt_<float>(float a) { return sqrtf(a); }
// one MUFU each; ~1 ulp.  (IEEE division/rsqrt sequences cost 6-10 issue slots; the parity budget
// of 1e-5 rad leaves two orders of magnitude of room for a 1e-7 relative error.)
template <> __device__ __forceinline__ float rcp_<float>(float a) {
  float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a)); return r;
}
template <> __device__ __forceinline__ float rsqrt_<float>(float a) {
  float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a)); return r;
}
#else
template <> inline float fma_<float>(float a, float b, float c) { return fmaf(a, b, c); }
template <> inline float sqrt_<float>(float a) { return sqrtf(a); }
template <> inline float rsqrt_<float>(float a) { return 1.0f / sqrtf(a); }
template <> inline double fma_<double>(double a, double b, double c) { return fma(a, b, c); }
template <> inline double sqrt_<double>(double a) { return sqrt(a); }
template <> inline double rsqrt_<double>(double a) { return 1.0 / sqrt(a); }
#endif
// natural logarithms of the innovation statistic (full precision: see log_pivots)
template <typename F> PKF_HD F log_(F a) { return (F)log((double)a); }
template <typename F> PKF_HD F log1p_(F a) { return (F)log1p((double)a); }
#if defined(__CUDA_ARCH__)
template <> __device__ __forceinline__ float log_<float>(float a) { return logf(a); }
template <> __device__ __forceinline__ float log1p_<float>(float a) { return log1pf(a); }
#else
template <> inline float log_<float>(float a) { return logf(a); }
template <> inline float log1p_<float>(float a) { return log1pf(a); }
template <> inline double log_<double>(double a) { return log(a); }
template <> inline double log1p_<double>(double a) { return log1p(a); }
#endif

template <typename F> PKF_HD F sel_(bool c, F a, F b) { return c ? a : b; }
PKF_HD bool any_(bool m) { return m; }
// Sign-bit helpers.  On sm_100 FSEL issues to the FP32 (FMA) pipe -- the pipe that bounds the fused step -- while
// the integer ALU is nearly idle, so the selections and conditional negations of the hot path are written on the
// bit patterns (LOP3 / SHF):
//   flipsign_(v, s)      v with its sign flipped when the sign bit of s is set
//   selsign_(s, a, b)    a when the sign bit of s is set, else b   (lop3 0xCA through inline PTX: the
//                        compiler folds a C-level bit blend back into a float select)
//   one_with_sign_(s)    +1 or -1 carrying the sign bit of s
//   signbit_(s)          that bit as a mask
#ifndef PKF_SEL_MODE
#define PKF_SEL_MODE 0
#endif
// PKF_FUSE: the plain (non-precise) step accumulates z = x + inc and X = z + K e through their FMAs and factors
// S = P + I with its "+ 1" folded into a constant (see rk4_predict_fused, kalman_gain_from_s): 12 FP32 operations fewer.
#ifndef PKF_FUSE
#define PKF_FUSE 2
#endif
#if defined(__CUDA_ARCH__)
__device__ __forceinline__ float flipsign_(float v, float s) {
#if PKF_SEL_MODE == 0
  return __float_as_int(s) < 0 ? -v : v;
#elif PKF_SEL_MODE == 2
  int r;      // v ^ (s & 0x80000000): one LOP3 with two register operands (integer pipe)
  // (a, b, c) = (v, s, mask); LUT = a ^ (b & c) = 0xF0 ^ (0xCC & 0xAA) = 0x78
  asm("lop3.b32 %0, %1, %2, 0x80000000, 0x78;" : "=r"(r) : "r"(__float_as_int(v)), "r"(__float_as_int(s)));
  return __int_as_float(r);
#else
  return __uint_as_float(__float_as_uint(v) ^ (__float_as_uint(s) & 0x80000000u));
#endif
}
__device__ __forceinline__ float selsign_(float s, float a, float b) {
#if PKF_SEL_MODE == 1
  int r;
  asm("lop3.b32 %0, %1, %2, %3, 0xCA;" : "=r"(r) : "r"(__float_as_int(s) >> 31), "r"(__float_as_int(a)), "r"(__float_as_int(b)));
  return __int_as_float(r);
#else
  return __float_as_int(s) < 0 ? a : b;
#endif
}
__device__ __forceinline__ bool signbit_(float s) { return (__float_as_uint(s) >> 31) != 0u; }
// |v| with the sign bit of s: one LOP3 ((v & 0x7fffffff) | (s & 0x80000000)) on the integer pipe
__device__ __forceinline__ float copysign_(float v, float s) {
  int r;
  // operands (a, b, c) = (s, v, mask); LUT = (c & a) | (~c & b) = (0xAA & 0xF0) | (0x55 & 0xCC) = 0xE4
  asm("lop3.b32 %0, %1, %2, 0x80000000, 0xE4;" : "=r"(r) : "r"(__float_as_int(s)), "r"(__float_as_int(v)));
  return __int_as_float(r);
}
__device__ __forceinline__ float one_with_sign_(float s) {
  return __uint_as_float((__float_as_uint(s) & 0x80000000u) | 0x3f800000u);
}
__device__ __forceinline__ double flipsign_(double v, double s) { return __double2hiint(s) < 0 ? -v : v; }   // rare exact path only
__device__ __forceinline__ double selsign_(double s, double a, double b) { return __double2hiint(s) < 0 ? a : b; }
__device__ __forceinline__ bool signbit_(double s) { return __double2hiint(s) < 0; }
__device__ __forceinline__ double one_with_sign_(double s) { return __double2hiint(s) < 0 ? -1.0 : 1.0; }
__device__ __forceinline__ double copysign_(double v, double s) { return copysign(v, s); }
#else
inline float flipsign_(float v, float s) { return __builtin_signbit(s) ? -v : v; }
inline float selsign_(float s, float a, float b) { return __builtin_signbit(s) ? a : b; }
inline bool signbit_(float s) { return __builtin_signbit(s); }
inline float one_with_sign_(float s) { return __builtin_signbit(s) ? -1.0f : 1.0f; }
inline float copysign_(float v, float s) { return __builtin_copysignf(v, s); }
inline double copysign_(double v, double s) { return __builtin_copysign(v, s); }
inline double flipsign_(double v, double s) { return __builtin_signbit(s) ? -v : v; }
inline double selsign_(double s, double a, double b) { return __builtin_signbit(s) ? a : b; }
inline bool signbit_(double s) { return __builtin_signbit(s); }
inline double one_with_sign_(double s) { return __builtin_signbit(s) ? -1.0 : 1.0; }
#endif

// ------------------------------------------------------------------------------------------
// f32x2: TWO filters per thread in the lanes of a 64-bit register pair.  On sm_100 every operator maps
// onto one packed instruction (FFMA2 / FMUL2 / FADD2, with negate modifiers, immediates and scalar
// broadcast operands), so the hot step issues half as many FP32 instructions per filter; the FP32
// pipe is busy for the same number of cycles, but the issue slots it frees absorb the non-FP32
// instructions (loads, barriers, MUFU) that otherwise compete with it.  On the host the lanes are
// plain floats (tests/hostsim).
// ------------------------------------------------------------------------------------------
struct mask2 { bool x, y; };
PKF_HD bool any_(mask2 m) { return m.x || m.y; }
PKF_HD mask2 operator&&(mask2 a, mask2 b) { return mask2{a.x && b.x, a.y && b.y}; }
PKF_HD mask2 operator!(mask2 a) { return mask2{!a.x, !a.y}; }

struct f32x2 {
  float x, y;
  PKF_HD f32x2() {}
  PKF_HD f32x2(float a) : x(a), y(a) {}
  PKF_HD f32x2(double a) : x((float)a), y((float)a) {}
  PKF_HD f32x2(int a) : x((float)a), y((float)a) {}
  PKF_HD f32x2(float a, float b) : x(a), y(b) {}
};
#if defined(__CUDA_ARCH__)
__device__ __forceinline__ float2 f2_(const f32x2& a) { return make_float2(a.x, a.y); }
__device__ __forceinline__ f32x2 operator+(const f32x2& a, const f32x2& b) { float2 r = __fadd2_rn(f2_(a), f2_(b)); return f32x2(r.x, r.y); }
__device__ __forceinline__ f32x2 operator-(const f32x2& a, const f32x2& b) { float2 r = __fadd2_rn(f2_(a), make_float2(-b.x, -b.y)); return f32x2(r.x, r.y); }
__device__ __forceinline__ f32x2 operator*(const f32x2& a, const f32x2& b) { float2 r = __fmul2_rn(f2_(a), f2_(b)); return f32x2(r.x, r.y); }
#else
inline f32x2 operator+(const f32x2& a, const f32x2& b) { return f32x2(a.x + b.x, a.y + b.y); }
inline f32x2 operator-(const f32x2& a, const f32x2& b) { return f32x2(a.x - b.x, a.y - b.y); }
inline f32x2 operator*(const f32x2& a, const f32x2& b) { return f32x2(a.x * b.x, a.y * b.y); }
#endif
PKF_HD f32x2 operator-(const f32x2& a) { return f32x2(-a.x, -a.y); }
PKF_HD f32x2 operator/(const f32x2& a, const f32x2& b) { return f32x2(a.x / b.x, a.y / b.y); }   // set-up code only
PKF_HD f32x2& operator*=(f32x2& a, const f32x2& b) { a = a * b; return a; }
PKF_HD mask2 operator<(const f32x2& a, const f32x2& b) { return mask2{a.x < b.x, a.y < b.y}; }
PKF_HD mask2 operator>(const f32x2& a, const f32x2& b) { return mask2{a.x > b.x, a.y > b.y}; }
PKF_HD mask2 operator==(const f32x2& a, const f32x2& b) { return mask2{a.x == b.x, a.y == b.y}; }
PKF_HD f32x2 sel_(mask2 c, const f32x2& a, const f32x2& b) { return f32x2(c.x ? a.x : b.x, c.y ? a.y : b.y); }
PKF_HD f32x2 selsign_(const f32x2& s, const f32x2& a, const f32x2& b) { return f32x2(selsign_(s.x, a.x, b.x), selsign_(s.y, a.y, b.y)); }
PKF_HD f32x2 flipsign_(const f32x2& v, const f32x2& s) { return f32x2(flipsign_(v.x, s.x), flipsign_(v.y, s.y)); }
PKF_HD mask2 signbit_(const f32x2& s) { return mask2{signbit_(s.x), signbit_(s.y)}; }
PKF_HD f32x2 one_with_sign_(const f32x2& s) { return f32x2(one_with_sign_(s.x), one_with_sign_(s.y)); }
PKF_HD f32x2 copysign_(const f32x2& v, const f32x2& s) { return f32x2(copysign_(v.x, s.x), copysign_(v.y, s.y)); }
template <> PKF_HD f32x2 fma_<f32x2>(f32x2 a, f32x2 b, f32x2 c) {
#if defined(__CUDA_ARCH__)
  float2 r = __ffma2_rn(f2_(a), f2_(b), f2_(c));
  return f32x2(r.x, r.y);
#else
  return f32x2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y));
#endif
}
template <> PKF_HD f32x2 abs_<f32x2>(f32x2 a) { return f32x2(abs_<float>(a.x), abs_<float>(a.y)); }
template <> PKF_HD f32x2 rcp_<f32x2>(f32x2 a) { return f32x2(rcp_<float>(a.x), rcp_<float>(a.y)); }
template <> PKF_HD f32x2 rsqrt_<f32x2>(f32x2 a) { return f32x2(rsqrt_<float>(a.x), rsqrt_<float>(a.y)); }
template <> PKF_HD f32x2 sqrt_<f32x2>(f32x2 a) { return f32x2(sqrt_<float>(a.x), sqrt_<float>(a.y)); }
template <> PKF_HD f32x2 log_<f32x2>(f32x2 a) { return f32x2(log_<float>(a.x), log_<float>(a.y)); }
template <> PKF_HD f32x2 log1p_<f32x2>(f32x2 a) { return f32x2(log1p_<float>(a.x), log1p_<float>(a.y)); }

// ------------------------------------------------------------------------------------------
// types
// ------------------------------------------------------------------------------------------
template <typename F> struct Vec3 { F x, y, z; };
template <typename F> struct Quat { F w, x, y, z; };

// symmetric 4x4, upper triangle, row-major order 00 01 02 03 11 12 13 22 23 33
template <typename F> struct Sym4 { F a00, a01, a02, a03, a11, a12, a13, a22, a23, a33; };

template <typename F> struct Mat3 { F m[3][3]; };
template <typename F> struct Mat4 { F m[4][4]; };

// Per-filter constants of the Wahba stage derived from the reference vectors (acc_0, mag_0):
// the right-handed frame E = [e1 e2 e3] from Gram-Schmidt on (r_a, r_m) and the 2x2 triangular
// factor  [r_a r_m] = [e1 e2] [[s11 s12],[0 s22]].
template <typename F> struct RefFrame {
  Vec3<F> e1, e2, e3;
  F s11, s12, s22;
  F r12, r22;       // s12/s11, s22/s11 (used by the closed-form measurement, whose scale is free)
};

template <typename F> PKF_HD F dot3(const Vec3<F>& a, const Vec3<F>& b) {
  return fma_(a.z, b.z, fma_(a.y, b.y, a.x * b.x));
}
template <typename F> PKF_HD Vec3<F> cross3(const Vec3<F>& a, const Vec3<F>& b) {
  Vec3<F> c;
  c.x = fma_(a.y, b.z, -(a.z * b.y));
  c.y = fma_(a.z, b.x, -(a.x * b.z));
  c.z = fma_(a.x, b.y, -(a.y * b.x));
  return c;
}
template <typename F> PKF_HD F dot4(const Quat<F>& a, const Quat<F>& b) {
  return fma_(a.z, b.z, fma_(a.y, b.y, fma_(a.x, b.x, a.w * b.w)));
}

// QR (Gram-Schmidt) of the 3x2 matrix [a m]:  [a m] = [f1 f2] [[t11 t12],[0 t22]], f3 = f1 x f2.
template <typename F> PKF_HD RefFrame<F> frame_from_pair(const Vec3<F>& a, const Vec3<F>& m) {
  RefFrame<F> fr;
  F na2 = dot3(a, a);
  F ia = rsqrt_(na2);
  fr.e1.x = a.x * ia; fr.e1.y = a.y * ia; fr.e1.z = a.z * ia;
  fr.s11 = na2 * ia;
  fr.s12 = dot3(m, fr.e1);
  Vec3<F> mp;
  mp.x = fma_(-fr.s12, fr.e1.x, m.x);
  mp.y = fma_(-fr.s12, fr.e1.y, m.y);
  mp.z = fma_(-fr.s12, fr.e1.z, m.z);
  F np2 = dot3(mp, mp);
  F ip = rsqrt_(np2);
  fr.e2.x = mp.x * ip; fr.e2.y = mp.y * ip; fr.e2.z = mp.z * ip;
  fr.s22 = np2 * ip;
  fr.e3 = cross3(fr.e1, fr.e2);
  fr.r12 = fr.s12 * ia; fr.r22 = fr.s22 * ia;      // ia = 1/s11
  return fr;
}

// ------------------------------------------------------------------------------------------
// low-pass  y <- alpha x + (1-alpha) y          (PKF/Test.py:27-33, SRV/KalmanFilter.cpp:21-24)
// ------------------------------------------------------------------------------------------
template <typename F> PKF_HD void lowpass(Vec3<F>& y, const Vec3<F>& x, F alpha, F one_minus_alpha) {
  y.x = fma_(alpha, x.x, one_minus_alpha * y.x);
  y.y = fma_(alpha, x.y, one_minus_alpha * y.y);
  y.z = fma_(alpha, x.z, one_minus_alpha * y.z);
}

// ------------------------------------------------------------------------------------------
// RK4 step of q' = 0.5*Omega(w) q over h seconds, then normalise.
//   (PKF/ExtendedKalmanFilter.py:25-41; hw = 0.5*w is passed in because the caller shares it with
//    the covariance propagation.)
// k1..k4 of the reference expand to  z = (1 - a2/2 + a2^2/24) q + h (1 - a2/6) (A q),
// a2 = h^2 |hw|^2, because A^2 = -|hw|^2 I.
// ------------------------------------------------------------------------------------------
template <typename F> PKF_HD Quat<F> rk4_step(const Quat<F>& q, const Vec3<F>& hw, F h) {
  Quat<F> u;   // u = A q
  u.w = fma_(-hw.z, q.z, fma_(-hw.y, q.y, -(hw.x * q.x)));
  u.x = fma_(-hw.y, q.z, fma_(hw.z, q.y, hw.x * q.w));
  u.y = fma_(hw.x, q.z, fma_(-hw.z, q.x, hw.y * q.w));
  u.z = fma_(-hw.x, q.y, fma_(hw.y, q.x, hw.z * q.w));
  F a2 = (h * h) * dot3(hw, hw);
  F c0 = fma_(a2, fma_(a2, F(1.0 / 24.0), F(-0.5)), F(1));
  F c1 = h * fma_(a2, F(-1.0 / 6.0), F(1));
  Quat<F> z;
  z.w = fma_(c1, u.w, c0 * q.w);
  z.x = fma_(c1, u.x, c0 * q.x);
  z.y = fma_(c1, u.y, c0 * q.y);
  z.z = fma_(c1, u.z, c0 * q.z);
  F r = rsqrt_(dot4(z, z));
  z.w *= r; z.x *= r; z.y *= r; z.z *= r;
  return z;
}

// Fused-step form of the same RK4 step: returns only the INCREMENT  (c0 - 1) x + c1 (A x), so that
// z = x + inc, WITHOUT the normalisation.  RK4 preserves the norm to O(a^6) (~1e-15 at 100 Hz), so
// dividing by |z| only re-rounds the state; the caller renormalises lazily (see ekf_step) and, in
// the compensated variant, folds the increment into a two-float state.
template <typename F> PKF_HD Quat<F> rk4_increment(const Quat<F>& q, const Vec3<F>& hw, F h) {
  Quat<F> u;   // u = A q
  u.w = fma_(-hw.z, q.z, fma_(-hw.y, q.y, -(hw.x * q.x)));
  u.x = fma_(-hw.y, q.z, fma_(hw.z, q.y, hw.x * q.w));
  u.y = fma_(hw.x, q.z, fma_(-hw.z, q.x, hw.y * q.w));
  u.z = fma_(-hw.x, q.y, fma_(hw.y, q.x, hw.z * q.w));
  F a2 = (h * h) * dot3(hw, hw);
  F cm = a2 * fma_(a2, F(1.0 / 24.0), F(-0.5));            // c0 - 1
  F c1 = h * fma_(a2, F(-1.0 / 6.0), F(1));
  Quat<F> inc;
  inc.w = fma_(c1, u.w, cm * q.w);
  inc.x = fma_(c1, u.x, cm * q.x);
  inc.y = fma_(c1, u.y, cm * q.y);
  inc.z = fma_(c1, u.z, cm * q.z);
  return inc;
}

// The time step of one sample with the two products of it that the RK4 polynomial needs.  They are launch constants
// when dt is (the usual case), so the kernels form them once, outside the time loop, instead of twice per step.
template <typename F> struct StepH {
  F h, hh, mh6;       // h, h^2, -h/6
  PKF_HD StepH() {}
  PKF_HD StepH(F h_) : h(h_), hh(h_ * h_), mh6(h_ * F(-1.0 / 6.0)) {}
  PKF_HD StepH(F h_, F hh_, F mh6_) : h(h_), hh(hh_), mh6(mh6_) {}
};

// Plain-variant form: the predicted state z = x + (c0 - 1) x + c1 (A x) accumulated by FMAs onto x (8 operations
// instead of 4 MUL + 4 FMA + 4 ADD); the state is rounded twice per component instead of once (~1 ulp per step,
// contracted by the filter's own gain; the precise variant keeps the increment apart, see ekf_update).
template <typename F> PKF_HD Quat<F> rk4_predict_fused(const Quat<F>& q, const Vec3<F>& hw, const StepH<F>& st) {
  Quat<F> u;   // u = A q
  u.w = fma_(-hw.z, q.z, fma_(-hw.y, q.y, -(hw.x * q.x)));
  u.x = fma_(-hw.y, q.z, fma_(hw.z, q.y, hw.x * q.w));
  u.y = fma_(hw.x, q.z, fma_(-hw.z, q.x, hw.y * q.w));
  u.z = fma_(-hw.x, q.y, fma_(hw.y, q.x, hw.z * q.w));
  F a2 = st.hh * dot3(hw, hw);
  F cm = a2 * fma_(a2, F(1.0 / 24.0), F(-0.5));            // c0 - 1
  F c1 = fma_(a2, st.mh6, st.h);                            // h (1 - a2/6)
  Quat<F> z;
  z.w = fma_(cm, q.w, fma_(c1, u.w, q.w));
  z.x = fma_(cm, q.x, fma_(c1, u.x, q.x));
  z.y = fma_(cm, q.y, fma_(c1, u.y, q.y));
  z.z = fma_(cm, q.z, fma_(c1, u.z, q.z));
  return z;
}

// Knuth two-sum: hi + lo == a + b exactly (no magnitude ordering assumed).
template <typename F> PKF_HD void two_sum(F a, F b, F& hi, F& lo) {
  F s = a + b;
  F bb = s - a;
  lo = (a - (s - bb)) + (b - bb);
  hi = s;
}

// ------------------------------------------------------------------------------------------
// Covariance propagation  P <- A P A^T + B(x) (q I3) B(x)^T,  A = 0.5*Omega(w)  (hw = 0.5 w),
// x = state BEFORE the RK4 step.        (PKF/ExtendedKalmanFilter.py:59-61)
//   B B^T = 0.25 (|x|^2 I - x x^T)  =>  second term = s (I - x^ x^T) with x^ = x/|x| and s = (q/4)|x|^2: the fused
//   step keeps its state normalised and passes s = q/4, except on the first step of a launch that was handed a
//   non-unit state (adopt_state); qq is unused when the noise is added here.
//
// A is the matrix of a RIGHT quaternion multiplication by the pure quaternion (0, hw).  Symmetric 4x4
// matrices split as  P = alpha I + sum_ij T_ij L_i R_j  (L_i / R_j: left / right multiplication by the
// imaginary units; each L_i R_j is a symmetric signed permutation), and a right multiplication acts on
// the 3x3 coefficient matrix T alone:
//     A P A^T  <->  alpha' = |hw|^2 alpha,   T' = 2 (T hw) hw^T - |hw|^2 T
// (|hw|^2 times a half-turn about hw).  With D_i = 4 T_ii and the pair sums/differences of the
// off-diagonal entries (14 additions), U = 2 T hw (12 operations), the result follows entry by entry:
//     diagonal:      alpha' -/+ T'_00 -/+ T'_11 -/+ T'_22,   T'_ii = U_i hw_i - (|hw|^2/4) D_i
//     off-diagonal:  e.g. P'_03 = Y U_0 - X U_1 - |hw|^2 P_03   (the pair sums collapse back to P_03)
// 74 operations including the process noise, against 88 for the two sparse products (A P) A^T.
// ------------------------------------------------------------------------------------------
template <typename F, bool NOISE = true>
PKF_HD Sym4<F> propagate_cov(const Sym4<F>& P, const Vec3<F>& hw, const Quat<F>& x, F qq, F s, F sd) {
  const F X = hw.x, Y = hw.y, Z = hw.z;
  const F p00 = P.a00, p01 = P.a01, p02 = P.a02, p03 = P.a03, p11 = P.a11, p12 = P.a12, p13 = P.a13,
          p22 = P.a22, p23 = P.a23, p33 = P.a33;
  // 4 alpha, 4 T_ii and twice the off-diagonal T_ij (E_ij = 2 T_ij, F_ij = -2 T_ij)
  const F s1 = p00 + p11, s2 = p22 + p33, d1 = p11 - p00, d2 = p33 - p22;
  const F A4 = s1 + s2, D0 = s2 - s1, D1 = d1 + d2, D2 = d1 - d2;
  const F E01 = p03 - p12, F10 = p03 + p12;
  const F F02 = p02 + p13, E20 = p02 - p13;
  const F E12 = p01 - p23, F21 = p01 + p23;
  // U = 2 T hw
  const F qX = F(0.5) * X, qY = F(0.5) * Y, qZ = F(0.5) * Z;
  const F U0 = fma_(-F02, Z, fma_(E01, Y, D0 * qX));
  const F U1 = fma_(E12, Z, fma_(-F10, X, D1 * qY));
  const F U2 = fma_(-F21, Y, fma_(E20, X, D2 * qZ));
  const F w2 = dot3(hw, hw);
  const F c4 = F(0.25) * w2;
  const F T00 = fma_(U0, X, -(c4 * D0)), T11 = fma_(U1, Y, -(c4 * D1)), T22 = fma_(U2, Z, -(c4 * D2));
  const F t1 = T11 + T22, t2 = T22 - T11;
  Sym4<F> N;
  if constexpr (NOISE) {
    const F al = fma_(c4, A4, sd);                     // alpha' + qq |x|^2; sd = s, or s + 1 when the caller wants S = P + I
    const F am = al - T00, ap = al + T00;
    const F yw = s * x.w, yx = s * x.x, yy = s * x.y, yz = s * x.z;     // |x| = 1 inside a launch (adopt_state)
    N.a00 = fma_(-yw, x.w, am - t1);
    N.a11 = fma_(-yx, x.x, am + t1);
    N.a22 = fma_(-yy, x.y, ap + t2);
    N.a33 = fma_(-yz, x.z, ap - t2);
    N.a01 = fma_(Z, U1, fma_(-Y, U2, fma_(-w2, p01, -(yw * x.x))));
    N.a02 = fma_(X, U2, fma_(-Z, U0, fma_(-w2, p02, -(yw * x.y))));
    N.a03 = fma_(Y, U0, fma_(-X, U1, fma_(-w2, p03, -(yw * x.z))));
    N.a12 = fma_(-Y, U0, fma_(-X, U1, fma_(-w2, p12, -(yx * x.y))));
    N.a13 = fma_(-Z, U0, fma_(-X, U2, fma_(-w2, p13, -(yx * x.z))));
    N.a23 = fma_(-Z, U1, fma_(-Y, U2, fma_(-w2, p23, -(yy * x.z))));
  } else {
    // A P A^T alone (the caller handles the process noise separately, see kalman_gain_sm)
    // (explicit fma_: a bare product feeding a sum is what a compiler may or may not contract, and the scalar and
    //  packed builds must round identically)
    const F am = fma_(c4, A4, -T00), ap = fma_(c4, A4, T00);
    N.a00 = am - t1; N.a11 = am + t1; N.a22 = ap + t2; N.a33 = ap - t2;
    N.a01 = fma_(Z, U1, fma_(-Y, U2, -(w2 * p01)));
    N.a02 = fma_(X, U2, fma_(-Z, U0, -(w2 * p02)));
    N.a03 = fma_(Y, U0, fma_(-X, U1, -(w2 * p03)));
    N.a12 = fma_(-Y, U0, fma_(-X, U1, -(w2 * p12)));
    N.a13 = fma_(-Z, U0, fma_(-X, U2, -(w2 * p13)));
    N.a23 = fma_(-Z, U1, fma_(-Y, U2, -(w2 * p23)));
  }
  return N;
}

template <typename F, bool NOISE = true>
PKF_HD Sym4<F> propagate_cov(const Sym4<F>& P, const Vec3<F>& hw, const Quat<F>& x, F qq, F s) {
  return propagate_cov<F, NOISE>(P, hw, x, qq, s, s);
}

// ------------------------------------------------------------------------------------------
// Kalman gain for R = r I:  K = P S^-1 = I - r S^-1,  S = P + r I  (symmetric positive definite).
// (replaces np.linalg.inv + matmul, PKF/ExtendedKalmanFilter.py:63-66.)
//
// S = L D L^T with the pivots kept SPLIT as d_k = r + delta_k (delta_k is the pivot of P's own
// elimination; it is never added to r and subtracted again).  With W = L^-1 = I + N (N strictly
// lower), rho_k = r/d_k and kappa_k = delta_k/d_k = 1 - rho_k:
// (The fused step keeps the covariance in units of r -- see ekf_step -- so r = 1 here.)
//     K = I - W^T diag(rho) W   =>   K_ii = kappa_i - sum_{k>i} n_ki rho_k n_ki
//                                    K_ij =        - (rho_j n_ji + sum_{k>j} n_ki rho_k n_kj)   (i<j)
// Forming the diagonal from kappa (a quotient) instead of 1 - rho (a difference) is what keeps the
// gain accurate to ~1e-7 relative when r >> P (K ~ P/r would otherwise cancel against I), i.e. for
// every (Q,R) tuning of the 1e-3..1e3 sweep (tests/test_gpu_replay.py::test_qr_sweep...).
// ------------------------------------------------------------------------------------------
template <typename F> struct Ldl4 {          // S = P + I = L D L^T;  N = L^-1 - I;  i_k = 1/d_k;  e_k = d_k - 1
  F n10, n20, n21, n30, n31, n32, i0, i1, i2, i3, e0, e1, e2, e3;
};

// ------------------------------------------------------------------------------------------
// Innovation likelihood (prediction-error decomposition of the filter's own Gaussian model):
//     l(Q,R) = 1/2 sum_t [ e_t^T S_t^-1 e_t + ln det S_t + 4 ln 2 pi ],   S = P^- + R,  e = sg y/|y| - z
// (S and e of PKF/ExtendedKalmanFilter.py:63,76).  The step carries S~ = S/r = P~ + I, so
//     NIS = e^T S^-1 e = (1/r) e^T S~^-1 e,     ln det S = 4 ln r + ln det S~.
// The gain stage hands over the factors it has already formed (InnovFactors); the step feeds the innovation e it
// forms anyway.  Both terms are invariant under the filter-frame rotation (e and S are rotated by the orthogonal
// L(p)), so no conversion back to the reference frame is needed.
//   plain   (kalman_gain_from_s): S~ = L D L^T;  e^T S~^-1 e = sum_k i_k t_k^2, t = (I + N) e;  ln det S~ = sum_k ln d_k
//   precise (kalman_gain_sm):     S~ = H - g x x^T;  Sherman-Morrison and the matrix-determinant lemma give
//           e^T S~^-1 e = sum_k i_k t_k^2 (H's factors) + beta (w.e)^2,   ln det S~ = sum_k ln d_k(H) + ln(num / |x|^2)
// (S~^-1 = I - K would cancel as K -> I: the factors are used instead.)
//
// TAN (tangent-space likelihood): the same model restricted to the 3-D tangent space of the prediction u = z/|z| --
// e_3 = E^T e, S_3 = E^T S E for any orthonormal basis E of u-perp, and
//     l_3(Q,R) = 1/2 sum_t [ e_3^T S_3^-1 e_3 + ln det S_3 + 3 ln 2 pi ].
// The 4-D model also scores the direction of u, where a unit-quaternion innovation has almost no component
// (e.u ~ -|e|^2/2) and P^- almost no variance, which drives its R axis towards zero.  No basis is formed: with
// c = z^T S~^-1 z, b = z^T S~^-1 e, s = e^T S~^-1 e the Schur complement of u gives
//     NIS_3 = (s - b^2/c) / r,     ln det S_3 = 3 ln r + ln det S~ + ln(c/|z|^2),   c/|z|^2 = 1 - z^T K z / |z|^2,
// with c and b from the same factors as s (v = (I + N) z; precise: + beta (w.z)^2, + beta (w.z)(w.e)).
// ------------------------------------------------------------------------------------------
template <typename F> struct InnovFactors {
  F n10, n20, n21, n30, n31, n32;   // N = L^-1 - I of S~ (plain) or of H (precise)
  F i0, i1, i2, i3;                 // 1/d_k
  F w0, w1, w2, w3, beta;           // precise only: w = H^-1 x, beta = g|x|^2 / x^T(I+M)w
  F logdet;                         // ln det S~
};
// Running sums of one filter (true units) and the launch constants that fold 1/r and dof ln r (4, TAN: 3) in per step:
// the sums are never rescaled, so a chunked replay accumulates exactly what the unchunked one does.
template <typename F> struct InnovAcc {
  F nis, logdet;
  F inv_r, log_rd;
};
// The terms one step adds (true units): NIS_t and ln det S_t (TAN: NIS3_t and ln det S3_t).  ln det S_t is the addend of
// acc.logdet exactly; NIS_t is the product that acc.nis's fused multiply-add adds before its one rounding, here rounded
// on its own.  Written only when the caller asks for them (per-step innovation output).
template <typename F> struct InnovTerms {
  F nis, logdet;
};
// 3 ln r, rounded once per lane: the packed lanes form it with scalar multiplications, which the compiler does not fuse
// into the per-step addition (a packed product by 3 would be, and that fused sum differs from the scalar kernels' in the
// last bit; 4 ln r is exact either way)
template <typename F> PKF_HD F log_r3_(F r) { return F(3) * log_(r); }
template <> PKF_HD f32x2 log_r3_<f32x2>(f32x2 r) { return f32x2(log_r3_<float>(r.x), log_r3_<float>(r.y)); }
template <typename F, bool TAN = false> PKF_HD InnovAcc<F> make_innov_acc(F nis, F logdet, F r) {
  InnovAcc<F> a;
  a.nis = nis; a.logdet = logdet;
  a.inv_r = F(1) / r;
  if constexpr (TAN) a.log_rd = log_r3_(r);
  else a.log_rd = F(4) * log_(r);
  return a;
}
// sum_k ln(1 + x_k) from the pivot excesses x_k = d_k - 1 >= 0: the excess of the product is formed first and its
// log1p taken, so that pivots near 1 (R >> Q, where ln det S~ is small) keep their relative accuracy.
template <typename F> PKF_HD F log_pivots(F x0, F x1, F x2, F x3) {
  const F a = fma_(x0, x1, x0 + x1), b = fma_(x2, x3, x2 + x3);
  return log1p_(fma_(a, b, a + b));
}
// K = I - S~^-1 (the step's gain) and z are read by TAN only.  step: the step's own terms (see InnovTerms), or null.
template <typename F, bool COMP, bool TAN = false>
PKF_HD void innov_accumulate(InnovAcc<F>& acc, const InnovFactors<F>& f, const Sym4<F>& K, const Quat<F>& z,
                             F e0, F e1, F e2, F e3, InnovTerms<F>* step = nullptr) {
  const F t1 = fma_(f.n10, e0, e1);
  const F t2 = fma_(f.n21, e1, fma_(f.n20, e0, e2));
  const F t3 = fma_(f.n32, e2, fma_(f.n31, e1, fma_(f.n30, e0, e3)));
  const F u0 = f.i0 * e0, u1 = f.i1 * t1, u2 = f.i2 * t2, u3 = f.i3 * t3;
  F s = fma_(u3, t3, fma_(u2, t2, fma_(u1, t1, u0 * e0)));
  if constexpr (COMP) {
    const F we = fma_(f.w3, e3, fma_(f.w2, e2, fma_(f.w1, e1, f.w0 * e0)));
    s = fma_(f.beta * we, we, s);
  }
  if constexpr (!TAN) {
    acc.nis = fma_(s, acc.inv_r, acc.nis);
    const F ld = f.logdet + acc.log_rd;
    acc.logdet = acc.logdet + ld;
    if (step) { step->nis = s * acc.inv_r; step->logdet = ld; }
  } else {
    const F v1 = fma_(f.n10, z.w, z.x);
    const F v2 = fma_(f.n21, z.x, fma_(f.n20, z.w, z.y));
    const F v3 = fma_(f.n32, z.y, fma_(f.n31, z.x, fma_(f.n30, z.w, z.z)));
    const F g0 = f.i0 * z.w, g1 = f.i1 * v1, g2 = f.i2 * v2, g3 = f.i3 * v3;
    F c = fma_(g3, v3, fma_(g2, v2, fma_(g1, v1, g0 * z.w)));
    F b = fma_(g3, t3, fma_(g2, t2, fma_(g1, t1, g0 * e0)));
    if constexpr (COMP) {
      const F we = fma_(f.w3, e3, fma_(f.w2, e2, fma_(f.w1, e1, f.w0 * e0)));   // (the same value as above)
      const F wz = fma_(f.w3, z.z, fma_(f.w2, z.y, fma_(f.w1, z.x, f.w0 * z.w)));
      const F bwz = f.beta * wz;
      c = fma_(bwz, wz, c);
      b = fma_(bwz, we, b);
    }
    // ln(c/|z|^2) = ln(1 - z^T K z/|z|^2): through log1p while z^T K z/|z|^2 is small (R >> Q, and Q >> R with a slow
    // state: there the empty direction of P^- is the previous x, close to z), through the quotient beyond
    const F k0 = fma_(F(2), fma_(K.a03, z.z, fma_(K.a02, z.y, K.a01 * z.x)), K.a00 * z.w);
    const F k1 = fma_(F(2), fma_(K.a13, z.z, K.a12 * z.y), K.a11 * z.x);
    const F k2 = fma_(F(2), K.a23 * z.z, K.a22 * z.y);
    const F zkz = fma_(K.a33 * z.z, z.z, fma_(k2, z.y, fma_(k1, z.x, k0 * z.w)));
    const F iz2 = rcp_(dot4(z, z));
    const F kz = zkz * iz2;
    const F lc = sel_(kz < F(0.5), log1p_(-kz), log_(c * iz2));
    const F nis_r = fma_(-b, b * rcp_(c), s);     // r NIS_3: the value tangent_nis_r gives the gate
    acc.nis = fma_(nis_r, acc.inv_r, acc.nis);
    const F ld = (f.logdet + lc) + acc.log_rd;
    acc.logdet = acc.logdet + ld;
    if (step) { step->nis = nis_r * acc.inv_r; step->logdet = ld; }
  }
}

// ------------------------------------------------------------------------------------------
// Innovation gate (GATE): a step whose tangent-space NIS is implausible under the filter's own model is not corrected.
//     gated  <=>  NIS_3 = (s - b^2/c) / r  >  gamma,   evaluated as  s - b^2/c > gamma r   (r > 0; strict: a NaN
//                                                                                       statistic is never gated)
// with s, b, c of innov_accumulate (TAN), formed here with the same operations, so the decision is the same whichever
// model a launch accumulates and needs no logarithm (gamma r is one launch constant per filter: two registers fewer than
// 1/r and gamma in the packed kernel).  On a gated step the innovation is zeroed per lane
// (X = z + K 0 = z, then normalised: the prediction) and the covariance becomes the propagated P^- instead of K; the
// innovation sums, the flip byte and the loss still see the step.  Under a consistent model NIS_3 ~ chi^2_3.
// ------------------------------------------------------------------------------------------
template <typename F> struct GateParams {
  F thr;       // gamma r: the threshold on r NIS_3 (+inf: never gated)
};
template <typename F> PKF_HD GateParams<F> make_gate_params(F r, float gamma) {
  GateParams<F> g;
  g.thr = F(gamma) * r;
  return g;
}
// r NIS_3 = s - b^2/c (the covariance in units of r)
template <typename F, bool COMP>
PKF_HD F tangent_nis_r(const InnovFactors<F>& f, const Quat<F>& z, F e0, F e1, F e2, F e3) {
  const F t1 = fma_(f.n10, e0, e1);
  const F t2 = fma_(f.n21, e1, fma_(f.n20, e0, e2));
  const F t3 = fma_(f.n32, e2, fma_(f.n31, e1, fma_(f.n30, e0, e3)));
  const F u0 = f.i0 * e0, u1 = f.i1 * t1, u2 = f.i2 * t2, u3 = f.i3 * t3;
  F s = fma_(u3, t3, fma_(u2, t2, fma_(u1, t1, u0 * e0)));
  const F v1 = fma_(f.n10, z.w, z.x);
  const F v2 = fma_(f.n21, z.x, fma_(f.n20, z.w, z.y));
  const F v3 = fma_(f.n32, z.y, fma_(f.n31, z.x, fma_(f.n30, z.w, z.z)));
  const F g0 = f.i0 * z.w, g1 = f.i1 * v1, g2 = f.i2 * v2, g3 = f.i3 * v3;
  F c = fma_(g3, v3, fma_(g2, v2, fma_(g1, v1, g0 * z.w)));
  F b = fma_(g3, t3, fma_(g2, t2, fma_(g1, t1, g0 * e0)));
  if constexpr (COMP) {
    const F we = fma_(f.w3, e3, fma_(f.w2, e2, fma_(f.w1, e1, f.w0 * e0)));
    s = fma_(f.beta * we, we, s);
    const F wz = fma_(f.w3, z.z, fma_(f.w2, z.y, fma_(f.w1, z.x, f.w0 * z.w)));
    const F bwz = f.beta * wz;
    c = fma_(bwz, wz, c);
    b = fma_(bwz, we, b);
  }
  return fma_(-b, b * rcp_(c), s);
}

template <typename F> PKF_HD Ldl4<F> ldl_unit(const Sym4<F>& P) {
  // P is the predicted covariance IN UNITS OF r (P/r), so S = P + I and rho_k = 1/d_k.
  const F p01 = P.a01, p02 = P.a02, p03 = P.a03, p12 = P.a12, p13 = P.a13, p23 = P.a23;
  Ldl4<F> f;
  f.e0 = P.a00;                                   // delta_0
  f.i0 = rcp_(f.e0 + F(1));
  F l10 = p01 * f.i0, l20 = p02 * f.i0, l30 = p03 * f.i0;
  f.e1 = fma_(-l10, p01, P.a11);
  f.i1 = rcp_(f.e1 + F(1));
  F t21 = fma_(-l10, p02, p12);
  F t31 = fma_(-l10, p03, p13);
  F l21 = t21 * f.i1, l31 = t31 * f.i1;
  f.e2 = fma_(-l21, t21, fma_(-l20, p02, P.a22));
  f.i2 = rcp_(f.e2 + F(1));
  F t32 = fma_(-l21, t31, fma_(-l20, p03, p23));
  F l32 = t32 * f.i2;
  f.e3 = fma_(-l32, t32, fma_(-l31, t31, fma_(-l30, p03, P.a33)));
  f.i3 = rcp_(f.e3 + F(1));
  // N = L^-1 - I
  f.n10 = -l10; f.n21 = -l21; f.n32 = -l32;
  f.n20 = fma_(-l21, f.n10, -l20);
  f.n31 = fma_(-l32, f.n21, -l31);
  f.n30 = fma_(-l32, f.n20, fma_(-l31, f.n10, -l30));
  return f;
}

template <typename F> PKF_HD Sym4<F> gain_from_ldl(const Ldl4<F>& f) {
  // v_kj = -rho_k n_kj
  F v30 = -(f.i3 * f.n30), v31 = -(f.i3 * f.n31), v32 = -(f.i3 * f.n32);
  F v20 = -(f.i2 * f.n20), v21 = -(f.i2 * f.n21);
  F v10 = -(f.i1 * f.n10);
  Sym4<F> K;
  K.a00 = fma_(f.n30, v30, fma_(f.n20, v20, fma_(f.n10, v10, f.e0 * f.i0)));
  K.a01 = fma_(f.n30, v31, fma_(f.n20, v21, v10));
  K.a02 = fma_(f.n30, v32, v20);
  K.a03 = v30;
  K.a11 = fma_(f.n31, v31, fma_(f.n21, v21, f.e1 * f.i1));
  K.a12 = fma_(f.n31, v32, v21);
  K.a13 = v31;
  K.a22 = fma_(f.n32, v32, f.e2 * f.i2);
  K.a23 = v32;
  K.a33 = f.e3 * f.i3;
  return K;
}

template <typename F> PKF_HD Sym4<F> kalman_gain_unit(const Sym4<F>& P) { return gain_from_ldl(ldl_unit(P)); }

// Plain-variant form: the caller hands over S = P + I itself (propagate_cov folds the "+ 1" into the constant of its
// diagonal), the pivots d_k come straight out of the elimination and the diagonal of the gain is formed as
// kappa_k = 1 - 1/d_k.  Four additions fewer than the split-pivot form; kappa loses eps/kappa of relative accuracy,
// i.e. 2.4e-5 at the edge of the plain variant's range (r/q = 100, kappa = 2.5e-3), which moves the state by 1e-9 --
// beyond that range the precise variant (split pivots, kalman_gain_sm) is selected.
// FAC hands the factors to `fac`; LOGDET adds ln det S~ (the innovation gate reads the factors only).
template <typename F, bool FAC = false, bool LOGDET = FAC>
PKF_HD Sym4<F> kalman_gain_from_s(const Sym4<F>& S, InnovFactors<F>* fac = nullptr) {
  const F p01 = S.a01, p02 = S.a02, p03 = S.a03, p12 = S.a12, p13 = S.a13, p23 = S.a23;
  const F i0 = rcp_(S.a00);
  const F l10 = p01 * i0, l20 = p02 * i0, l30 = p03 * i0;
  const F d1 = fma_(-l10, p01, S.a11);
  const F i1 = rcp_(d1);
  const F t21 = fma_(-l10, p02, p12);
  const F t31 = fma_(-l10, p03, p13);
  const F l21 = t21 * i1, l31 = t31 * i1;
  const F d2 = fma_(-l21, t21, fma_(-l20, p02, S.a22));
  const F i2 = rcp_(d2);
  const F t32 = fma_(-l21, t31, fma_(-l20, p03, p23));
  const F l32 = t32 * i2;
  const F d3 = fma_(-l32, t32, fma_(-l31, t31, fma_(-l30, p03, S.a33)));
  const F i3 = rcp_(d3);
  // N = L^-1 - I
  const F n10 = -l10, n21 = -l21, n32 = -l32;
  const F n20 = fma_(-l21, n10, -l20);
  const F n31 = fma_(-l32, n21, -l31);
  const F n30 = fma_(-l32, n20, fma_(-l31, n10, -l30));
  if constexpr (FAC) {       // the pivots d_k of S~ = P~ + I are >= 1: their excesses d_k - 1 are exact differences
    fac->n10 = n10; fac->n20 = n20; fac->n21 = n21; fac->n30 = n30; fac->n31 = n31; fac->n32 = n32;
    fac->i0 = i0; fac->i1 = i1; fac->i2 = i2; fac->i3 = i3;
    if constexpr (LOGDET) fac->logdet = log_pivots(S.a00 - F(1), d1 - F(1), d2 - F(1), d3 - F(1));
  }
  const F v30 = -(i3 * n30), v31 = -(i3 * n31), v32 = -(i3 * n32);
  const F v20 = -(i2 * n20), v21 = -(i2 * n21);
  const F v10 = -(i1 * n10);
  Sym4<F> K;
  K.a00 = fma_(n30, v30, fma_(n20, v20, fma_(n10, v10, F(1) - i0)));
  K.a01 = fma_(n30, v31, fma_(n20, v21, v10));
  K.a02 = fma_(n30, v32, v20);
  K.a03 = v30;
  K.a11 = fma_(n31, v31, fma_(n21, v21, F(1) - i1));
  K.a12 = fma_(n31, v32, v21);
  K.a13 = v31;
  K.a22 = fma_(n32, v32, F(1) - i2);
  K.a23 = v32;
  K.a33 = F(1) - i3;
  return K;
}

// Gain for Q >> R (used by the compensated variant).  The predicted covariance in units of r is
//   P = M + g (|x|^2 I - x x^T),   M = A K A^T = O(1),   g = q/4r up to ~1e6,
// whose x-direction carries only M: forming P in float32 rounds M (and the "+ I" of S) away at
// eps*g, i.e. a 2 % error in the gain along x at g = 2.5e5.  Keep the two parts apart instead:
//   S = P + I = H - g x x^T,  H = I + M + g|x|^2 I  (condition number ~1),
//   Sherman-Morrison:  S^-1 = H^-1 + (g/den) w w^T,  w = H^-1 x,
//   den = 1 - g x^T w = x^T (I + M) w / |x|^2   (from (I + M) w + g|x|^2 w = x; no cancellation;
//         w itself comes from the LDL^T factors of H, not from x - K_H x),
//   K = I - S^-1 = K_H - beta w w^T,  K_H = I - H^-1 (split-pivot form above),  beta = g|x|^2 / x^T(I+M)w.
template <typename F, bool FAC = false, bool LOGDET = FAC>
PKF_HD Sym4<F> kalman_gain_sm(const Sym4<F>& M, const Quat<F>& x, F g, InnovFactors<F>* fac = nullptr) {
  const F x2 = dot4(x, x);
  const F c = g * x2;
  Sym4<F> PH = M;
  PH.a00 = fma_(g, x2, M.a00); PH.a11 = fma_(g, x2, M.a11); PH.a22 = fma_(g, x2, M.a22); PH.a33 = fma_(g, x2, M.a33);
  const Ldl4<F> f = ldl_unit(PH);
  const Sym4<F> KH = gain_from_ldl(f);
  // w = H^-1 x = W^T D^-1 W x, W = I + N (solved through the factors: x - K_H x would cancel when g >> 1)
  F t0 = x.w;
  F t1 = fma_(f.n10, x.w, x.x);
  F t2 = fma_(f.n21, x.x, fma_(f.n20, x.w, x.y));
  F t3 = fma_(f.n32, x.y, fma_(f.n31, x.x, fma_(f.n30, x.w, x.z)));
  F u0 = f.i0 * t0, u1 = f.i1 * t1, u2 = f.i2 * t2, u3 = f.i3 * t3;
  F w3 = u3;
  F w2 = fma_(f.n32, u3, u2);
  F w1 = fma_(f.n31, u3, fma_(f.n21, u2, u1));
  F w0 = fma_(f.n30, u3, fma_(f.n20, u2, fma_(f.n10, u1, u0)));
  // (I + M) w
  F g0 = fma_(M.a03, w3, fma_(M.a02, w2, fma_(M.a01, w1, fma_(M.a00, w0, w0))));
  F g1 = fma_(M.a13, w3, fma_(M.a12, w2, fma_(M.a11, w1, fma_(M.a01, w0, w1))));
  F g2 = fma_(M.a23, w3, fma_(M.a22, w2, fma_(M.a12, w1, fma_(M.a02, w0, w2))));
  F g3 = fma_(M.a33, w3, fma_(M.a23, w2, fma_(M.a13, w1, fma_(M.a03, w0, w3))));
  F num = fma_(x.z, g3, fma_(x.y, g2, fma_(x.x, g1, x.w * g0)));
  F nb = -(c * rcp_(num));                     // -beta
  if constexpr (FAC) {
    fac->n10 = f.n10; fac->n20 = f.n20; fac->n21 = f.n21; fac->n30 = f.n30; fac->n31 = f.n31; fac->n32 = f.n32;
    fac->i0 = f.i0; fac->i1 = f.i1; fac->i2 = f.i2; fac->i3 = f.i3;
    fac->w0 = w0; fac->w1 = w1; fac->w2 = w2; fac->w3 = w3; fac->beta = -nb;
    if constexpr (LOGDET) {
      // ln(num/|x|^2) = ln(1 - g x.w): through log1p while g x.w is small (R >> Q: the term is ~ -g and the quotient
      // would round it away), through the quotient itself when it is small (Q >> R: 1 - g x.w would cancel)
      const F u = g * fma_(x.z, w3, fma_(x.y, w2, fma_(x.x, w1, x.w * w0)));
      const F lden = sel_(u < F(0.5), log1p_(-u), log_(num * rcp_(x2)));
      fac->logdet = log_pivots(f.e0, f.e1, f.e2, f.e3) + lden;
    }
  }
  F b0 = nb * w0, b1 = nb * w1, b2 = nb * w2, b3 = nb * w3;
  Sym4<F> K;
  K.a00 = fma_(b0, w0, KH.a00); K.a01 = fma_(b0, w1, KH.a01); K.a02 = fma_(b0, w2, KH.a02); K.a03 = fma_(b0, w3, KH.a03);
  K.a11 = fma_(b1, w1, KH.a11); K.a12 = fma_(b1, w2, KH.a12); K.a13 = fma_(b1, w3, KH.a13);
  K.a22 = fma_(b2, w2, KH.a22); K.a23 = fma_(b2, w3, KH.a23);
  K.a33 = fma_(b3, w3, KH.a33);
  return K;
}

// ------------------------------------------------------------------------------------------
// Wahba, rank-2 form.   B = ka r_a a^T + km r_m m^T = [e1 e2] C [f1 f2]^T  with
//   C = [[s11 s12],[0 s22]] diag(ka,km) [[t11 0],[t12 t22]]   (2x2).
// SVD of C = Uc S Vc^T  =>  U = [E2 Uc, e3], V = [F2 Vc, f3] and the reference's
//   R = U diag(1,1,det U det V^T) V^T = E blockdiag(Uc Vc^T, det(Uc Vc^T)) F^T   (PKF/Wahba.py:14-16).
// Uc Vc^T is the orthogonal polar factor of C, closed form for 2x2:
//   sg = sign(det C) = sign(ka km)  (all other factors of det C are norms),
//   p = c00 + sg c11, r = c10 - sg c01,  Uc Vc^T = [[p, -sg r],[r, sg p]] / hypot(p,r).
// rank(C) < 2 (ka km == 0, or a || m, or r_a || r_m) is the case where LAPACK's null-space choice
// decides the reference's answer ("parity unpinned", SURVEY.md section 7.3); here it yields the
// limit of the rank-2 formula (or NaN if a vector is zero).
// ------------------------------------------------------------------------------------------
// wahba_qr2_local returns the rotation IN THE COORDINATES OF THE REFERENCE FRAME E, i.e. E^T R =
// blockdiag(Uc Vc^T, det) F^T -- twelve multiply-adds instead of the 39 of the full product.  The fused
// step runs the whole filter in that frame (see "filter frame" below); wahba_qr2 = E * local is the
// reference's R for the stand-alone entry points.
template <typename F>
PKF_HD Mat3<F> wahba_qr2_local(const RefFrame<F>& E, const Vec3<F>& a, const Vec3<F>& m, F ka, F km) {
  RefFrame<F> Fb = frame_from_pair(a, m);
  // (every product that feeds a sum is an explicit fma_: nothing is left to the compiler's
  //  contraction heuristics, so the scalar, packed and host builds round identically)
  const auto neg = (ka * km) < F(0);
  F g = km * Fb.s12, hh = km * Fb.s22;
  // sg = sign(ka km) is +1 whenever both weights are positive (always for normalised accelerometer
  // input: ka = |a_z| <= 1); the reflected case flips the sign of c01 and c11.
  if (any_(neg)) hh = sel_(neg, -hh, hh);
  F c00 = fma_(E.s12, g, (E.s11 * ka) * Fb.s11);
  F c01 = E.s12 * hh;                      // sg c01
  F p = fma_(E.s22, hh, c00);              // c00 + sg c11
  F r = fma_(E.s22, g, -c01);              // c10 - sg c01
  F inv = rsqrt_(fma_(p, p, r * r));
  F cs = p * inv, sn = r * inv;
  // rows of blockdiag([[cs, -sg sn],[sn, sg cs]], sg) F^T
  F g01 = -sn, g11 = cs;
  Vec3<F> f3 = Fb.e3;
  if (any_(neg)) {
    g01 = sel_(neg, sn, g01); g11 = sel_(neg, -cs, g11);
    f3.x = sel_(neg, -f3.x, f3.x); f3.y = sel_(neg, -f3.y, f3.y); f3.z = sel_(neg, -f3.z, f3.z);
  }
  const Vec3<F>&f1 = Fb.e1, &f2 = Fb.e2;
  Mat3<F> R;
  R.m[0][0] = fma_(g01, f2.x, cs * f1.x); R.m[0][1] = fma_(g01, f2.y, cs * f1.y); R.m[0][2] = fma_(g01, f2.z, cs * f1.z);
  R.m[1][0] = fma_(g11, f2.x, sn * f1.x); R.m[1][1] = fma_(g11, f2.y, sn * f1.y); R.m[1][2] = fma_(g11, f2.z, sn * f1.z);
  R.m[2][0] = f3.x; R.m[2][1] = f3.y; R.m[2][2] = f3.z;
  return R;
}

// ------------------------------------------------------------------------------------------
// Wahba, two observations, solved DIRECTLY AS A QUATERNION in the filter frame (fused step).
// For two weighted observations the maximiser of tr(R B^T) has a closed form in the quaternion
// itself (F. L. Markley, "Fast quaternion attitude estimation from two vector measurements", 2002):
// with the unit normals b3 = u1 x u2 / |.| of the reference pair and r3 = v1 x v2 / |.| of the
// measured pair, S = sum w_i u_i.v_i and V = sum w_i u_i x v_i,
//     alpha = (1 + b3.r3) S + (b3 x r3).V,   beta = (b3 + r3).V,   gamma = hypot(alpha, beta),
//     q ~ [ (gamma+alpha)(1 + b3.r3) ;  (gamma+alpha)(b3 x r3) + beta (b3 + r3) ]        alpha >= 0
//     q ~ [  beta (1 + b3.r3)        ;   beta (b3 x r3) + (gamma-alpha)(b3 + r3) ]       alpha <  0
// (vector part conjugated for the Hamilton body->reference convention of the reference's
// RotationMatrix2Quart).  It is the same rotation as U diag(1,1,det U det V^T) V^T of PKF/Wahba.py:14-16
// whenever both weights are positive (rank-2 B): like wahba_qr2 it never forms B, the weights enter
// linearly, so it stays accurate to float32 rounding for |a_z| -> 0 or 1.  Un-normalised vectors are
// weights (w_1 u_1.v_1 = ka (r_a.a), ...), so nothing but the normal r3 is normalised.
// In the filter frame r_a = (s11,0,0), r_m = (s12,s22,0), b3 = (0,0,1), and most products vanish.
// 1 + b3.r3 -> 0 (measured normal opposite to the reference normal) is the formula's singularity:
// when r3.z < 0 the measured pair is first half-turned about the body x axis (y and z components
// negated, so r3.z -> |r3.z|) and the half-turn is composed back into the result, q (x) (0,1,0,0) =
// (-x, w, z, -y); 1 + b3.r3 >= 1 always.
// 50 FP32 operations + 3 MUFU for the quaternion and its inverse norm (sign arbitrary), against 92 for frame, 2x2
// polar factor, rotation matrix and matrix->quaternion.
// ------------------------------------------------------------------------------------------
// Returns the UN-NORMALISED quaternion and, through inv_norm, 1/|y|: the fused step folds the normalisation into
// its innovation (e = (sg/|y|) y - z), one multiplication instead of four.
template <typename F>
PKF_HD Quat<F> wahba_quat2_local(const RefFrame<F>& E, const Vec3<F>& a, const Vec3<F>& m, F ka, F km, F& inv_norm) {
  const Vec3<F> c = cross3(a, m);
  // half-turn of the measured pair when c.z < 0: sigma = sign(c.z) multiplies the y and z components of a, m
  // and c; it cancels in every product of two flipped quantities, four conditional negations remain
  const F ays = flipsign_(a.y, c.z), mys = flipsign_(m.y, c.z);
  const F ic = rsqrt_(dot3(c, c));
  const F rx = c.x * ic, ry0 = c.y * ic;                          // r3 = (rx, sigma ry0, |c.z| ic)
  const F rxs = flipsign_(rx, c.z), ry = flipsign_(ry0, c.z);
  // weights times the reference pair (s11,0,0), (s12,s22,0), all divided by s11 (the result's scale is free)
  const F A1 = ka, B1 = km * E.r12, B2 = km * E.r22;
  const F S = fma_(B2, mys, fma_(B1, m.x, A1 * a.x));             // sum w_i u_i.v_i
  const F Vx0 = B2 * m.z;                                         // sum w_i u_i x v_i = (sigma Vx0, sigma Vy0, Vz)
  const F Vy0 = -fma_(B1, m.z, A1 * a.z);
  const F Vz = fma_(-B2, m.x, fma_(B1, mys, A1 * ays));
  const F d = fma_(abs_(c.z), ic, F(1));                          // 1 + b3.r3  (explicit fma_: see propagate_cov)
  const F al = fma_(-ry0, Vx0, fma_(rxs, Vy0, d * S));
  const F be = fma_(d, Vz, fma_(ry0, Vy0, rxs * Vx0));
  const F g2 = fma_(al, al, be * be);
  const F t = fma_(g2, rsqrt_(g2), abs_(al));                     // gamma + |alpha|
  const F p = selsign_(al, be, t), q = selsign_(al, t, be);       // alpha < 0: the other, cancellation-free form
  // [sc; vec] = [p d; p (b3 x r3) + q (b3 + r3)],  b3 x r3 = (-ry, rx, 0),  b3 + r3 = (rx, ry, d)
  Quat<F> y;
  y.w = p * d;
  y.x = -fma_(q, rx, -(p * ry));
  y.y = -fma_(q, ry, p * rx);
  y.z = -(q * d);
  inv_norm = rsqrt_(dot4(y, y));
  // undo the half-turn of the measured pair:  y (x) (0,1,0,0) = (-x, w, z, -y)
  Quat<F> o;
  o.w = flipsign_(selsign_(c.z, y.x, y.w), c.z); o.x = selsign_(c.z, y.w, y.x);
  o.y = selsign_(c.z, y.z, y.y); o.z = flipsign_(selsign_(c.z, y.y, y.z), c.z);
  return o;
}

// columns of E times the rows of a local-frame matrix:  R = E L
template <typename F> PKF_HD Mat3<F> frame_times(const RefFrame<F>& E, const Mat3<F>& L) {
  Mat3<F> R;
  const F ex[3] = {E.e1.x, E.e1.y, E.e1.z}, ey[3] = {E.e2.x, E.e2.y, E.e2.z}, ez[3] = {E.e3.x, E.e3.y, E.e3.z};
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int i = 0; i < 3; ++i) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int j = 0; j < 3; ++j) R.m[i][j] = fma_(ez[i], L.m[2][j], fma_(ey[i], L.m[1][j], ex[i] * L.m[0][j]));
  }
  return R;
}
// E^T R: a reference-frame rotation expressed in the coordinates of E
template <typename F> PKF_HD Mat3<F> frame_transposed_times(const RefFrame<F>& E, const Mat3<F>& R) {
  Mat3<F> L;
  const Vec3<F> e[3] = {E.e1, E.e2, E.e3};
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int k = 0; k < 3; ++k) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int j = 0; j < 3; ++j) L.m[k][j] = fma_(e[k].z, R.m[2][j], fma_(e[k].y, R.m[1][j], e[k].x * R.m[0][j]));
  }
  return L;
}

template <typename F>
PKF_HD Mat3<F> wahba_qr2(const RefFrame<F>& E, const Vec3<F>& a, const Vec3<F>& m, F ka, F km) {
  return frame_times(E, wahba_qr2_local(E, a, m, ka, km));
}

// ------------------------------------------------------------------------------------------
// Wahba by a one-sided (Hestenes) Jacobi SVD, QR-preconditioned                         (PKF/Wahba.py:8-17)
//
// The reference takes the SVD of the 3x3 B = ka r_a a^T + km r_m m^T.  In float32 that matrix cannot be FORMED
// without losing the answer: its weights ka = |a_z|, km = 1 - |a_z| drive it to rank 1, and rounding B's entries
// costs eps * sigma1/sigma2 in the rotation (1.5e-2 rad measured on the synthetic set with a plain float32 Jacobi
// of B, 2.9e-5 rad on config 4 -- round 1).  The remedy is the standard one for Jacobi SVDs (Drmac & Veselic: QR
// factorisation first, Jacobi on the triangular factor): B has rank 2 by construction,
//     B = [u1 u2] diag(w1, w2) [v1 v2]^T = E2 (S W T^T) F2^T,   [u1 u2] = E2 S,  [v1 v2] = F2 T   (S, T upper triangular)
// so the SVD that matters is that of the 2x2 core C = S W T^T, whose four entries are products of norms and dot
// products -- nothing is summed across scales except in c00.  With the pairs ORDERED so that the heavier one comes
// first (column pivoting) C is graded: a dominant c00 and three entries of the lighter pair's size, which is the
// shape one-sided Jacobi resolves to full relative accuracy.  A 2x2 needs exactly ONE rotation:
//     columns c0, c1 of C;  t = sgn(d) 2 c0.c1 / (|d| + hypot(d, 2 c0.c1)),  d = |c1|^2 - |c0|^2;
//     G = C J (orthogonal columns g0, g1), V = J, U = [g0/|g0|, g1/|g1|]
// and with U = [E2 Uc, e3], V = [F2 Vc, f3] the reference's R = U diag(1,1,det U det V^T) V^T becomes
//     R = E blockdiag(Uc Vc^T, det(Uc Vc^T)) F^T.
// `sweeps` is accepted for interface compatibility (the 3x3 form iterated; one rotation is exact here).
// There is nothing left to spread over a quad of lanes or to shuffle: the rotation is 30 operations in registers.
// ------------------------------------------------------------------------------------------
template <typename F>
PKF_HD Mat3<F> wahba_jacobi(const Vec3<F>& ra, const Vec3<F>& rm, const Vec3<F>& a, const Vec3<F>& m, F ka, F km, int /*sweeps*/) {
  // column pivoting: the pair with the larger weighted size |w| |u| |v| first (compared squared)
  const F za = (ka * ka) * (dot3(ra, ra) * dot3(a, a)), zm = (km * km) * (dot3(rm, rm) * dot3(m, m));
  const auto swap = zm > za;
  Vec3<F> u1, u2, v1, v2;
  u1.x = sel_(swap, rm.x, ra.x); u1.y = sel_(swap, rm.y, ra.y); u1.z = sel_(swap, rm.z, ra.z);
  u2.x = sel_(swap, ra.x, rm.x); u2.y = sel_(swap, ra.y, rm.y); u2.z = sel_(swap, ra.z, rm.z);
  v1.x = sel_(swap, m.x, a.x); v1.y = sel_(swap, m.y, a.y); v1.z = sel_(swap, m.z, a.z);
  v2.x = sel_(swap, a.x, m.x); v2.y = sel_(swap, a.y, m.y); v2.z = sel_(swap, a.z, m.z);
  const F w1 = sel_(swap, km, ka), w2 = sel_(swap, ka, km);
  const RefFrame<F> E = frame_from_pair(u1, u2), Fb = frame_from_pair(v1, v2);
  // C = S diag(w1, w2) T^T
  const F e12 = E.s12 * w2, e22 = E.s22 * w2;
  const F c00 = fma_(e12, Fb.s12, (E.s11 * w1) * Fb.s11), c01 = e12 * Fb.s22;
  const F c10 = e22 * Fb.s12, c11 = e22 * Fb.s22;
  // the one Jacobi rotation that makes the columns of C orthogonal
  const F al = fma_(c10, c10, c00 * c00), be = fma_(c11, c11, c01 * c01), ga = fma_(c10, c11, c00 * c01);
  const F d = be - al, g2 = ga + ga;
  const F den = abs_(d) + sqrt_(fma_(d, d, g2 * g2));
  const F t = sel_(den > F(0), sel_(d < F(0), -g2, g2) * rcp_(den), F(0));
  const F c = rsqrt_(fma_(t, t, F(1))), sn = c * t;
  const F g00 = fma_(-sn, c01, c * c00), g10 = fma_(-sn, c11, c * c10);      // g0 = c c0 - s c1
  const F g01 = fma_(sn, c00, c * c01), g11 = fma_(sn, c10, c * c11);        // g1 = s c0 + c c1
  const F i0 = rsqrt_(fma_(g10, g10, g00 * g00)), i1 = rsqrt_(fma_(g11, g11, g01 * g01));
  const F u00 = g00 * i0, u10 = g10 * i0, u01 = g01 * i1, u11 = g11 * i1;    // Uc = [u0 u1]
  // M = Uc Vc^T with Vc = [[c, s], [-s, c]] (columns v0 = (c, -s), v1 = (s, c))
  const F m00 = fma_(u01, sn, u00 * c), m01 = fma_(u01, c, -(u00 * sn));
  const F m10 = fma_(u11, sn, u10 * c), m11 = fma_(u11, c, -(u10 * sn));
  const F dt = one_with_sign_(fma_(m00, m11, -(m01 * m10)));                 // det(Uc Vc^T) = +-1
  Mat3<F> L;                                                                 // blockdiag(M, det) F^T
  L.m[0][0] = fma_(m01, Fb.e2.x, m00 * Fb.e1.x); L.m[0][1] = fma_(m01, Fb.e2.y, m00 * Fb.e1.y); L.m[0][2] = fma_(m01, Fb.e2.z, m00 * Fb.e1.z);
  L.m[1][0] = fma_(m11, Fb.e2.x, m10 * Fb.e1.x); L.m[1][1] = fma_(m11, Fb.e2.y, m10 * Fb.e1.y); L.m[1][2] = fma_(m11, Fb.e2.z, m10 * Fb.e1.z);
  L.m[2][0] = dt * Fb.e3.x; L.m[2][1] = dt * Fb.e3.y; L.m[2][2] = dt * Fb.e3.z;
  return frame_times(E, L);
}

// ------------------------------------------------------------------------------------------
// Rotation matrix -> quaternion.                                    (PKF/Wahba.py:20-47)
// The reference picks branch i in {x,y,z} by the strict maximum of tr1,tr2,tr3 (ties -> z) and
// returns the quaternion whose component i is >= 0; it has no "w largest" branch, so close to the
// identity its formula divides by a vanishing S (harmless in float64, not in float32).  Here the
// components come from the best conditioned of the four Shepperd candidates, then the reference's
// SIGN convention is applied from its own branch rule, so the value equals the reference's output
// up to rounding.  At M == I exactly the reference returns [nan,nan,nan,0]; so does this.
// `q` is returned with the reference sign; it is normalised (the reference's is unit to rounding
// when M is a rotation).
// ------------------------------------------------------------------------------------------
template <typename F> PKF_HD Quat<F> rotation_to_quat_ref(const Mat3<F>& M) {
  const F r00 = M.m[0][0], r11 = M.m[1][1], r22 = M.m[2][2];
  // the reference's three traces, evaluated in the reference's order of operations
  F tr1 = F(1) + r00 - r11 - r22;
  F tr2 = F(1) - r00 + r11 - r22;
  F tr3 = F(1) - r00 - r11 + r22;
  F tr0 = F(1) + r00 + r11 + r22;
  F dx = M.m[2][1] - M.m[1][2], dy = M.m[0][2] - M.m[2][0], dz = M.m[1][0] - M.m[0][1];
  F sxy = M.m[0][1] + M.m[1][0], sxz = M.m[0][2] + M.m[2][0], syz = M.m[1][2] + M.m[2][1];
  // reference branch (sign convention): 1 -> x, 2 -> y, else z
  auto b1 = (tr1 > tr2) && (tr1 > tr3);
  auto b2 = !b1 && ((tr2 > tr1) && (tr2 > tr3));
  // best-conditioned candidate among (w,x,y,z): the largest of the four traces (independent of the
  // reference's tie rule, which only fixes the sign)
  auto w_gt_x = tr0 > tr1, y_gt_z = tr2 > tr3;
  F mwx = sel_(w_gt_x, tr0, tr1), myz = sel_(y_gt_z, tr2, tr3);
  auto lo = mwx > myz;                           // winner is w or x, else y or z
  auto kw = lo && w_gt_x, kx = lo && !w_gt_x, ky = !lo && y_gt_z;
  Quat<F> c;
  c.w = sel_(kw, tr0, sel_(kx, dx, sel_(ky, dy, dz)));
  c.x = sel_(kw, dx, sel_(kx, tr1, sel_(ky, sxy, sxz)));
  c.y = sel_(kw, dy, sel_(kx, sxy, sel_(ky, tr2, syz)));
  c.z = sel_(kw, dz, sel_(kx, sxz, sel_(ky, syz, tr3)));
  F inv = rsqrt_(dot4(c, c));
  // sign: the reference's component i (= 0.25 S) is positive
  F ci = sel_(b1, c.x, sel_(b2, c.y, c.z));
  inv = sel_(ci < F(0), -inv, inv);
  Quat<F> q;
  q.w = c.w * inv; q.x = c.x * inv; q.y = c.y * inv; q.z = c.z * inv;
  // exact identity: S = 0 in the reference's last branch -> 0/0, 0/0, 0/0, 0.25*0
  auto ident = ((tr1 == F(0)) && (tr2 == F(0))) && ((tr3 == F(0)) && (dx == F(0))) && ((dy == F(0)) && (dz == F(0)));
  F nanv = F(NAN);
  q.w = sel_(ident, nanv, q.w); q.x = sel_(ident, nanv, q.x); q.y = sel_(ident, nanv, q.y); q.z = sel_(ident, F(0), q.z);
  return q;
}

// Rotation matrix -> unit quaternion of EITHER sign from the best-conditioned Shepperd candidate; no
// reference sign rule and no NaN at the identity (used for the filter-frame quaternion of E).
template <typename F> PKF_HD Quat<F> rotation_to_quat_best(const Mat3<F>& M) {
  const F r00 = M.m[0][0], r11 = M.m[1][1], r22 = M.m[2][2];
  F tr1 = F(1) + r00 - r11 - r22, tr2 = F(1) - r00 + r11 - r22, tr3 = F(1) - r00 - r11 + r22, tr0 = F(1) + r00 + r11 + r22;
  F dx = M.m[2][1] - M.m[1][2], dy = M.m[0][2] - M.m[2][0], dz = M.m[1][0] - M.m[0][1];
  F sxy = M.m[0][1] + M.m[1][0], sxz = M.m[0][2] + M.m[2][0], syz = M.m[1][2] + M.m[2][1];
  auto w_gt_x = tr0 > tr1, y_gt_z = tr2 > tr3;
  F mwx = sel_(w_gt_x, tr0, tr1), myz = sel_(y_gt_z, tr2, tr3);
  auto lo = mwx > myz;
  auto kw = lo && w_gt_x, kx = lo && !w_gt_x, ky = !lo && y_gt_z;
  Quat<F> c;
  c.w = sel_(kw, tr0, sel_(kx, dx, sel_(ky, dy, dz)));
  c.x = sel_(kw, dx, sel_(kx, tr1, sel_(ky, sxy, sxz)));
  c.y = sel_(kw, dy, sel_(kx, sxy, sel_(ky, tr2, syz)));
  c.z = sel_(kw, dz, sel_(kx, sxz, sel_(ky, syz, tr3)));
  F inv = rsqrt_(dot4(c, c));
  c.w *= inv; c.x *= inv; c.y *= inv; c.z *= inv;
  return c;
}

// Hamilton product a (x) b, scalar first
template <typename F> PKF_HD Quat<F> qmul(const Quat<F>& a, const Quat<F>& b) {
  Quat<F> c;
  c.w = fma_(-a.z, b.z, fma_(-a.y, b.y, fma_(-a.x, b.x, a.w * b.w)));
  c.x = fma_(-a.z, b.y, fma_(a.y, b.z, fma_(a.x, b.w, a.w * b.x)));
  c.y = fma_(a.z, b.x, fma_(a.y, b.w, fma_(-a.x, b.z, a.w * b.y)));
  c.z = fma_(a.z, b.w, fma_(-a.y, b.x, fma_(a.x, b.y, a.w * b.z)));
  return c;
}
template <typename F> PKF_HD Quat<F> qconj(const Quat<F>& a) { Quat<F> c = {a.w, -a.x, -a.y, -a.z}; return c; }

// L(p) P L(p)^T for the left-multiplication matrix L(p) of a unit quaternion p (orthogonal), P symmetric:
// the covariance of p (x) x when P is the covariance of x.
template <typename F> PKF_HD Sym4<F> rotate_cov(const Quat<F>& p, const Sym4<F>& P) {
  const F a = p.w, b = p.x, c = p.y, d = p.z;
  const F L[4][4] = {{a, -b, -c, -d}, {b, a, -d, c}, {c, d, a, -b}, {d, -c, b, a}};
  const F S[4][4] = {{P.a00, P.a01, P.a02, P.a03}, {P.a01, P.a11, P.a12, P.a13}, {P.a02, P.a12, P.a22, P.a23},
                     {P.a03, P.a13, P.a23, P.a33}};
  F M[4][4];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int i = 0; i < 4; ++i) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int j = 0; j < 4; ++j) M[i][j] = fma_(L[i][3], S[3][j], fma_(L[i][2], S[2][j], fma_(L[i][1], S[1][j], L[i][0] * S[0][j])));
  }
  auto e = [&](int i, int j) { return fma_(M[i][3], L[j][3], fma_(M[i][2], L[j][2], fma_(M[i][1], L[j][1], M[i][0] * L[j][0]))); };
  Sym4<F> N = {e(0, 0), e(0, 1), e(0, 2), e(0, 3), e(1, 1), e(1, 2), e(1, 3), e(2, 2), e(2, 3), e(3, 3)};
  return N;
}

// ------------------------------------------------------------------------------------------
// Rotation matrix -> quaternion ALIGNED WITH A PREDICTION z (fused-step form).
// For a rotation M = R(y) the symmetric 4x4 matrix built from the four Shepperd candidates is
// 4 y y^T (rows: [tr0 dx dy dz], [dx tr1 sxy sxz], [dy sxy tr2 syz], [dz sxz syz tr3]), so
//     (4 y y^T) z = 4 (y.z) y
// is y with the sign that makes y.z >= 0 -- exactly the vector the reference has after its
// q/-q fix (PKF/ExtendedKalmanFilter.py:73-75) -- obtained without any compare/select and
// conditioned by |y.z| (~1 in a tracking filter) instead of by the largest trace.  The caller
// falls back to rotation_to_quat_ref when |y.z| is small (prediction and measurement ~180 deg
// apart in 4-D, i.e. unrelated).  Returns the un-normalised 4 (y.z) y and its squared norm
// 16 (y.z)^2 through n2.
// ------------------------------------------------------------------------------------------
template <typename F> PKF_HD Quat<F> rotation_to_quat_aligned(const Mat3<F>& M, const Quat<F>& z, F& n2) {
  const F r00 = M.m[0][0], r11 = M.m[1][1], r22 = M.m[2][2];
  F a = r00 + r11, b = r00 - r11, p1 = F(1) + r22, m1 = F(1) - r22;
  F tr0 = p1 + a, tr3 = p1 - a, tr1 = m1 + b, tr2 = m1 - b;
  F dx = M.m[2][1] - M.m[1][2], dy = M.m[0][2] - M.m[2][0], dz = M.m[1][0] - M.m[0][1];
  F sxy = M.m[0][1] + M.m[1][0], sxz = M.m[0][2] + M.m[2][0], syz = M.m[1][2] + M.m[2][1];
  Quat<F> c;
  c.w = fma_(dz, z.z, fma_(dy, z.y, fma_(dx, z.x, tr0 * z.w)));
  c.x = fma_(sxz, z.z, fma_(sxy, z.y, fma_(tr1, z.x, dx * z.w)));
  c.y = fma_(syz, z.z, fma_(tr2, z.y, fma_(sxy, z.x, dy * z.w)));
  c.z = fma_(tr3, z.z, fma_(syz, z.y, fma_(sxz, z.x, dz * z.w)));
  n2 = dot4(c, c);
  return c;
}

// The reference's q/-q decision for a measurement whose aligned form is y (y.z >= 0): the
// reference's raw quaternion has component i >= 0 (i = its branch), so it negated iff y_i < 0.
template <typename F> PKF_HD auto reference_flip(const Mat3<F>& M, const Quat<F>& y) -> decltype(y.w < y.w) {
  const F r00 = M.m[0][0], r11 = M.m[1][1], r22 = M.m[2][2];
  F tr1 = F(1) + r00 - r11 - r22, tr2 = F(1) - r00 + r11 - r22, tr3 = F(1) - r00 - r11 + r22;
  auto b1 = (tr1 > tr2) && (tr1 > tr3);
  auto b2 = !b1 && ((tr2 > tr1) && (tr2 > tr3));
  return sel_(b1, y.x, sel_(b2, y.y, y.z)) < F(0);
}

// Same decision when the rotation Ml and the aligned measurement yl are given in the filter frame: the
// reference's branch rule looks at the diagonal of R = E Ml and at the components of qE (x) yl.
template <typename F, typename FC>
PKF_HD auto reference_flip_local(const FC& fc, const Mat3<F>& Ml, const Quat<F>& yl) -> decltype(yl.w < yl.w) {
  const RefFrame<F>& E = fc.E;
  const F r00 = fma_(E.e3.x, Ml.m[2][0], fma_(E.e2.x, Ml.m[1][0], E.e1.x * Ml.m[0][0]));
  const F r11 = fma_(E.e3.y, Ml.m[2][1], fma_(E.e2.y, Ml.m[1][1], E.e1.y * Ml.m[0][1]));
  const F r22 = fma_(E.e3.z, Ml.m[2][2], fma_(E.e2.z, Ml.m[1][2], E.e1.z * Ml.m[0][2]));
  F tr1 = F(1) + r00 - r11 - r22, tr2 = F(1) - r00 + r11 - r22, tr3 = F(1) - r00 - r11 + r22;
  auto b1 = (tr1 > tr2) && (tr1 > tr3);
  auto b2 = !b1 && ((tr2 > tr1) && (tr2 > tr3));
  const Quat<F> y = qmul(fc.qE, yl);
  return sel_(b1, y.x, sel_(b2, y.y, y.z)) < F(0);
}

// ------------------------------------------------------------------------------------------
// EXACT form of the reference's sign rule, for the rare samples where float32 cannot decide it.
// RotationMatrix2Quart (PKF/Wahba.py:20-47) returns the quaternion whose component i is >= 0, i being the strict
// maximum of tr1, tr2, tr3 = 4x^2, 4y^2, 4z^2 (else the third).  When two of the squares agree to ~1e-5 the float32
// quaternion (error ~1e-7) may order them differently from the float64 reference, and the q/-q flip mask -- which
// north_star requires to be IDENTICAL -- would differ.  Those samples (a few per 1e5) redo the measurement in
// float64 from the raw float32 sensor and reference vectors, exactly the values the reference consumes, and decide
// there.  Returns the reference's branch: 0, 1, 2 for the x, y, z component.
// ------------------------------------------------------------------------------------------
PKF_HD_RARE int reference_branch_exact(float rax, float ray, float raz, float rmx, float rmy, float rmz,
                                       float ax, float ay, float az, float mx, float my, float mz, float ka_f, float km_f) {
  const Vec3<double> ra = {(double)rax, (double)ray, (double)raz}, rm = {(double)rmx, (double)rmy, (double)rmz};
  const Vec3<double> a = {(double)ax, (double)ay, (double)az}, m = {(double)mx, (double)my, (double)mz};
  const double ka = (double)ka_f, km = (double)km_f;
  const RefFrame<double> E = frame_from_pair<double>(ra, rm);
  Quat<double> yl;
  if (ka * km < 0.0 || ka < 0.0) {                    // reflected Wahba problem: the rank-2 SVD form
    yl = rotation_to_quat_best<double>(wahba_qr2_local<double>(E, a, m, ka, km));
  } else {
    double inv_norm;
    yl = wahba_quat2_local<double>(E, a, m, ka, km, inv_norm);
  }
  Mat3<double> Em;
  Em.m[0][0] = E.e1.x; Em.m[1][0] = E.e1.y; Em.m[2][0] = E.e1.z;
  Em.m[0][1] = E.e2.x; Em.m[1][1] = E.e2.y; Em.m[2][1] = E.e2.z;
  Em.m[0][2] = E.e3.x; Em.m[1][2] = E.e3.y; Em.m[2][2] = E.e3.z;
  const Quat<double> y = qmul(rotation_to_quat_best<double>(Em), yl);
  const double sx = y.x * y.x, sy = y.y * y.y, sz = y.z * y.z;
  return (sx > sy && sx > sz) ? 0 : ((sy > sx && sy > sz) ? 1 : 2);       // PKF/Wahba.py:26,33: strict maximum, else the third
}

// |gap| between two of the squared vector components below kTieTol * |y|^2: hand the sign rule to the exact form
// (cheap over-approximation of "the two LARGEST are close"; a few samples per 1e5).
constexpr float kTieTol = 1e-5f;
PKF_HD bool near_tie_(float sx, float sy, float sz, float n2) {
  const float t = kTieTol * n2;
  return abs_(sx - sy) < t || abs_(sx - sz) < t || abs_(sy - sz) < t;
}
PKF_HD bool near_tie_(double, double, double, double) { return false; }     // the float64 build is its own exact form
PKF_HD mask2 near_tie_(const f32x2& sx, const f32x2& sy, const f32x2& sz, const f32x2& n2) {
  return mask2{near_tie_(sx.x, sy.x, sz.x, n2.x), near_tie_(sx.y, sy.y, sz.y, n2.y)};
}
// component of lane `lane`
PKF_HD float lane_(float v, int) { return v; }
PKF_HD double lane_(double v, int) { return v; }
PKF_HD float lane_(const f32x2& v, int lane) { return lane ? v.y : v.x; }
PKF_HD bool lane_(bool v, int) { return v; }
PKF_HD bool lane_(const mask2& v, int lane) { return lane ? v.y : v.x; }
PKF_HD void set_lane_(bool& m, int, bool v) { m = v; }
PKF_HD void set_lane_(mask2& m, int lane, bool v) { if (lane) m.y = v; else m.x = v; }
PKF_HD void negate_lane_(Quat<float>& q, int) { q.w = -q.w; q.x = -q.x; q.y = -q.y; q.z = -q.z; }
PKF_HD void negate_lane_(Quat<double>& q, int) { q.w = -q.w; q.x = -q.x; q.y = -q.y; q.z = -q.z; }
PKF_HD void negate_lane_(Quat<f32x2>& q, int lane) {
  if (lane) { q.w.y = -q.w.y; q.x.y = -q.x.y; q.y.y = -q.y.y; q.z.y = -q.z.y; }
  else { q.w.x = -q.w.x; q.x.x = -q.x.x; q.y.x = -q.y.x; q.z.x = -q.z.x; }
}
template <typename F> struct Lanes { static constexpr int n = 1; };
template <> struct Lanes<f32x2> { static constexpr int n = 2; };

// The same decision from the quaternion alone: for a rotation matrix the three traces of
// RotationMatrix2Quart are 4x^2, 4y^2, 4z^2 of its quaternion, so the reference's branch is the largest of
// |x|, |y|, |z| (strictly; else the third), its raw quaternion has that component >= 0, and it negated iff the
// comparator-aligned quaternion (sg * y, expressed in the reference frame) has it negative.
// Near a tie of two squares float32 cannot reproduce the float64 reference's choice; the flip-mask byte then carries,
// beside the float32 decision (bit 0), what the decision would be for each of the three branches (bits 1-3: x, y, z)
// and a tie marker (bit 7), and flip_fixup_kernel (ops_kernels.cuh) settles those few bytes in float64 after the
// launch (reference_branch_exact).  The hot kernels never call the float64 path.
struct FlipCode2 { unsigned x, y; };
PKF_HD unsigned flip_code_(bool flip, bool tie, bool fx, bool fy, bool fz) {
  return (flip ? 1u : 0u) | (tie ? (0x80u | (fx ? 2u : 0u) | (fy ? 4u : 0u) | (fz ? 8u : 0u)) : 0u);
}
PKF_HD FlipCode2 flip_code_(const mask2& flip, const mask2& tie, const mask2& fx, const mask2& fy, const mask2& fz) {
  return FlipCode2{flip_code_(flip.x, tie.x, fx.x, fy.x, fz.x), flip_code_(flip.y, tie.y, fx.y, fy.y, fz.y)};
}
template <typename F> struct FlipCodeOf { typedef unsigned type; };
template <> struct FlipCodeOf<f32x2> { typedef FlipCode2 type; };

template <typename F, typename FC>
PKF_HD auto reference_flip_quat(const FC& fc, const Quat<F>& yl, F sg, typename FlipCodeOf<F>::type* code = nullptr)
    -> decltype(yl.w < yl.w) {
  const Quat<F> y = qmul(fc.qE, yl);
  const F ax = y.x * y.x, ay = y.y * y.y, az = y.z * y.z;
  auto b1 = (ax > ay) && (ax > az);
  auto b2 = !b1 && ((ay > ax) && (ay > az));
  const F sx = sg * y.x, sy = sg * y.y, sz = sg * y.z;
  auto flip = sel_(b1, sx, sel_(b2, sy, sz)) < F(0);
  if (code) *code = flip_code_(flip, near_tie_(ax, ay, az, fma_(y.w, y.w, ax + ay + az)), sx < F(0), sy < F(0), sz < F(0));
  return flip;
}

// ------------------------------------------------------------------------------------------
// One fused filter step (Prediction + Correction, PKF/main_file.py:39,43), scalar Q and R.
// The covariance argument P is carried IN UNITS OF r (P/r): with R = r I the whole recursion is
// homogeneous in r --  P/r <- A (P/r) A^T + (q/4r)(|x|^2 I - x x^T),  K = (P/r)(P/r + I)^-1,
// P_post/r = K -- so the scaled form saves the r multiplications and makes the post-update
// covariance literally equal to the gain.  Callers convert at launch boundaries (r > 0 required).
// ------------------------------------------------------------------------------------------
// WAHBA_PRECOMPUTED: the measurement quaternion (reference sign convention) comes with the stream instead of
// acc/mag -- a (Q,R) sweep replays every trajectory thousands of times and its Wahba solution does not
// depend on Q or R, so it is solved once per trajectory and step (measurement_stream_kernel).
enum WahbaAlgo { WAHBA_QR2 = 0, WAHBA_JACOBI = 1, WAHBA_PRECOMPUTED = 2 };
constexpr int kJacobiSweepsFused = 4;

template <typename F> struct FilterConst {
  RefFrame<F> E;          // from (acc_0, mag_0)
  Vec3<F> ra, rm;         // raw reference vectors (used by the Jacobi variant only)
  F g;                    // Q/(4R): process noise in units of r
  F gs;                   // g |x|^2 of the CURRENT state: g after any step of the filter (it normalises), see adopt_state
  F g1, gs1;              // g + 1, gs + 1: the constant of S's diagonal (plain variant, see kalman_gain_from_s)
  Quat<F> qE;             // unit quaternion of the rotation [e1 e2 e3]: filter frame -> reference frame
};

PKF_HD void quat_fallback_unaligned(const Mat3<float>& Rm, const Quat<float>& z, bool, Quat<float>& y) {
  y = rotation_to_quat_ref(Rm);
  float sg = dot4(y, z) < 0.f ? -1.f : 1.f;
  y.w *= sg; y.x *= sg; y.y *= sg; y.z *= sg;
}
PKF_HD void quat_fallback_unaligned(const Mat3<double>& Rm, const Quat<double>& z, bool, Quat<double>& y) {
  y = rotation_to_quat_ref(Rm);
  double sg = dot4(y, z) < 0.0 ? -1.0 : 1.0;
  y.w *= sg; y.x *= sg; y.y *= sg; y.z *= sg;
}
PKF_HD void quat_fallback_unaligned(const Mat3<f32x2>& Rm, const Quat<f32x2>& z, mask2 which, Quat<f32x2>& y) {
  // rare path: redo the affected lane(s) with the scalar code
  for (int lane = 0; lane < 2; ++lane) {
    if (!(lane ? which.y : which.x)) continue;
    Mat3<float> R1;
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) R1.m[i][j] = lane ? Rm.m[i][j].y : Rm.m[i][j].x;
    Quat<float> z1 = {lane ? z.w.y : z.w.x, lane ? z.x.y : z.x.x, lane ? z.y.y : z.y.x, lane ? z.z.y : z.z.x}, y1;
    quat_fallback_unaligned(R1, z1, true, y1);
    if (lane) { y.w.y = y1.w; y.x.y = y1.x; y.y.y = y1.y; y.z.y = y1.z; }
    else { y.w.x = y1.w; y.x.x = y1.x; y.y.x = y1.y; y.z.x = y1.z; }
  }
}
// COMP selects the "precise" variant: (i) the Sherman-Morrison gain (kalman_gain_sm) that keeps the
// process noise apart from A K A^T, for Q >> R; (ii) the compensated state for R >> Q:
// X is carried as x + xlo (two floats per component).  With a
// single float, increments below half an ulp of the state (K e ~ 2e-8 per step when R >> Q) are
// absorbed by the addition and the filter silently stops following its measurement -- the float64
// reference does not (2.4e-5 rad apart after 5000 steps at Q=1e-3, R=1e3).  The compensated form
// sums the step's three small terms (RK4 increment, K e, norm correction) first and folds them into
// the state with one exact two-sum per component.
// ---- the three parts of a step -------------------------------------------------------------------
// Prediction (PKF/ExtendedKalmanFilter.py:58-68): gain K (= the post-update covariance in units of r), RK4
// increment inc and predicted state z = x + inc.
// INNOV: the gain stage also hands its factors of S~ to `fac` (innovation likelihood, see InnovFactors).
// GATE: the factors go to `fac` for the gate statistic as well, and the propagated covariance P^- (units of r) to *Pm.
template <typename F, bool COMP, bool INNOV = false, bool GATE = false>
PKF_HD void ekf_predict(const Quat<F>& x, const Sym4<F>& P, const FilterConst<F>& fc, const Vec3<F>& gyro, const StepH<F>& h,
                        Sym4<F>& K, Quat<F>& inc, Quat<F>& z, InnovFactors<F>* fac = nullptr, Sym4<F>* Pm = nullptr) {
  Vec3<F> hw;
  hw.x = F(0.5) * gyro.x; hw.y = F(0.5) * gyro.y; hw.z = F(0.5) * gyro.z;
  if constexpr (COMP) {
    Sym4<F> M = propagate_cov<F, false>(P, hw, x, fc.g, fc.gs);               // :59-61, noise kept apart
    K = kalman_gain_sm<F, INNOV || GATE, INNOV>(M, x, fc.gs, fac);            // :63-66
    if constexpr (GATE) {     // P^- = M + gs (|x|^2 I - x x^T), the diagonal formed as kalman_gain_sm forms H's
      const F x2 = dot4(x, x);
      const F yw = fc.gs * x.w, yx = fc.gs * x.x, yy = fc.gs * x.y, yz = fc.gs * x.z;
      Pm->a00 = fma_(-yw, x.w, fma_(fc.gs, x2, M.a00)); Pm->a11 = fma_(-yx, x.x, fma_(fc.gs, x2, M.a11));
      Pm->a22 = fma_(-yy, x.y, fma_(fc.gs, x2, M.a22)); Pm->a33 = fma_(-yz, x.z, fma_(fc.gs, x2, M.a33));
      Pm->a01 = fma_(-yw, x.x, M.a01); Pm->a02 = fma_(-yw, x.y, M.a02); Pm->a03 = fma_(-yw, x.z, M.a03);
      Pm->a12 = fma_(-yx, x.y, M.a12); Pm->a13 = fma_(-yx, x.z, M.a13); Pm->a23 = fma_(-yy, x.z, M.a23);
    }
  } else {
#if PKF_FUSE
    Sym4<F> S = propagate_cov<F, true>(P, hw, x, fc.g, fc.gs, fc.gs1);        // :59-61 and S = P + R :63 (in units of r)
    K = kalman_gain_from_s<F, INNOV || GATE, INNOV>(S, fac);                  // :64-66
    // GATE: P^- itself, its diagonal constant gs instead of gs + 1 (S - I would round P^-'s diagonal at ulp(1): 9 bits
    // of a 2.5e-3 entry); the off-diagonal entries are S's, shared with it
    if constexpr (GATE) *Pm = propagate_cov<F, true>(P, hw, x, fc.g, fc.gs, fc.gs);
    z = rk4_predict_fused(x, hw, h);                                          // :62
    inc = z;                                                                  // (unused by the plain update)
    return;
#else
    static_assert(!INNOV && !GATE, "the innovation statistic takes its factors from the fused plain gain (PKF_FUSE)");
    Sym4<F> Pp = propagate_cov<F, true>(P, hw, x, fc.g, fc.gs);               // :59-61 (in units of r)
    K = kalman_gain_unit(Pp);                                                 // :63-66
#endif
  }
  inc = rk4_increment(x, hw, h.h);                                            // :62
  z.w = x.w + inc.w; z.x = x.x + inc.x; z.y = x.y + inc.y; z.z = x.z + inc.z;   // |z| = 1 to rounding
}

// State and covariance update (PKF/ExtendedKalmanFilter.py:77-79) from the innovation e = y - z.
template <typename F, bool COMP>
PKF_HD void ekf_update(Quat<F>& x, Quat<F>& xlo, Sym4<F>& P, FilterConst<F>& fc, const Sym4<F>& K, const Quat<F>& z,
                       const Quat<F>& inc, F e0, F e1, F e2, F e3) {
  // X = z + K e                                                              :77
#if PKF_FUSE
  if (!COMP) {    // the sum is accumulated onto z by the FMAs themselves (no separate products, no final additions)
    Quat<F> xn;
#if PKF_FUSE >= 2
    // column by column: four consecutive FMAs share e_j in the same operand slot (register reuse cache)
    xn.w = fma_(K.a00, e0, z.w); xn.x = fma_(K.a01, e0, z.x); xn.y = fma_(K.a02, e0, z.y); xn.z = fma_(K.a03, e0, z.z);
    xn.w = fma_(K.a01, e1, xn.w); xn.x = fma_(K.a11, e1, xn.x); xn.y = fma_(K.a12, e1, xn.y); xn.z = fma_(K.a13, e1, xn.z);
    xn.w = fma_(K.a02, e2, xn.w); xn.x = fma_(K.a12, e2, xn.x); xn.y = fma_(K.a22, e2, xn.y); xn.z = fma_(K.a23, e2, xn.z);
    xn.w = fma_(K.a03, e3, xn.w); xn.x = fma_(K.a13, e3, xn.x); xn.y = fma_(K.a23, e3, xn.y); xn.z = fma_(K.a33, e3, xn.z);
#else
    xn.w = fma_(K.a03, e3, fma_(K.a02, e2, fma_(K.a01, e1, fma_(K.a00, e0, z.w))));
    xn.x = fma_(K.a13, e3, fma_(K.a12, e2, fma_(K.a11, e1, fma_(K.a01, e0, z.x))));
    xn.y = fma_(K.a23, e3, fma_(K.a22, e2, fma_(K.a12, e1, fma_(K.a02, e0, z.y))));
    xn.z = fma_(K.a33, e3, fma_(K.a23, e2, fma_(K.a13, e1, fma_(K.a03, e0, z.z))));
#endif
    F d = rsqrt_(dot4(xn, xn)) - F(1);
    x.w = fma_(xn.w, d, xn.w); x.x = fma_(xn.x, d, xn.x); x.y = fma_(xn.y, d, xn.y); x.z = fma_(xn.z, d, xn.z);
    P = K;
    fc.gs = fc.g;
    fc.gs1 = fc.g1;
    return;
  }
#endif
  Quat<F> ke;
  ke.w = fma_(K.a03, e3, fma_(K.a02, e2, fma_(K.a01, e1, K.a00 * e0)));
  ke.x = fma_(K.a13, e3, fma_(K.a12, e2, fma_(K.a11, e1, K.a01 * e0)));
  ke.y = fma_(K.a23, e3, fma_(K.a22, e2, fma_(K.a12, e1, K.a02 * e0)));
  ke.z = fma_(K.a33, e3, fma_(K.a23, e2, fma_(K.a13, e1, K.a03 * e0)));
  // X / |X| is applied as X + X (1/|X| - 1): when the norm is already 1 to rounding the correction
  // is below half an ulp, so normalising every step does not re-round the state              :79
  if (!COMP) {
    Quat<F> xn;
    xn.w = z.w + ke.w; xn.x = z.x + ke.x; xn.y = z.y + ke.y; xn.z = z.z + ke.z;
    F d = rsqrt_(dot4(xn, xn)) - F(1);
    x.w = fma_(xn.w, d, xn.w); x.x = fma_(xn.x, d, xn.x); x.y = fma_(xn.y, d, xn.y); x.z = fma_(xn.z, d, xn.z);
  } else {
    Quat<F> dl, xn;     // all small terms first, then one exact fold into (x, xlo)
    dl.w = (inc.w + xlo.w) + ke.w; dl.x = (inc.x + xlo.x) + ke.x; dl.y = (inc.y + xlo.y) + ke.y; dl.z = (inc.z + xlo.z) + ke.z;
    xn.w = x.w + dl.w; xn.x = x.x + dl.x; xn.y = x.y + dl.y; xn.z = x.z + dl.z;
    F d = rsqrt_(dot4(xn, xn)) - F(1);
    dl.w = fma_(xn.w, d, dl.w); dl.x = fma_(xn.x, d, dl.x); dl.y = fma_(xn.y, d, dl.y); dl.z = fma_(xn.z, d, dl.z);
    two_sum(x.w, dl.w, x.w, xlo.w); two_sum(x.x, dl.x, x.x, xlo.x);
    two_sum(x.y, dl.y, x.y, xlo.y); two_sum(x.z, dl.z, x.z, xlo.z);
  }
  // P = P - K P = r K  (R = r I): in units of r the new covariance IS the gain     :78
  P = K;
  fc.gs = fc.g;        // the state leaves every step normalised: |x|^2 = 1 for the next step's B Q B^T
  fc.gs1 = fc.g1;
}

// The measurement of one sample: getQuarternion(acc, mag, |a_z|, 1 - |a_z|) (PKF/ExtendedKalmanFilter.py:71) as a
// quaternion in the filter frame, sign arbitrary, un-normalised, with 1/|y| in inv_norm.  It depends on the sample
// and the filter's reference frame only -- not on the state.
template <typename F>
PKF_HD Quat<F> measure_quat(const FilterConst<F>& fc, const Vec3<F>& acc, const Vec3<F>& mag, F& inv_norm) {
  const F ka = abs_(acc.z), km = F(1) - ka;
  Quat<F> y = wahba_quat2_local(fc.E, acc, mag, ka, km, inv_norm);
  const auto reflected = km < F(0);      // |a_z| > 1 (un-normalised accelerometer): a negative weight, the closed
  if (any_(reflected)) {                 // form does not apply -- rank-2 SVD form for those lanes (rare path)
    const Quat<F> yr = rotation_to_quat_best(wahba_qr2_local(fc.E, acc, mag, ka, km));
    y.w = sel_(reflected, yr.w, y.w); y.x = sel_(reflected, yr.x, y.x);
    y.y = sel_(reflected, yr.y, y.y); y.z = sel_(reflected, yr.z, y.z);
    inv_norm = sel_(reflected, F(1), inv_norm);
  }
  return y;
}

// GATE (see GateParams): the step's gate decision goes to *gated; a gated lane keeps its prediction and P^-.
template <typename F, bool COMP, typename FlagT>
PKF_HD void gate_apply(const GateParams<F>& gp, const InnovFactors<F>& fac, const Quat<F>& z, const Sym4<F>& Pm, Sym4<F>& K,
                       F& e0, F& e1, F& e2, F& e3, FlagT& gated) {
  const auto g = tangent_nis_r<F, COMP>(fac, z, e0, e1, e2, e3) > gp.thr;
  gated = g;
  e0 = sel_(g, F(0), e0); e1 = sel_(g, F(0), e1); e2 = sel_(g, F(0), e2); e3 = sel_(g, F(0), e3);
  K.a00 = sel_(g, Pm.a00, K.a00); K.a01 = sel_(g, Pm.a01, K.a01); K.a02 = sel_(g, Pm.a02, K.a02); K.a03 = sel_(g, Pm.a03, K.a03);
  K.a11 = sel_(g, Pm.a11, K.a11); K.a12 = sel_(g, Pm.a12, K.a12); K.a13 = sel_(g, Pm.a13, K.a13);
  K.a22 = sel_(g, Pm.a22, K.a22); K.a23 = sel_(g, Pm.a23, K.a23); K.a33 = sel_(g, Pm.a33, K.a33);
}

// ------------------------------------------------------------------------------------------
// GENERAL Q AND R (GEN): Q any symmetric positive semidefinite 3x3, R any symmetric positive definite 4x4 -- the
// reference's KalmanFilter with its Q and R attributes assigned (PKF/ExtendedKalmanFilter.py:58-79).  Neither the
// closed form of B Q B^T nor the units-of-r scaling applies, so P is carried unscaled (plain variant only).
//   B(x) Q B(x)^T: B(x) v = (0, v) (x) x / 2 is linear in x.  With Q4 = Q/4 and 2B (entries +-x_i),
//     M = (2B) Q4 (4x3),   P^-_ij = (A P A^T)_ij + sum_c M_ic (2B)_jc          (propagate_cov_general)
//   and the first step of a launch handed a non-unit state gets |x|^2 B(x^) Q B(x^)^T through fc.gs (fc.g = 1, see
//   adopt_state), so the second factor is formed from gs x.
//   Gain: S = P^- + R = L D L^T (kalman_gain_general).  K = P^- S^-1 = I - R S^-1, and with G = L^-1 R, H = D^-1 G:
//     K e = e - H^T (L^-1 e),     P^+ = P^- - K P^- = K R = R - R S^-1 R = R - G^T H
//   (upper triangle only, symmetric by construction; no backward substitution).  For R = r I this is the isotropic
//   step's own algebra (K = I - r S^-1, P^+ = r K), so it loses accuracy where that one does (see kalman_gain_from_s).
//   Filter frame: with x' = p (x) x, L(p) B(x) v = B(x') Rot(p) v, so the recursion stays equivariant when Q and R are
//   carried as Rot(p) Q Rot(p)^T and L(p) R L(p)^T (make_gen_qr).
// ------------------------------------------------------------------------------------------
template <typename F> struct Sym3 { F a00, a01, a02, a11, a12, a22; };      // upper triangle, row-major
template <typename F> struct GenQR {
  Sym3<F> q4;     // Q/4 in the step's frame
  Sym4<F> R;      // R in the step's frame
};
template <typename F> struct GainGen {
  Sym4<F> Pp;                          // P^+
  F l10, l20, l30, l21, l31, l32;      // L of S = L D L^T
  F h[4][4];                           // H = D^-1 L^-1 R
};
struct NoGainGen {};
template <typename F, bool GEN> struct GainGenOf { typedef GainGen<F> type; };   // (empty in the other instantiations)
template <typename F> struct GainGenOf<F, false> { typedef NoGainGen type; };
// GEN with INNOV or GATE: the pivots d_k of S = L D L^T (the innovation terms) and, gated only, P^- (see GEN INNOVATION
// below).  Empty in every other instantiation, like GainGen: declared state that a kernel does not use still moves the
// code of the others.
template <typename F> struct GenInnov {
  F d0, d1, d2, d3;   // pivots
  F i0, i1, i2, i3;   // 1/d_k, as the gain uses them
  Sym4<F> Pm;         // GATE only
};
template <typename F, bool ON> struct GenInnovOf { typedef GenInnov<F> type; };
template <typename F> struct GenInnovOf<F, false> { typedef NoGainGen type; };

// q [6], r [10]: the upper triangles of Q and R in the reference frame (row-major, the order of Sym4).  filter_frame:
// express them in the filter frame of fc (p = conj(qE), Rot(p) = E^T).
template <typename F>
PKF_HD GenQR<F> make_gen_qr(const FilterConst<F>& fc, const F (&q)[6], const F (&r)[10], bool filter_frame) {
  F Q[3][3] = {{q[0], q[1], q[2]}, {q[1], q[3], q[4]}, {q[2], q[4], q[5]}};
  Sym4<F> R = {r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[7], r[8], r[9]};
  if (filter_frame) {
    const F e[3][3] = {{fc.E.e1.x, fc.E.e1.y, fc.E.e1.z}, {fc.E.e2.x, fc.E.e2.y, fc.E.e2.z}, {fc.E.e3.x, fc.E.e3.y, fc.E.e3.z}};
    F QE[3][3], Qf[3][3];     // Q e_j, then e_i^T Q e_j
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) QE[i][j] = fma_(Q[i][2], e[j][2], fma_(Q[i][1], e[j][1], Q[i][0] * e[j][0]));
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) Qf[i][j] = fma_(e[i][2], QE[2][j], fma_(e[i][1], QE[1][j], e[i][0] * QE[0][j]));
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) Q[i][j] = Qf[i][j];
    R = rotate_cov(qconj(fc.qE), R);
  }
  GenQR<F> g;
  g.q4 = {F(0.25) * Q[0][0], F(0.25) * Q[0][1], F(0.25) * Q[0][2], F(0.25) * Q[1][1], F(0.25) * Q[1][2], F(0.25) * Q[2][2]};
  g.R = R;
  return g;
}

// P^- = A P A^T + B(x) Q B(x)^T, Q = 4 q4; s = |x|^2 of the state handed to the launch on its first step, else 1.
template <typename F>
PKF_HD Sym4<F> propagate_cov_general(const Sym4<F>& P, const Vec3<F>& hw, const Quat<F>& x, F s, const Sym3<F>& q4) {
  Sym4<F> N = propagate_cov<F, false>(P, hw, x, F(0), F(0));
  const F Q[3][3] = {{q4.a00, q4.a01, q4.a02}, {q4.a01, q4.a11, q4.a12}, {q4.a02, q4.a12, q4.a22}};
  // rows of 2B(x): column c is (0, e_c) (x) x
  const F b[4][3] = {{-x.x, -x.y, -x.z}, {x.w, x.z, -x.y}, {-x.z, x.w, x.x}, {x.y, -x.x, x.w}};
  const Quat<F> y = {s * x.w, s * x.x, s * x.y, s * x.z};
  const F bs[4][3] = {{-y.x, -y.y, -y.z}, {y.w, y.z, -y.y}, {-y.z, y.w, y.x}, {y.y, -y.x, y.w}};
  F M[4][3];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int i = 0; i < 4; ++i) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int c = 0; c < 3; ++c) M[i][c] = fma_(b[i][2], Q[2][c], fma_(b[i][1], Q[1][c], b[i][0] * Q[0][c]));
  }
  auto add = [&](F n, int i, int j) { return fma_(M[i][2], bs[j][2], fma_(M[i][1], bs[j][1], fma_(M[i][0], bs[j][0], n))); };
  N.a00 = add(N.a00, 0, 0); N.a01 = add(N.a01, 0, 1); N.a02 = add(N.a02, 0, 2); N.a03 = add(N.a03, 0, 3);
  N.a11 = add(N.a11, 1, 1); N.a12 = add(N.a12, 1, 2); N.a13 = add(N.a13, 1, 3);
  N.a22 = add(N.a22, 2, 2); N.a23 = add(N.a23, 2, 3);
  N.a33 = add(N.a33, 3, 3);
  return N;
}

// S = P^- + R = L D L^T, H = D^-1 L^-1 R and P^+ = R - (L^-1 R)^T H (see GENERAL Q AND R above).
// PIV: the pivots d_k also go to *gi.
template <typename F, bool PIV = false>
PKF_HD GainGen<F> kalman_gain_general(const Sym4<F>& Pm, const Sym4<F>& R, GenInnov<F>* gi = nullptr) {
  const F s00 = Pm.a00 + R.a00, s01 = Pm.a01 + R.a01, s02 = Pm.a02 + R.a02, s03 = Pm.a03 + R.a03;
  const F s11 = Pm.a11 + R.a11, s12 = Pm.a12 + R.a12, s13 = Pm.a13 + R.a13;
  const F s22 = Pm.a22 + R.a22, s23 = Pm.a23 + R.a23, s33 = Pm.a33 + R.a33;
  GainGen<F> g;
  const F i0 = rcp_(s00);
  g.l10 = s01 * i0; g.l20 = s02 * i0; g.l30 = s03 * i0;
  const F d1 = fma_(-g.l10, s01, s11);
  const F i1 = rcp_(d1);
  const F t21 = fma_(-g.l10, s02, s12), t31 = fma_(-g.l10, s03, s13);
  g.l21 = t21 * i1; g.l31 = t31 * i1;
  const F d2 = fma_(-g.l21, t21, fma_(-g.l20, s02, s22));
  const F i2 = rcp_(d2);
  const F t32 = fma_(-g.l21, t31, fma_(-g.l20, s03, s23));
  g.l32 = t32 * i2;
  const F d3 = fma_(-g.l32, t32, fma_(-g.l31, t31, fma_(-g.l30, s03, s33)));
  const F i3 = rcp_(d3);
  if constexpr (PIV) {
    gi->d0 = s00; gi->d1 = d1; gi->d2 = d2; gi->d3 = d3;
    gi->i0 = i0; gi->i1 = i1; gi->i2 = i2; gi->i3 = i3;
  }
  const F Rm[4][4] = {{R.a00, R.a01, R.a02, R.a03}, {R.a01, R.a11, R.a12, R.a13}, {R.a02, R.a12, R.a22, R.a23},
                      {R.a03, R.a13, R.a23, R.a33}};
  F G[4][4];      // L^-1 R, column by column
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int j = 0; j < 4; ++j) {
    G[0][j] = Rm[0][j];
    G[1][j] = fma_(-g.l10, G[0][j], Rm[1][j]);
    G[2][j] = fma_(-g.l21, G[1][j], fma_(-g.l20, G[0][j], Rm[2][j]));
    G[3][j] = fma_(-g.l32, G[2][j], fma_(-g.l31, G[1][j], fma_(-g.l30, G[0][j], Rm[3][j])));
    g.h[0][j] = i0 * G[0][j]; g.h[1][j] = i1 * G[1][j]; g.h[2][j] = i2 * G[2][j]; g.h[3][j] = i3 * G[3][j];
  }
  auto pp = [&](int i, int j) {
    return fma_(-G[3][i], g.h[3][j], fma_(-G[2][i], g.h[2][j], fma_(-G[1][i], g.h[1][j], fma_(-G[0][i], g.h[0][j], Rm[i][j]))));
  };
  g.Pp = {pp(0, 0), pp(0, 1), pp(0, 2), pp(0, 3), pp(1, 1), pp(1, 2), pp(1, 3), pp(2, 2), pp(2, 3), pp(3, 3)};
  return g;
}

// Prediction with general Q and R: the gain stage and the RK4 prediction z (plain-variant form).
// PIV: the pivots of S go to *gi (INNOV / GATE); PM: P^- too (GATE).
template <typename F, bool PIV = false, bool PM = false>
PKF_HD void ekf_predict_general(const Quat<F>& x, const Sym4<F>& P, const FilterConst<F>& fc, const GenQR<F>& gq,
                                const Vec3<F>& gyro, const StepH<F>& h, GainGen<F>& gg, Quat<F>& z,
                                GenInnov<F>* gi = nullptr) {
  Vec3<F> hw;
  hw.x = F(0.5) * gyro.x; hw.y = F(0.5) * gyro.y; hw.z = F(0.5) * gyro.z;
  if constexpr (PIV) {
    const Sym4<F> Pm = propagate_cov_general(P, hw, x, fc.gs, gq.q4);                  // :59-61
    if constexpr (PM) gi->Pm = Pm;
    gg = kalman_gain_general<F, true>(Pm, gq.R, gi);                                     // :63-66
  } else {
    gg = kalman_gain_general(propagate_cov_general(P, hw, x, fc.gs, gq.q4), gq.R);     // :59-66
  }
  z = rk4_predict_fused(x, hw, h);                                                       // :62
}

// ------------------------------------------------------------------------------------------
// GEN INNOVATION: the innovation terms and the gate of a filter with general Q and R, in true units (the covariance is
// not scaled: no 1/r, no dof ln r).  S = P^- + R = L D L^T is already factored by the gain stage, and t = L^-1 e is the
// quantity the update forms; S^-1 itself is never formed.
//   4-D:      NIS = e^T S^-1 e = s = sum_k t_k^2 / d_k,      ln det S = sum_k ln d_k
//   tangent:  v = L^-1 z,  c = z^T S^-1 z = sum_k v_k^2 / d_k,  b = z^T S^-1 e = sum_k v_k t_k / d_k;  for any orthonormal
//             basis E of z-perp, e_3 = E^T e and S_3 = E^T S E,
//               NIS_3 = e_3^T S_3^-1 e_3 = s - b^2/c                          (Schur complement of u = z/|z|)
//               ln det S_3 = ln det S + ln(c/|z|^2)                           (det(E^T S E) = det S . u^T S^-1 u)
// The log-determinant is summed from the logs of two pivot products, never the log of the product of four: pivots in
// [1e-18, 1e18] then neither underflow nor overflow.  The sums add each step's terms as they are written out (one
// addition each), so a sum is exactly the float32 running sum of its per-step terms.
// Gate: gated <=> NIS_3 > gamma (strict: NaN is never gated).  A gated lane zeroes its innovation (X = z, normalised) and
// keeps P^-, selected per lane.
// ------------------------------------------------------------------------------------------
template <typename F, bool TAN>
PKF_HD void gen_innov_terms(const GainGen<F>& gg, const GenInnov<F>& gi, const Quat<F>& z, F e0, F e1, F e2, F e3,
                            F& nis, F& logdet) {
  const F t0 = e0;                                 // t = L^-1 e (the update's)
  const F t1 = fma_(-gg.l10, t0, e1);
  const F t2 = fma_(-gg.l21, t1, fma_(-gg.l20, t0, e2));
  const F t3 = fma_(-gg.l32, t2, fma_(-gg.l31, t1, fma_(-gg.l30, t0, e3)));
  const F u0 = gi.i0 * t0, u1 = gi.i1 * t1, u2 = gi.i2 * t2, u3 = gi.i3 * t3;
  const F s = fma_(u3, t3, fma_(u2, t2, fma_(u1, t1, u0 * t0)));
  const F ld = log_(gi.d0 * gi.d1) + log_(gi.d2 * gi.d3);
  if constexpr (!TAN) {
    nis = s;
    logdet = ld;
  } else {
    const F v0 = z.w;                                // v = L^-1 z
    const F v1 = fma_(-gg.l10, v0, z.x);
    const F v2 = fma_(-gg.l21, v1, fma_(-gg.l20, v0, z.y));
    const F v3 = fma_(-gg.l32, v2, fma_(-gg.l31, v1, fma_(-gg.l30, v0, z.z)));
    const F g0 = gi.i0 * v0, g1 = gi.i1 * v1, g2 = gi.i2 * v2, g3 = gi.i3 * v3;
    const F c = fma_(g3, v3, fma_(g2, v2, fma_(g1, v1, g0 * v0)));
    const F b = fma_(g3, t3, fma_(g2, t2, fma_(g1, t1, g0 * t0)));
    nis = fma_(-b, b * rcp_(c), s);
    logdet = ld + log_(c * rcp_(dot4(z, z)));
  }
}

// INNOV: the step's terms are added to *acc (acc.inv_r / acc.log_rd unused) and handed to *step when it is set
template <typename F, bool TAN>
PKF_HD void gen_innov_accumulate(InnovAcc<F>& acc, const GainGen<F>& gg, const GenInnov<F>& gi, const Quat<F>& z, F e0,
                                 F e1, F e2, F e3, InnovTerms<F>* step = nullptr) {
  F nis, ld;
  gen_innov_terms<F, TAN>(gg, gi, z, e0, e1, e2, e3, nis, ld);
  acc.nis = acc.nis + nis;
  acc.logdet = acc.logdet + ld;
  if (step) { step->nis = nis; step->logdet = ld; }
}

// GATE: the decision on NIS_3 (the same value as the tangent term), applied per lane to e and P^+
template <typename F, typename FlagT>
PKF_HD void gen_gate_apply(const GateParams<F>& gp, GainGen<F>& gg, const GenInnov<F>& gi, const Quat<F>& z, F& e0, F& e1,
                           F& e2, F& e3, FlagT& gated) {
  F nis3, ld;
  gen_innov_terms<F, true>(gg, gi, z, e0, e1, e2, e3, nis3, ld);
  const auto g = nis3 > gp.thr;
  gated = g;
  e0 = sel_(g, F(0), e0); e1 = sel_(g, F(0), e1); e2 = sel_(g, F(0), e2); e3 = sel_(g, F(0), e3);
  Sym4<F>& P = gg.Pp;
  const Sym4<F>& Pm = gi.Pm;
  P.a00 = sel_(g, Pm.a00, P.a00); P.a01 = sel_(g, Pm.a01, P.a01); P.a02 = sel_(g, Pm.a02, P.a02); P.a03 = sel_(g, Pm.a03, P.a03);
  P.a11 = sel_(g, Pm.a11, P.a11); P.a12 = sel_(g, Pm.a12, P.a12); P.a13 = sel_(g, Pm.a13, P.a13);
  P.a22 = sel_(g, Pm.a22, P.a22); P.a23 = sel_(g, Pm.a23, P.a23); P.a33 = sel_(g, Pm.a33, P.a33);
}

// X = z + K e, normalised; P = P^+                                                         :77-79
template <typename F>
PKF_HD void ekf_update_general(Quat<F>& x, Sym4<F>& P, FilterConst<F>& fc, const GainGen<F>& gg, const Quat<F>& z,
                               F e0, F e1, F e2, F e3) {
  const F t0 = e0;                                 // t = L^-1 e
  const F t1 = fma_(-gg.l10, t0, e1);
  const F t2 = fma_(-gg.l21, t1, fma_(-gg.l20, t0, e2));
  const F t3 = fma_(-gg.l32, t2, fma_(-gg.l31, t1, fma_(-gg.l30, t0, e3)));
  auto ke = [&](int i, F ei) { return fma_(-gg.h[3][i], t3, fma_(-gg.h[2][i], t2, fma_(-gg.h[1][i], t1, fma_(-gg.h[0][i], t0, ei)))); };
  Quat<F> xn;
  xn.w = z.w + ke(0, e0); xn.x = z.x + ke(1, e1); xn.y = z.y + ke(2, e2); xn.z = z.z + ke(3, e3);
  const F d = rsqrt_(dot4(xn, xn)) - F(1);
  x.w = fma_(xn.w, d, xn.w); x.x = fma_(xn.x, d, xn.x); x.y = fma_(xn.y, d, xn.y); x.z = fma_(xn.z, d, xn.z);
  P = gg.Pp;
  fc.gs = fc.g;        // the state leaves every step normalised
}

// Prediction + Correction with the measurement quaternion y (filter frame, any sign, norm 1/inv_norm) already computed.
// INNOV: the innovation likelihood of the step is added to *innov (see InnovAcc); the filter itself is unchanged.
// TAN: its tangent-space form (see innov_accumulate).  GATE: the innovation gate (see GateParams), decision in *gated.
// GEN: general Q and R from *gen (see GENERAL Q AND R); P is unscaled, plain variant only.  With INNOV / GATE: the terms
// and the gate of GEN INNOVATION.
// terms (INNOV): the step's own innovation terms (see InnovTerms), or null.
template <typename F, bool WANT_FLIP, bool COMP, bool INNOV = false, bool TAN = false, bool GATE = false, bool GEN = false,
          typename FlagT>
PKF_HD void ekf_step_measured(Quat<F>& x, Quat<F>& xlo, Sym4<F>& P, FilterConst<F>& fc, const Vec3<F>& gyro,
                              const Quat<F>& y, F inv_norm, const StepH<F>& h, FlagT& flip, bool flip_wanted = true,
                              typename FlipCodeOf<F>::type* code = nullptr, InnovAcc<F>* innov = nullptr,
                              const GateParams<F>* gate = nullptr, FlagT* gated = nullptr, const GenQR<F>* gen = nullptr,
                              InnovTerms<F>* terms = nullptr) {
  static_assert(!GEN || !COMP, "general Q and R: plain variant only");
  Sym4<F> K, Pm;
  Quat<F> inc, z;
  InnovFactors<F> fac;
  [[maybe_unused]] typename GainGenOf<F, GEN>::type gg;
  [[maybe_unused]] typename GenInnovOf<F, GEN && (INNOV || GATE)>::type gi;
  if constexpr (GEN && (INNOV || GATE)) ekf_predict_general<F, true, GATE>(x, P, fc, *gen, gyro, h, gg, z, &gi);
  else if constexpr (GEN) ekf_predict_general(x, P, fc, *gen, gyro, h, gg, z);
  else ekf_predict<F, COMP, INNOV, GATE>(x, P, fc, gyro, h, K, inc, z, &fac, &Pm);
  const F dyz = dot4(y, z);                       // the comparator, literally: negate when dot(y, z) < 0  :73-75
  flip = FlagT();
  if (WANT_FLIP && flip_wanted) flip = reference_flip_quat(fc, y, one_with_sign_(dyz), code);
  const F sn = copysign_(inv_norm, dyz);          // e = sg y/|y| - z, sg = sign(dot): the sign bit moves onto 1/|y| > 0  :76
  F e0 = fma_(sn, y.w, -z.w), e1 = fma_(sn, y.x, -z.x), e2 = fma_(sn, y.y, -z.y), e3 = fma_(sn, y.z, -z.z);
  if constexpr (GEN) {
    if constexpr (INNOV) gen_innov_accumulate<F, TAN>(*innov, gg, gi, z, e0, e1, e2, e3, terms);
    if constexpr (GATE) gen_gate_apply(*gate, gg, gi, z, e0, e1, e2, e3, *gated);
  } else {
    if constexpr (INNOV) innov_accumulate<F, COMP, TAN>(*innov, fac, K, z, e0, e1, e2, e3, terms);
    if constexpr (GATE) gate_apply<F, COMP>(*gate, fac, z, Pm, K, e0, e1, e2, e3, *gated);
  }
  if constexpr (GEN) ekf_update_general(x, P, fc, gg, z, e0, e1, e2, e3);
  else ekf_update<F, COMP>(x, xlo, P, fc, K, z, inc, e0, e1, e2, e3);
}

// The common case of ekf_step<WAHBA_QR2>: both Wahba weights are non-negative (|a_z| <= 1, i.e. a normalised
// accelerometer), so the closed-form measurement applies and the step has no data-dependent branch.  The caller
// guarantees the precondition (the packed kernel checks a whole tile of samples before taking this path).
template <typename F, bool WANT_FLIP, bool COMP, bool INNOV = false, bool TAN = false, bool GATE = false, typename FlagT>
PKF_HD void ekf_step_plain_measured(Quat<F>& x, Quat<F>& xlo, Sym4<F>& P, FilterConst<F>& fc, const Vec3<F>& gyro,
                                    const Vec3<F>& acc, const Vec3<F>& mag, const StepH<F>& h, FlagT& flip, bool flip_wanted = true,
                                    typename FlipCodeOf<F>::type* code = nullptr, InnovAcc<F>* innov = nullptr,
                                    const GateParams<F>* gate = nullptr, FlagT* gated = nullptr) {
  const F ka = abs_(acc.z), km = F(1) - ka;
  F inv_norm;
  const Quat<F> y = wahba_quat2_local(fc.E, acc, mag, ka, km, inv_norm);
  ekf_step_measured<F, WANT_FLIP, COMP, INNOV, TAN, GATE>(x, xlo, P, fc, gyro, y, inv_norm, h, flip, flip_wanted, code, innov,
                                                          gate, gated);
}

template <typename F, int ALGO, bool WANT_FLIP, bool COMP, bool INNOV = false, bool TAN = false, bool GATE = false,
          bool GEN = false, typename FlagT>
PKF_HD void ekf_step(Quat<F>& x, Quat<F>& xlo, Sym4<F>& P, FilterConst<F>& fc, const Vec3<F>& gyro,
                     const Vec3<F>& acc, const Vec3<F>& mag, const StepH<F>& h, FlagT& flip, bool flip_wanted = true,
                     typename FlipCodeOf<F>::type* code = nullptr, InnovAcc<F>* innov = nullptr,
                     const GateParams<F>* gate = nullptr, FlagT* gated = nullptr, const GenQR<F>* gen = nullptr,
                     InnovTerms<F>* terms = nullptr) {
  // flip_wanted: launch-uniform run-time switch under WANT_FLIP -- a launch that stores the trajectory but
  // not the flip mask skips the reference's branch rule altogether
  if constexpr (ALGO == WAHBA_QR2) {
    F inv_norm;
    const Quat<F> y = measure_quat(fc, acc, mag, inv_norm);
    ekf_step_measured<F, WANT_FLIP, COMP, INNOV, TAN, GATE, GEN>(x, xlo, P, fc, gyro, y, inv_norm, h, flip, flip_wanted, code,
                                                                 innov, gate, gated, gen, terms);
  } else {
    static_assert(!GEN || !COMP, "general Q and R: plain variant only");
    Sym4<F> K, Pm;
    Quat<F> inc, z;
    InnovFactors<F> fac;
    [[maybe_unused]] typename GainGenOf<F, GEN>::type gg;
    [[maybe_unused]] typename GenInnovOf<F, GEN && (INNOV || GATE)>::type gi;
    if constexpr (GEN && (INNOV || GATE)) ekf_predict_general<F, true, GATE>(x, P, fc, *gen, gyro, h, gg, z, &gi);
    else if constexpr (GEN) ekf_predict_general(x, P, fc, *gen, gyro, h, gg, z);
    else ekf_predict<F, COMP, INNOV, GATE>(x, P, fc, gyro, h, K, inc, z, &fac, &Pm);
    // ---- Correction (PKF/ExtendedKalmanFilter.py:70-80) ----
    F e0, e1, e2, e3;
    if constexpr (ALGO == WAHBA_PRECOMPUTED) {
      // stream rows 3..6 carry the Wahba quaternion in the reference's own sign convention (the output of
      // getQuarternion, :71): apply the comparator literally -- negate when dot(y, z) < 0            :73-75
      const Quat<F> y = {acc.x, acc.y, acc.z, mag.x};
      const auto neg = dot4(y, z) < F(0);
      flip = neg;
      const F sg = sel_(neg, F(-1), F(1));
      e0 = fma_(sg, y.w, -z.w); e1 = fma_(sg, y.x, -z.x); e2 = fma_(sg, y.y, -z.y); e3 = fma_(sg, y.z, -z.z);   // :76
    } else {
      F ka = abs_(acc.z), km = F(1) - ka;                                       // :71
      // Rm: the Wahba rotation in the filter frame (E^T R)
      Mat3<F> Rm = frame_transposed_times(fc.E, wahba_jacobi(fc.ra, fc.rm, acc, mag, ka, km, kJacobiSweepsFused));
      // measurement quaternion with the comparator's sign already applied          :73-75
      F n2;
      Quat<F> y = rotation_to_quat_aligned(Rm, z, n2);     // un-normalised: 4 (y.z) y
      flip = FlagT();
      if (WANT_FLIP && flip_wanted) flip = reference_flip_local(fc, Rm, y);   // only the signs of y matter
      // innovation e = y/|y| - z, the normalisation folded into the subtraction     :76
      const F inv = rsqrt_(n2);
      e0 = fma_(y.w, inv, -z.w); e1 = fma_(y.x, inv, -z.x); e2 = fma_(y.y, inv, -z.y); e3 = fma_(y.z, inv, -z.z);
      const auto unrelated = n2 < F(0.16);
      if (any_(unrelated)) {
        // |y.z| < 0.1: prediction and measurement are unrelated (never in a tracking filter; can happen
        // on the first sample of a badly initialised one).  Use the selection-based conversion there.
        Quat<F> yf = y;
        quat_fallback_unaligned(Rm, z, unrelated, yf);
        if (WANT_FLIP && flip_wanted) flip = reference_flip_local(fc, Rm, yf);
        e0 = sel_(unrelated, yf.w - z.w, e0); e1 = sel_(unrelated, yf.x - z.x, e1);
        e2 = sel_(unrelated, yf.y - z.y, e2); e3 = sel_(unrelated, yf.z - z.z, e3);
      }
    }
    if constexpr (GEN) {
      if constexpr (INNOV) gen_innov_accumulate<F, TAN>(*innov, gg, gi, z, e0, e1, e2, e3, terms);
      if constexpr (GATE) gen_gate_apply(*gate, gg, gi, z, e0, e1, e2, e3, *gated);
    } else {
      if constexpr (INNOV) innov_accumulate<F, COMP, TAN>(*innov, fac, K, z, e0, e1, e2, e3, terms);
      if constexpr (GATE) gate_apply<F, COMP>(*gate, fac, z, Pm, K, e0, e1, e2, e3, *gated);
    }
    if constexpr (GEN) ekf_update_general(x, P, fc, gg, z, e0, e1, e2, e3);
    else ekf_update<F, COMP>(x, xlo, P, fc, K, z, inc, e0, e1, e2, e3);
  }
}

// A state handed to a launch.  The reference normalises at the end of every step (and the predicted state right
// after RK4, PKF/ExtendedKalmanFilter.py:40), so the only place a non-unit |x| ever acts is the process noise of the
// FIRST step, B(x) Q B(x)^T = (q/4)|x|^2 (I - x^ x^T); RK4 is linear, so everything else sees x^ = x/|x|.  The
// launch therefore normalises the incoming state once and carries g|x|^2 as the noise scale of its first step
// (fc.gs; every later step has g).  A state within 1e-5 of unit norm -- the initial [1,0,0,0], or anything this
// filter produced -- is taken as is, so that a replay cut into chunks stays bit-identical to the unchunked one.
template <typename F> PKF_HD void adopt_state(FilterConst<F>& fc, Quat<F>& x, Quat<F>& xlo) {
  const F n2 = dot4(x, x);
  const auto unit = abs_(n2 - F(1)) < F(1e-5);
  fc.gs = sel_(unit, fc.g, fc.g * n2);
  fc.gs1 = fc.gs + F(1);
  const F sc = sel_(unit, F(1), rsqrt_(n2));
  x.w *= sc; x.x *= sc; x.y *= sc; x.z *= sc;
  xlo.w *= sc; xlo.x *= sc; xlo.y *= sc; xlo.z *= sc;
}

template <typename F>
PKF_HD FilterConst<F> make_filter_const(const Vec3<F>& acc_ref, const Vec3<F>& mag_ref, F q, F r) {
  FilterConst<F> fc;
  fc.E = frame_from_pair(acc_ref, mag_ref);
  fc.ra = acc_ref; fc.rm = mag_ref;
  fc.g = (F(0.25) * q) / r;
  fc.gs = fc.g;
  fc.g1 = fc.g + F(1); fc.gs1 = fc.g1;
  Mat3<F> Em;
  Em.m[0][0] = fc.E.e1.x; Em.m[1][0] = fc.E.e1.y; Em.m[2][0] = fc.E.e1.z;
  Em.m[0][1] = fc.E.e2.x; Em.m[1][1] = fc.E.e2.y; Em.m[2][1] = fc.E.e2.z;
  Em.m[0][2] = fc.E.e3.x; Em.m[1][2] = fc.E.e3.y; Em.m[2][2] = fc.E.e3.z;
  fc.qE = rotation_to_quat_best(Em);
  return fc;
}

// ------------------------------------------------------------------------------------------
// FILTER FRAME.  The whole recursion is equivariant under a fixed left rotation of the state: with
// x' = p (x) x and P' = L(p) P L(p)^T (L orthogonal), RK4 (a right multiplication) commutes with L(p),
// B Q B^T = (q/4)(|x|^2 I - x x^T) and R = r I transform covariantly, the gain is a spectral function of
// P, and the comparator's dot product is invariant.  The fused step therefore runs in the coordinates of
// the reference frame E = [e1 e2 e3] built from (acc_0, mag_0), p = conj(qE): there the Wahba rotation
// is blockdiag(G, det G) F^T (wahba_qr2_local) and the 27 multiply-adds of E * (...) per step disappear.
// State enters and leaves the frame once per launch (or not at all when the caller keeps it there between
// launches, see POSEKF_STATE_*_FILTER_FRAME); outputs per step (trajectory, flip mask, loss) are mapped back.
// WAHBA_PRECOMPUTED launches have no Wahba stage: their filter frame IS the reference frame.
// ------------------------------------------------------------------------------------------
template <int ALGO> PKF_HD constexpr bool uses_filter_frame() { return ALGO != WAHBA_PRECOMPUTED; }

template <typename F>
PKF_HD void enter_filter_frame(const FilterConst<F>& fc, Quat<F>& x, Quat<F>& xlo, Sym4<F>& P, bool comp) {
  const Quat<F> p = qconj(fc.qE);
  x = qmul(p, x);
  if (comp) xlo = qmul(p, xlo);
  P = rotate_cov(p, P);
}
template <typename F>
PKF_HD void leave_filter_frame(const FilterConst<F>& fc, Quat<F>& x, Quat<F>& xlo, Sym4<F>& P, bool comp) {
  x = qmul(fc.qE, x);
  if (comp) xlo = qmul(fc.qE, xlo);
  P = rotate_cov(fc.qE, P);
}
// the state of one step in the reference frame (what the reference's X_k list holds)
template <typename F> PKF_HD Quat<F> state_in_reference_frame(const FilterConst<F>& fc, const Quat<F>& x) {
  return qmul(fc.qE, x);
}

// ------------------------------------------------------------------------------------------
// General (full-matrix) forms used by the stand-alone Prediction / Correction entry points, which
// must accept whatever the reference accepts: any 4x4 P and K, any 3x3 Q and 4x4 R.
// ------------------------------------------------------------------------------------------
template <typename F> PKF_HD void half_omega(const Vec3<F>& w, Mat4<F>& A) {   // PKF/ExtendedKalmanFilter.py:43-48
  F X = F(0.5) * w.x, Y = F(0.5) * w.y, Z = F(0.5) * w.z;
  A.m[0][0] = F(0); A.m[0][1] = -X; A.m[0][2] = -Y; A.m[0][3] = -Z;
  A.m[1][0] = X; A.m[1][1] = F(0); A.m[1][2] = Z; A.m[1][3] = -Y;
  A.m[2][0] = Y; A.m[2][1] = -Z; A.m[2][2] = F(0); A.m[2][3] = X;
  A.m[3][0] = Z; A.m[3][1] = Y; A.m[3][2] = -X; A.m[3][3] = F(0);
}

// general 4x4 inverse by 2x2 sub-determinants (Laplace expansion); no pivoting needed for S = P + R
template <typename F> PKF_HD void inverse4(const Mat4<F>& Min, Mat4<F>& Out) {
  const F(*a)[4] = Min.m;
  F s0 = a[0][0] * a[1][1] - a[1][0] * a[0][1];
  F s1 = a[0][0] * a[1][2] - a[1][0] * a[0][2];
  F s2 = a[0][0] * a[1][3] - a[1][0] * a[0][3];
  F s3 = a[0][1] * a[1][2] - a[1][1] * a[0][2];
  F s4 = a[0][1] * a[1][3] - a[1][1] * a[0][3];
  F s5 = a[0][2] * a[1][3] - a[1][2] * a[0][3];
  F c5 = a[2][2] * a[3][3] - a[3][2] * a[2][3];
  F c4 = a[2][1] * a[3][3] - a[3][1] * a[2][3];
  F c3 = a[2][1] * a[3][2] - a[3][1] * a[2][2];
  F c2 = a[2][0] * a[3][3] - a[3][0] * a[2][3];
  F c1 = a[2][0] * a[3][2] - a[3][0] * a[2][2];
  F c0 = a[2][0] * a[3][1] - a[3][0] * a[2][1];
  F det = s0 * c5 - s1 * c4 + s2 * c3 + s3 * c2 - s4 * c1 + s5 * c0;
  F id = F(1) / det;
  F(*b)[4] = Out.m;
  b[0][0] = (a[1][1] * c5 - a[1][2] * c4 + a[1][3] * c3) * id;
  b[0][1] = (-a[0][1] * c5 + a[0][2] * c4 - a[0][3] * c3) * id;
  b[0][2] = (a[3][1] * s5 - a[3][2] * s4 + a[3][3] * s3) * id;
  b[0][3] = (-a[2][1] * s5 + a[2][2] * s4 - a[2][3] * s3) * id;
  b[1][0] = (-a[1][0] * c5 + a[1][2] * c2 - a[1][3] * c1) * id;
  b[1][1] = (a[0][0] * c5 - a[0][2] * c2 + a[0][3] * c1) * id;
  b[1][2] = (-a[3][0] * s5 + a[3][2] * s2 - a[3][3] * s1) * id;
  b[1][3] = (a[2][0] * s5 - a[2][2] * s2 + a[2][3] * s1) * id;
  b[2][0] = (a[1][0] * c4 - a[1][1] * c2 + a[1][3] * c0) * id;
  b[2][1] = (-a[0][0] * c4 + a[0][1] * c2 - a[0][3] * c0) * id;
  b[2][2] = (a[3][0] * s4 - a[3][1] * s2 + a[3][3] * s0) * id;
  b[2][3] = (-a[2][0] * s4 + a[2][1] * s2 - a[2][3] * s0) * id;
  b[3][0] = (-a[1][0] * c3 + a[1][1] * c1 - a[1][2] * c0) * id;
  b[3][1] = (a[0][0] * c3 - a[0][1] * c1 + a[0][2] * c0) * id;
  b[3][2] = (-a[3][0] * s3 + a[3][1] * s1 - a[3][2] * s0) * id;
  b[3][3] = (a[2][0] * s3 - a[2][1] * s1 + a[2][2] * s0) * id;
}

// Quaternion -> roll/pitch/yaw in degrees, asin not clamped   (PKF/UtilityFunctions.py:3-14)
template <typename F> PKF_HD Vec3<F> quat_to_rpy_deg(const Quat<F>& q) {
  const F k = F(180.0 / 3.14159265358979323846);
  Vec3<F> o;
  o.x = (F)atan2((double)(F(2) * (q.w * q.x + q.y * q.z)), (double)(F(1) - F(2) * (q.x * q.x + q.y * q.y))) * k;
  o.y = (F)asin((double)(F(2) * (q.w * q.y - q.z * q.x))) * k;
  o.z = (F)atan2((double)(F(2) * (q.w * q.z + q.x * q.y)), (double)(F(1) - F(2) * (q.y * q.y + q.z * q.z))) * k;
  return o;
}

}  // namespace pkf
