// pnp_math.cuh — fp64 device math of the P3P RANSAC (pnp.cu): the counter-based sampler, the Lambda Twist
// P3P solver (Persson & Nordberg, ECCV 2018) and the inlier test.
//
// Every arithmetic operation from the sampler to the inlier count is an IEEE correctly rounded +, -, x, / or
// sqrt on the type F below, whose operators are __dadd_rn / __dsub_rn / __dmul_rn / __ddiv_rn / __dsqrt_rn
// (ptxas never contracts those into FMAs), and every loop has a fixed trip count.  tests/pnp_ref.cpp states
// the same expressions on plain double, compiled with -ffp-contract=off, and so reproduces hypotheses,
// counts and flags bit for bit.  The constants below are shared with it (it includes this header; the
// device code is compiled only by nvcc).
#pragma once
#include <stdint.h>

namespace lorb {
namespace pnp {

constexpr int MAX_DRAW = 255;            // draws k = 0 .. MAX_DRAW of one hypothesis
constexpr double COLLINEAR_TOL = 1e-10;  // |d12 x d13|^2 <= tol |d12|^2 |d13|^2: collinear (or coincident) world triple
constexpr double BEARING_TOL = 1e-12;    // 1 - (yi . yj)^2 <= tol: coincident bearings
constexpr int CUBIC_ITERS = 50;          // Newton steps on the cubic of Lambda Twist
constexpr int REFINE_ITERS = 5;          // Gauss-Newton steps on the depths

// SplitMix64 (Steele, Lea & Flood 2014)
#ifdef __CUDACC__
__host__ __device__
#endif
inline uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  uint64_t z = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

#ifdef __CUDACC__

// An fp64 value whose arithmetic is correctly rounded and never contracted.
struct F {
  double v;
};
__device__ __forceinline__ F operator+(F a, F b) { return F{__dadd_rn(a.v, b.v)}; }
__device__ __forceinline__ F operator-(F a, F b) { return F{__dsub_rn(a.v, b.v)}; }
__device__ __forceinline__ F operator*(F a, F b) { return F{__dmul_rn(a.v, b.v)}; }
__device__ __forceinline__ F operator/(F a, F b) { return F{__ddiv_rn(a.v, b.v)}; }
__device__ __forceinline__ F operator-(F a) { return F{-a.v}; }
#define LORB_PNP_MIXED(op)                                                         \
  __device__ __forceinline__ F operator op(double a, F b) { return F{a} op b; }    \
  __device__ __forceinline__ F operator op(F a, double b) { return a op F{b}; }
LORB_PNP_MIXED(+)
LORB_PNP_MIXED(-)
LORB_PNP_MIXED(*)
LORB_PNP_MIXED(/)
#undef LORB_PNP_MIXED
#define LORB_PNP_CMP(op)                                                                  \
  __device__ __forceinline__ bool operator op(F a, F b) { return a.v op b.v; }            \
  __device__ __forceinline__ bool operator op(F a, double b) { return a.v op b; }
LORB_PNP_CMP(<)
LORB_PNP_CMP(<=)
LORB_PNP_CMP(>)
LORB_PNP_CMP(>=)
LORB_PNP_CMP(!=)
#undef LORB_PNP_CMP
__device__ __forceinline__ F sqrt_rn(F a) { return F{__dsqrt_rn(a.v)}; }
__device__ __forceinline__ F abs_(F a) { return F{fabs(a.v)}; }
__device__ __forceinline__ F max_(F a, F b) { return F{fmax(a.v, b.v)}; }
__device__ __forceinline__ bool finite_(F a) { return isfinite(a.v); }

struct Cam {
  double fx, fy, cx, cy;  // float intrinsics widened
};

// The pose of one hypothesis: x_c = R X + t (R row-major).
struct Pose {
  F R[9], t[3];
};

// The four distinct indices of hypothesis h among n correspondences (the sampler of lorb_pnp_ransac_batched).
__device__ __forceinline__ bool draw4(uint64_t seed, uint32_t h, uint32_t n, int idx[4]) {
  int i0 = -1, i1 = -1, i2 = -1, i3 = -1, taken = 0;
#pragma unroll 1
  for (uint32_t k = 0; k <= (uint32_t)MAX_DRAW && taken < 4; k++) {
    const uint64_t r = splitmix64(seed ^ splitmix64(((uint64_t)h << 8) | k));
    const int i = (int)(((r >> 32) * (uint64_t)n) >> 32);
    if (i == i0 || i == i1 || i == i2) continue;
    if (taken == 0) i0 = i;
    else if (taken == 1) i1 = i;
    else if (taken == 2) i2 = i;
    else i3 = i;
    taken++;
  }
  idx[0] = i0; idx[1] = i1; idx[2] = i2; idx[3] = i3;
  return taken == 4;
}

__device__ __forceinline__ F dot3(const F a[3], const F b[3]) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
__device__ __forceinline__ void cross3(const F a[3], const F b[3], F c[3]) {
  c[0] = a[1] * b[2] - a[2] * b[1];
  c[1] = a[2] * b[0] - a[0] * b[2];
  c[2] = a[0] * b[1] - a[1] * b[0];
}

// Roots of x^2 + b x + c (Lambda Twist's root2real): r1 the larger in magnitude, r2 = c / r1.
__device__ __forceinline__ bool root2real(F b, F c, F& r1, F& r2) {
  const F v = b * b - 4.0 * c;
  if (v < 0.0) {
    r1 = r2 = 0.5 * b;
    return false;
  }
  const F y = sqrt_rn(v);
  if (b < 0.0) r1 = 0.5 * (-b + y);
  else r1 = 0.5 * (-b - y);
  r2 = c / r1;
  return true;
}

// A real root of x^3 + b x^2 + c x + d (Lambda Twist's cubick), with a fixed number of Newton steps.
__device__ __forceinline__ F cubic_root(F b, F c, F d) {
  F r0;
  if (b * b >= 3.0 * c) {
    const F v = sqrt_rn(b * b - 3.0 * c);
    const F t1 = (-b - v) / 3.0;
    F k = ((t1 + b) * t1 + c) * t1 + d;
    if (k > 0.0) {
      r0 = t1 - sqrt_rn(-k / (3.0 * t1 + b));
    } else {
      const F t2 = (-b + v) / 3.0;
      k = ((t2 + b) * t2 + c) * t2 + d;
      r0 = t2 + sqrt_rn(-k / (3.0 * t2 + b));
    }
  } else {
    r0 = -b / 3.0;
    if (abs_((3.0 * r0 + 2.0 * b) * r0 + c) < 1e-4) r0 = r0 + 1.0;
  }
#pragma unroll 1
  for (int i = 0; i < CUBIC_ITERS; i++) {
    const F fx = ((r0 + b) * r0 + c) * r0 + d;
    const F fpx = (3.0 * r0 + 2.0 * b) * r0 + c;
    if (fpx != 0.0) r0 = r0 - fx / fpx;
  }
  return r0;
}

// Gauss-Newton on the three depth equations; a step that raises |r1| + |r2| + |r3| is not taken.
__device__ __forceinline__ void refine_depths(F& l1, F& l2, F& l3, F a12, F a13, F a23, F b12, F b13, F b23) {
#pragma unroll 1
  for (int it = 0; it < REFINE_ITERS; it++) {
    const F r1 = l1 * l1 + l2 * l2 + b12 * l1 * l2 - a12;
    const F r2 = l1 * l1 + l3 * l3 + b13 * l1 * l3 - a13;
    const F r3 = l2 * l2 + l3 * l3 + b23 * l2 * l3 - a23;
    const F v0 = 2.0 * l1 + b12 * l2, v1 = 2.0 * l2 + b12 * l1;
    const F v3 = 2.0 * l1 + b13 * l3, v5 = 2.0 * l3 + b13 * l1;
    const F v7 = 2.0 * l2 + b23 * l3, v8 = 2.0 * l3 + b23 * l2;
    const F det = 1.0 / (-v0 * v5 * v7 - v1 * v3 * v8);
    const F n1 = l1 - det * (-v5 * v7 * r1 - v1 * v8 * r2 + v1 * v5 * r3);
    const F n2 = l2 - det * (-v3 * v8 * r1 + v0 * v8 * r2 - v0 * v5 * r3);
    const F n3 = l3 - det * (v3 * v7 * r1 - v0 * v7 * r2 - v1 * v3 * r3);
    const F q1 = n1 * n1 + n2 * n2 + b12 * n1 * n2 - a12;
    const F q2 = n1 * n1 + n3 * n3 + b13 * n1 * n3 - a13;
    const F q3 = n2 * n2 + n3 * n3 + b23 * n2 * n3 - a23;
    if (abs_(q1) + abs_(q2) + abs_(q3) <= abs_(r1) + abs_(r2) + abs_(r3)) {
      l1 = n1;
      l2 = n2;
      l3 = n3;
    }
  }
}

// Lambda Twist P3P on unit bearings y1..y3 of world points x1..x3.  emit(R, t) is called for every solution
// with positive depths l1 >= 0, l2, l3 > 0, in solver order (+v: tau1, tau2; -v: tau1, tau2).  A collinear
// world triple or coincident bearings give no call.
template <class Emit>
__device__ __forceinline__ void p3p(const F y1[3], const F y2[3], const F y3[3], const F x1[3], const F x2[3],
                                    const F x3[3], Emit&& emit) {
  const F b12 = -2.0 * dot3(y1, y2), b13 = -2.0 * dot3(y1, y3), b23 = -2.0 * dot3(y2, y3);
  F d12[3], d13[3], d23[3], n[3];
#pragma unroll
  for (int i = 0; i < 3; i++) {
    d12[i] = x1[i] - x2[i];
    d13[i] = x1[i] - x3[i];
    d23[i] = x2[i] - x3[i];
  }
  cross3(d12, d13, n);
  const F a12 = dot3(d12, d12), a13 = dot3(d13, d13), a23 = dot3(d23, d23);
  const F c31 = -0.5 * b13, c23 = -0.5 * b23, c12 = -0.5 * b12;
  const F s31 = 1.0 - c31 * c31, s23 = 1.0 - c23 * c23, s12 = 1.0 - c12 * c12;
  if (!(dot3(n, n) > COLLINEAR_TOL * a12 * a13)) return;
  if (!(s12 > BEARING_TOL) || !(s31 > BEARING_TOL) || !(s23 > BEARING_TOL)) return;
  // X = [d12 d13 n] (columns); its inverse has rows (d13 x n, n x d12, d12 x d13) / det
  F xi0[3], xi1[3];
  cross3(d13, n, xi0);
  cross3(n, d12, xi1);
  const F idet = 1.0 / dot3(d12, xi0);
#pragma unroll
  for (int i = 0; i < 3; i++) {
    xi0[i] = xi0[i] * idet;
    xi1[i] = xi1[i] * idet;
  }
  const F xi2[3] = {n[0] * idet, n[1] * idet, n[2] * idet};

  const F blob = c12 * c23 * c31 - 1.0;
  F p3 = a13 * (a23 * s31 - a13 * s23);
  F p2 = 2.0 * blob * a23 * a13 + a13 * (2.0 * a12 + a13) * s23 + a23 * (a23 - a12) * s31;
  F p1 = a23 * (a13 - a23) * s12 - a12 * a12 * s23 - 2.0 * a12 * (blob * a23 + a13 * s23);
  F p0 = a12 * (a12 * s23 - a23 * s12);
  p3 = 1.0 / p3;
  p2 = p2 * p3;
  p1 = p1 * p3;
  p0 = p0 * p3;
  const F g = cubic_root(p2, p1, p0);

  // A = D1 - g D2 (symmetric, one eigenvalue 0); eigenvectors of the other two
  const F A00 = a23 * (1.0 - g), A01 = a23 * b12 * 0.5, A02 = a23 * b13 * g * -0.5;
  const F A11 = a23 - a12 + a13 * g, A12 = b23 * (a13 * g - a12) * 0.5, A22 = g * (a13 - a23) - a12;
  const F x01s = A01 * A01;
  const F eb = -A00 - A11 - A22;
  const F ec = -x01s - A02 * A02 - A12 * A12 + A00 * (A11 + A22) + A11 * A22;
  F e1, e2;
  root2real(eb, ec, e1, e2);
  if (abs_(e1) < abs_(e2)) {
    const F tmp = e1;
    e1 = e2;
    e2 = tmp;
  }
  const F mx0011 = -A00 * A11;
  const F prec0 = A01 * A12 - A02 * A11, prec1 = A01 * A02 - A00 * A12;
  const F tm1 = 1.0 / (e1 * (A00 + A11) + mx0011 - e1 * e1 + x01s);
  const F a11 = -(e1 * A02 + prec0) * tm1, a21 = -(e1 * A12 + prec1) * tm1;
  const F rn1 = 1.0 / sqrt_rn(a11 * a11 + a21 * a21 + 1.0);
  const F tm2 = 1.0 / (e2 * (A00 + A11) + mx0011 - e2 * e2 + x01s);
  const F a12v = -(e2 * A02 + prec0) * tm2, a22v = -(e2 * A12 + prec1) * tm2;
  const F rn2 = 1.0 / sqrt_rn(a12v * a12v + a22v * a22v + 1.0);
  const F V00 = a11 * rn1, V10 = a21 * rn1, V20 = rn1;
  const F V01 = a12v * rn2, V11 = a22v * rn2, V21 = rn2;
  const F vv = sqrt_rn(max_(F{0.0}, -e2 / e1));

#pragma unroll 1
  for (int sgn = 0; sgn < 2; sgn++) {
    const F s = sgn == 0 ? vv : -vv;
    const F w2 = 1.0 / (s * V01 - V00);
    const F w0 = (V10 - s * V11) * w2;
    const F w1 = (V20 - s * V21) * w2;
    const F a = 1.0 / ((a13 - a12) * w1 * w1 - a12 * b13 * w1 - a12);
    const F b = (a13 * b12 * w1 - a12 * b13 * w0 - 2.0 * w0 * w1 * (a12 - a13)) * a;
    const F c = ((a13 - a12) * w0 * w0 + a13 * b12 * w0 + a13) * a;
    if (!(b * b - 4.0 * c >= 0.0)) continue;
    F tau[2];
    root2real(b, c, tau[0], tau[1]);
#pragma unroll 1
    for (int j = 0; j < 2; j++) {
      const F ta = j == 0 ? tau[0] : tau[1];
      if (!(ta > 0.0)) continue;
      const F d = a23 / (ta * (b23 + ta) + 1.0);
      if (!(d > 0.0)) continue;
      F l2 = sqrt_rn(d);
      F l3 = ta * l2;
      F l1 = w0 * l2 + w1 * l3;
      if (!(l1 >= 0.0)) continue;
      refine_depths(l1, l2, l3, a12, a13, a23, b12, b13, b23);
      F ry1[3], yd1[3], yd2[3], yx[3];
#pragma unroll
      for (int i = 0; i < 3; i++) {
        ry1[i] = y1[i] * l1;
        yd1[i] = ry1[i] - y2[i] * l2;
        yd2[i] = ry1[i] - y3[i] * l3;
      }
      cross3(yd1, yd2, yx);
      Pose P;
#pragma unroll
      for (int i = 0; i < 3; i++)
#pragma unroll
        for (int k = 0; k < 3; k++) P.R[3 * i + k] = yd1[i] * xi0[k] + yd2[i] * xi1[k] + yx[i] * xi2[k];
#pragma unroll
      for (int i = 0; i < 3; i++)
        P.t[i] = ry1[i] - (P.R[3 * i] * x1[0] + P.R[3 * i + 1] * x1[1] + P.R[3 * i + 2] * x1[2]);
      emit(P);
    }
  }
}

// Camera coordinates of X at pose P.
__device__ __forceinline__ void to_cam(const Pose& P, const F X[3], F q[3]) {
#pragma unroll
  for (int i = 0; i < 3; i++) q[i] = P.R[3 * i] * X[0] + P.R[3 * i + 1] * X[1] + P.R[3 * i + 2] * X[2] + P.t[i];
}

// Squared pixel error |r|^2 of (X, u, v) at P (pinhole fx, fy) and whether the point is in front (z > 0).
__device__ __forceinline__ bool reproj2(const Pose& P, const F X[3], F u, F v, const Cam& K, F& e) {
  F q[3];
  to_cam(P, X, q);
  const F iz = 1.0 / q[2];
  const F ru = F{K.fx} * (q[0] * iz) + F{K.cx} - u;
  const F rv = F{K.fy} * (q[1] * iz) + F{K.cy} - v;
  e = ru * ru + rv * rv;
  return q[2] > 0.0;
}

__device__ __forceinline__ void bearing(F u, F v, const Cam& K, F y[3]) {
  const F bx = (u - K.cx) / F{K.fx}, by = (v - K.cy) / F{K.fy};
  const F nn = sqrt_rn(bx * bx + by * by + 1.0);
  y[0] = bx / nn;
  y[1] = by / nn;
  y[2] = 1.0 / nn;
}

// Hypothesis h of one problem (xw / uv point at its first correspondence): the P3P solution on draws 0-2
// with every sample depth > 0, finite, and the smallest squared pixel error at draw 3 (in front of the
// camera); ties keep the earlier solution.  false: the hypothesis is invalid.
__device__ __forceinline__ bool hypothesis(uint64_t seed, uint32_t h, int n, const float* __restrict__ xw,
                                           const float* __restrict__ uv, const Cam& K, Pose& best) {
  int idx[4];
  if (!draw4(seed, h, (uint32_t)n, idx)) return false;
  F X[4][3], y[3][3];
#pragma unroll
  for (int s = 0; s < 4; s++)
#pragma unroll
    for (int i = 0; i < 3; i++) X[s][i] = F{(double)xw[3 * idx[s] + i]};
#pragma unroll
  for (int s = 0; s < 3; s++) bearing(F{(double)uv[2 * idx[s]]}, F{(double)uv[2 * idx[s] + 1]}, K, y[s]);
  const F u4 = F{(double)uv[2 * idx[3]]}, v4 = F{(double)uv[2 * idx[3] + 1]};
  F best_e = F{__longlong_as_double(0x7FF0000000000000ll)};  // +inf
  bool found = false;
  p3p(y[0], y[1], y[2], X[0], X[1], X[2], [&](const Pose& P) {
    bool ok = true;
#pragma unroll
    for (int i = 0; i < 9; i++) ok = ok && finite_(P.R[i]);
#pragma unroll
    for (int i = 0; i < 3; i++) ok = ok && finite_(P.t[i]);
#pragma unroll
    for (int s = 0; s < 3; s++) {
      F q[3];
      to_cam(P, X[s], q);
      ok = ok && q[2] > 0.0;
    }
    if (!ok) return;
    F e;
    if (reproj2(P, X[3], u4, v4, K, e) && e < best_e) {
      best_e = e;
      best = P;
      found = true;
    }
  });
  return found;
}

#endif  // __CUDACC__

}  // namespace pnp
}  // namespace lorb
