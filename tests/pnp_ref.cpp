// pnp_ref.cpp — TEST INFRASTRUCTURE ONLY: a C++ restatement of lorb_pnp_ransac_batched (csrc/pnp.cu,
// csrc/pnp_math.cuh): the counter-based sampler, Lambda Twist P3P, the check point, the inlier score, the
// selection and the finalize pass, in the same operation order.  Built with -ffp-contract=off
// (tests/pnp_ref.py), so every + - * / sqrt is one correctly rounded operation as on the device, and the
// selected hypothesis, counts and flags agree bit for bit.  Only the angle-axis conversion uses libm.
#include <cmath>
#include <cstdint>
#include <cstring>

#include "pnp_math.cuh"  // MAX_DRAW, the tolerances, the iteration counts and splitmix64

using namespace lorb::pnp;

namespace {

typedef double F;
inline F sqrt_rn(F a) { return std::sqrt(a); }
inline F abs_(F a) { return std::fabs(a); }
inline F max_(F a, F b) { return std::fmax(a, b); }
inline bool finite_(F a) { return std::isfinite(a); }

struct Cam {
  double fx, fy, cx, cy;
};
struct Pose {
  F R[9], t[3];
};

bool draw4(uint64_t seed, uint32_t h, uint32_t n, int idx[4]) {
  int taken = 0;
  for (uint32_t k = 0; k <= (uint32_t)MAX_DRAW && taken < 4; k++) {
    const uint64_t r = splitmix64(seed ^ splitmix64(((uint64_t)h << 8) | k));
    const int i = (int)(((r >> 32) * (uint64_t)n) >> 32);
    bool dup = false;
    for (int j = 0; j < taken; j++) dup = dup || idx[j] == i;
    if (!dup) idx[taken++] = i;
  }
  return taken == 4;
}

F dot3(const F a[3], const F b[3]) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
void cross3(const F a[3], const F b[3], F c[3]) {
  c[0] = a[1] * b[2] - a[2] * b[1];
  c[1] = a[2] * b[0] - a[0] * b[2];
  c[2] = a[0] * b[1] - a[1] * b[0];
}

bool root2real(F b, F c, F& r1, F& r2) {
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

F cubic_root(F b, F c, F d) {
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
  for (int i = 0; i < CUBIC_ITERS; i++) {
    const F fx = ((r0 + b) * r0 + c) * r0 + d;
    const F fpx = (3.0 * r0 + 2.0 * b) * r0 + c;
    if (fpx != 0.0) r0 = r0 - fx / fpx;
  }
  return r0;
}

void refine_depths(F& l1, F& l2, F& l3, F a12, F a13, F a23, F b12, F b13, F b23) {
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

// Every Lambda Twist solution in solver order -> sols (up to 4); returns their number.
int p3p(const F y1[3], const F y2[3], const F y3[3], const F x1[3], const F x2[3], const F x3[3], Pose sols[4]) {
  int ns = 0;
  const F b12 = -2.0 * dot3(y1, y2), b13 = -2.0 * dot3(y1, y3), b23 = -2.0 * dot3(y2, y3);
  F d12[3], d13[3], d23[3], n[3];
  for (int i = 0; i < 3; i++) {
    d12[i] = x1[i] - x2[i];
    d13[i] = x1[i] - x3[i];
    d23[i] = x2[i] - x3[i];
  }
  cross3(d12, d13, n);
  const F a12 = dot3(d12, d12), a13 = dot3(d13, d13), a23 = dot3(d23, d23);
  const F c31 = -0.5 * b13, c23 = -0.5 * b23, c12 = -0.5 * b12;
  const F s31 = 1.0 - c31 * c31, s23 = 1.0 - c23 * c23, s12 = 1.0 - c12 * c12;
  if (!(dot3(n, n) > COLLINEAR_TOL * a12 * a13)) return 0;
  if (!(s12 > BEARING_TOL) || !(s31 > BEARING_TOL) || !(s23 > BEARING_TOL)) return 0;
  F xi0[3], xi1[3];
  cross3(d13, n, xi0);
  cross3(n, d12, xi1);
  const F idet = 1.0 / dot3(d12, xi0);
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
  const F vv = sqrt_rn(max_(0.0, -e2 / e1));

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
    for (int j = 0; j < 2; j++) {
      const F ta = tau[j];
      if (!(ta > 0.0)) continue;
      const F d = a23 / (ta * (b23 + ta) + 1.0);
      if (!(d > 0.0)) continue;
      F l2 = sqrt_rn(d);
      F l3 = ta * l2;
      F l1 = w0 * l2 + w1 * l3;
      if (!(l1 >= 0.0)) continue;
      refine_depths(l1, l2, l3, a12, a13, a23, b12, b13, b23);
      F ry1[3], yd1[3], yd2[3], yx[3];
      for (int i = 0; i < 3; i++) {
        ry1[i] = y1[i] * l1;
        yd1[i] = ry1[i] - y2[i] * l2;
        yd2[i] = ry1[i] - y3[i] * l3;
      }
      cross3(yd1, yd2, yx);
      Pose& P = sols[ns++];
      for (int i = 0; i < 3; i++)
        for (int k = 0; k < 3; k++) P.R[3 * i + k] = yd1[i] * xi0[k] + yd2[i] * xi1[k] + yx[i] * xi2[k];
      for (int i = 0; i < 3; i++)
        P.t[i] = ry1[i] - (P.R[3 * i] * x1[0] + P.R[3 * i + 1] * x1[1] + P.R[3 * i + 2] * x1[2]);
    }
  }
  return ns;
}

void to_cam(const Pose& P, const F X[3], F q[3]) {
  for (int i = 0; i < 3; i++) q[i] = P.R[3 * i] * X[0] + P.R[3 * i + 1] * X[1] + P.R[3 * i + 2] * X[2] + P.t[i];
}

bool reproj2(const Pose& P, const F X[3], F u, F v, const Cam& K, F& e) {
  F q[3];
  to_cam(P, X, q);
  const F iz = 1.0 / q[2];
  const F ru = K.fx * (q[0] * iz) + K.cx - u;
  const F rv = K.fy * (q[1] * iz) + K.cy - v;
  e = ru * ru + rv * rv;
  return q[2] > 0.0;
}

void bearing(F u, F v, const Cam& K, F y[3]) {
  const F bx = (u - K.cx) / K.fx, by = (v - K.cy) / K.fy;
  const F nn = sqrt_rn(bx * bx + by * by + 1.0);
  y[0] = bx / nn;
  y[1] = by / nn;
  y[2] = 1.0 / nn;
}

bool hypothesis(uint64_t seed, uint32_t h, int n, const float* xw, const float* uv, const Cam& K, Pose& best) {
  int idx[4];
  if (!draw4(seed, h, (uint32_t)n, idx)) return false;
  F X[4][3], y[3][3];
  for (int s = 0; s < 4; s++)
    for (int i = 0; i < 3; i++) X[s][i] = (double)xw[3 * idx[s] + i];
  for (int s = 0; s < 3; s++) bearing((double)uv[2 * idx[s]], (double)uv[2 * idx[s] + 1], K, y[s]);
  const F u4 = (double)uv[2 * idx[3]], v4 = (double)uv[2 * idx[3] + 1];
  Pose sols[4];
  const int ns = p3p(y[0], y[1], y[2], X[0], X[1], X[2], sols);
  F best_e = INFINITY;
  bool found = false;
  for (int k = 0; k < ns; k++) {
    const Pose& P = sols[k];
    bool ok = true;
    for (int i = 0; i < 9; i++) ok = ok && finite_(P.R[i]);
    for (int i = 0; i < 3; i++) ok = ok && finite_(P.t[i]);
    for (int s = 0; s < 3; s++) {
      F q[3];
      to_cam(P, X[s], q);
      ok = ok && q[2] > 0.0;
    }
    if (!ok) continue;
    F e;
    if (reproj2(P, X[3], u4, v4, K, e) && e < best_e) {
      best_e = e;
      best = P;
      found = true;
    }
  }
  return found;
}

bool classify(const Pose& P, const F X[3], F u, F v, F w, const Cam& K, double chi2, double& c2) {
  F e;
  const bool front = reproj2(P, X, u, v, K, e);
  const F s = w * e;
  c2 = front ? s : INFINITY;
  return front && s <= chi2;
}

void rotation_to_angle_axis(const double R[9], double aa[3]) {
  const double tr = R[0] + R[4] + R[8];
  double q[4];
  if (tr >= R[0] && tr >= R[4] && tr >= R[8]) {
    q[0] = 0.5 * std::sqrt(1.0 + tr);
    const double f = 0.25 / q[0];
    q[1] = (R[7] - R[5]) * f;
    q[2] = (R[2] - R[6]) * f;
    q[3] = (R[3] - R[1]) * f;
  } else if (R[0] >= R[4] && R[0] >= R[8]) {
    q[1] = 0.5 * std::sqrt(1.0 + R[0] - R[4] - R[8]);
    const double f = 0.25 / q[1];
    q[0] = (R[7] - R[5]) * f;
    q[2] = (R[1] + R[3]) * f;
    q[3] = (R[2] + R[6]) * f;
  } else if (R[4] >= R[8]) {
    q[2] = 0.5 * std::sqrt(1.0 - R[0] + R[4] - R[8]);
    const double f = 0.25 / q[2];
    q[0] = (R[2] - R[6]) * f;
    q[1] = (R[1] + R[3]) * f;
    q[3] = (R[5] + R[7]) * f;
  } else {
    q[3] = 0.5 * std::sqrt(1.0 - R[0] - R[4] + R[8]);
    const double f = 0.25 / q[3];
    q[0] = (R[3] - R[1]) * f;
    q[1] = (R[2] + R[6]) * f;
    q[2] = (R[5] + R[7]) * f;
  }
  const double qn = 1.0 / std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  for (int i = 0; i < 4; i++) q[i] *= qn;
  const double s2 = q[1] * q[1] + q[2] * q[2] + q[3] * q[3];
  double k = 2.0;
  if (s2 > 0.0) {
    const double s = std::sqrt(s2), c = q[0];
    k = 2.0 * (c < 0.0 ? std::atan2(-s, -c) : std::atan2(s, c)) / s;
  }
  for (int i = 0; i < 3; i++) aa[i] = q[i + 1] * k;
}

}  // namespace

extern "C" {

int pnr_draw4(uint64_t seed, uint32_t h, uint32_t n, int* idx) { return draw4(seed, h, n, idx) ? 1 : 0; }

// Every P3P solution of three pixel / world correspondences: R_out [4 x 9] row-major, t_out [4 x 3].
int pnr_p3p(const float* xw, const float* uv, const float* K4, double* R_out, double* t_out) {
  const Cam K = {K4[0], K4[1], K4[2], K4[3]};
  F X[3][3], y[3][3];
  for (int s = 0; s < 3; s++) {
    for (int i = 0; i < 3; i++) X[s][i] = (double)xw[3 * s + i];
    bearing((double)uv[2 * s], (double)uv[2 * s + 1], K, y[s]);
  }
  Pose sols[4];
  const int ns = p3p(y[0], y[1], y[2], X[0], X[1], X[2], sols);
  for (int k = 0; k < ns; k++) {
    std::memcpy(R_out + 9 * k, sols[k].R, 72);
    std::memcpy(t_out + 3 * k, sols[k].t, 24);
  }
  return ns;
}

void pnr_rotation_to_angle_axis(const double* R, double* aa) { rotation_to_angle_axis(R, aa); }

// lorb_pnp_ransac_batched on the host (no argument checks: the tests pass valid inputs).
void pnr_ransac(int n_problems, const int* corr_off, const float* xw, const float* uv, const float* info,
                const float* K4, const uint64_t* seeds, int H, double chi2, double* out_rt, int* best_hyp,
                int* n_inliers, uint8_t* out_inlier, double* out_chi2) {
  const Cam K = {K4[0], K4[1], K4[2], K4[3]};
#pragma omp parallel for schedule(dynamic)
  for (int b = 0; b < n_problems; b++) {
    const int o0 = corr_off[b], n = corr_off[b + 1] - o0;
    const float* pxw = xw + 3 * (size_t)o0;
    const float* puv = uv + 2 * (size_t)o0;
    const uint64_t seed = seeds ? seeds[b] : (uint64_t)b;
    int best_h = -1, best_c = -1;
    Pose best;
    for (int h = 0; n >= 4 && h < H; h++) {
      Pose P;
      if (!hypothesis(seed, (uint32_t)h, n, pxw, puv, K, P)) continue;
      int cnt = 0;
      for (int i = 0; i < n; i++) {
        const F X[3] = {(double)pxw[3 * i], (double)pxw[3 * i + 1], (double)pxw[3 * i + 2]};
        F e;
        const bool front = reproj2(P, X, (double)puv[2 * i], (double)puv[2 * i + 1], K, e);
        const F w = info ? (double)info[o0 + i] : 1.0;
        cnt += (front && w * e <= chi2) ? 1 : 0;
      }
      if (cnt > best_c) {
        best_c = cnt;
        best_h = h;
        best = P;
      }
    }
    const bool ok = best_h >= 0;
    double aa[3] = {0.0, 0.0, 0.0};
    if (ok) rotation_to_angle_axis(best.R, aa);
    for (int i = 0; i < 3; i++) {
      out_rt[6 * (size_t)b + i] = aa[i];
      out_rt[6 * (size_t)b + 3 + i] = ok ? best.t[i] : 0.0;
    }
    best_hyp[b] = best_h;
    int cnt = 0;
    for (int i = 0; i < n; i++) {
      double c2 = INFINITY;
      bool in = false;
      if (ok) {
        const F X[3] = {(double)pxw[3 * i], (double)pxw[3 * i + 1], (double)pxw[3 * i + 2]};
        in = classify(best, X, (double)puv[2 * i], (double)puv[2 * i + 1], info ? (double)info[o0 + i] : 1.0, K,
                      chi2, c2);
      }
      out_inlier[o0 + i] = in ? 1 : 0;
      if (out_chi2) out_chi2[o0 + i] = c2;
      cnt += in;
    }
    n_inliers[b] = cnt;
  }
}

}  // extern "C"
