// ba_math.cuh — fp64 device math shared by the bundle-adjustment kernels.
//
// Residual model = the reference's three Ceres functors (reference
// src/bundle_adjust.cpp:22-64 PoseCost, :68-113 MPCost, :116-151 PoseMPCost):
//     q = R(w) X + t ,  r = ( q0/q2*fu + cx - u , q1/q2*fv + cy - v )
// with R(w) = ceres::AngleAxisRotatePoint (Rodrigues for |w|^2 > DBL_EPSILON,
// X + w x X otherwise).  The Jacobians are the analytic derivatives of exactly
// that function (additive angle-axis parametrisation, as Ceres autodiff sees
// it, SURVEY §7.2), factored per camera: R and dR/dw_m are built once per
// linearisation (cam_rotation), so the per-observation work has no
// trigonometry.
#pragma once
#include <float.h>

#include "common.cuh"

namespace lorb {

// 36 doubles per camera: R (row-major 3x3) then dR/dw_0, dR/dw_1, dR/dw_2.
constexpr int CAMROT = 36;

__device__ __forceinline__ void cam_rotation(const double* __restrict__ w, double* __restrict__ out,
                                             bool with_derivs) {
  const double w0 = w[0], w1 = w[1], w2 = w[2];
  const double th2 = w0 * w0 + w1 * w1 + w2 * w2;
  double* R = out;
  if (th2 > DBL_EPSILON) {
    const double th = sqrt(th2);
    double s, c;
    sincos(th, &s, &c);
    const double ith = 1.0 / th;
    const double k[3] = {w0 * ith, w1 * ith, w2 * ith};
    const double omc = 1.0 - c;
    // R = c I + s [k]x + (1-c) k k^T
    R[0] = c + omc * k[0] * k[0];
    R[1] = -s * k[2] + omc * k[0] * k[1];
    R[2] = s * k[1] + omc * k[0] * k[2];
    R[3] = s * k[2] + omc * k[1] * k[0];
    R[4] = c + omc * k[1] * k[1];
    R[5] = -s * k[0] + omc * k[1] * k[2];
    R[6] = -s * k[1] + omc * k[2] * k[0];
    R[7] = s * k[0] + omc * k[2] * k[1];
    R[8] = c + omc * k[2] * k[2];
    if (with_derivs) {
#pragma unroll
      for (int m = 0; m < 3; m++) {
        double* D = out + 9 * (m + 1);
        const double km = k[m];
        // dk/dw_m = (e_m - k k_m) / th
        double dk[3];
#pragma unroll
        for (int a = 0; a < 3; a++) dk[a] = ((a == m ? 1.0 : 0.0) - k[a] * km) * ith;
        const double d_c = -s * km;  // d cos / dw_m
        const double d_s = c * km;   // d sin / dw_m
        // d/dw_m [ c I + s K + (1-c) k k^T ]
#pragma unroll
        for (int a = 0; a < 3; a++)
#pragma unroll
          for (int b = 0; b < 3; b++) {
            double v = (a == b ? d_c : 0.0);
            v += (s * km) * k[a] * k[b] + omc * (dk[a] * k[b] + k[a] * dk[b]);
            D[3 * a + b] = v;
          }
        // + d_s [k]x + s [dk]x
        const double x0 = d_s * k[0] + s * dk[0], x1 = d_s * k[1] + s * dk[1],
                     x2 = d_s * k[2] + s * dk[2];
        D[1] -= x2; D[2] += x1;
        D[3] += x2; D[5] -= x0;
        D[6] -= x1; D[7] += x0;
      }
    }
  } else {
    // Ceres small-angle branch: R X = X + w x X
    R[0] = 1.0; R[1] = -w2; R[2] = w1;
    R[3] = w2;  R[4] = 1.0; R[5] = -w0;
    R[6] = -w1; R[7] = w0;  R[8] = 1.0;
    if (with_derivs) {
#pragma unroll
      for (int i = 9; i < CAMROT; i++) out[i] = 0.0;
      // d/dw_0: [e0]x, d/dw_1: [e1]x, d/dw_2: [e2]x
      out[9 + 5] = -1.0;  out[9 + 7] = 1.0;
      out[18 + 2] = 1.0;  out[18 + 6] = -1.0;
      out[27 + 1] = -1.0; out[27 + 3] = 1.0;
    }
  }
}

struct Intr {
  double fu, fv, cx, cy;  // float intrinsics widened (T(mpCamera->fx) ...)
};

// residual + Jacobian blocks of one observation.
//   rot: CAMROT doubles (R, dR) of the observing camera (dR unused when !CAM)
//   Jc[12] = d r / d (w, t) row-major 2x6 ; Jp[6] = d r / d X row-major 2x3
template <bool CAM, bool PT>
__device__ __forceinline__ void obs_eval(const double* __restrict__ rot, const double t[3],
                                         const double X[3], const Intr& K, double u, double v,
                                         double r[2], double* Jc, double* Jp) {
  const double* R = rot;
  const double q0 = R[0] * X[0] + R[1] * X[1] + R[2] * X[2] + t[0];
  const double q1 = R[3] * X[0] + R[4] * X[1] + R[5] * X[2] + t[1];
  const double q2 = R[6] * X[0] + R[7] * X[1] + R[8] * X[2] + t[2];
  const double iz = 1.0 / q2;
  const double pu = q0 * iz, pv = q1 * iz;
  r[0] = pu * K.fu + K.cx - u;
  r[1] = pv * K.fv + K.cy - v;
  const double a0 = K.fu * iz, a1 = K.fv * iz;
  const double b0 = -a0 * pu, b1 = -a1 * pv;
  if (PT) {
#pragma unroll
    for (int a = 0; a < 3; a++) {
      Jp[a] = a0 * R[a] + b0 * R[6 + a];
      Jp[3 + a] = a1 * R[3 + a] + b1 * R[6 + a];
    }
  }
  if (CAM) {
#pragma unroll
    for (int m = 0; m < 3; m++) {
      const double* D = rot + 9 * (m + 1);
      const double d0 = D[0] * X[0] + D[1] * X[1] + D[2] * X[2];
      const double d1 = D[3] * X[0] + D[4] * X[1] + D[5] * X[2];
      const double d2 = D[6] * X[0] + D[7] * X[1] + D[8] * X[2];
      Jc[m] = a0 * d0 + b0 * d2;
      Jc[6 + m] = a1 * d1 + b1 * d2;
    }
    Jc[3] = a0;  Jc[4] = 0.0; Jc[5] = b0;
    Jc[9] = 0.0; Jc[10] = a1; Jc[11] = b1;
  }
}

// Robust loss of one residual block, s = |r|^2, scale a (LORB_LOSS_*; Ceres HuberLoss,
// SoftLOneLoss, CauchyLoss): rho(s) and rho'(s).  rho of soft-L1 and Cauchy is written without the
// cancellation of 2b (sqrt(1 + s/b) - 1) and log(1 + s/b) for s << b (a scale far above the residuals
// would otherwise leave five significant digits of the cost).  rho'' is not needed: it is <= 0 for all three, so
// Ceres' Corrector drops its curvature term and scales r and J by sqrt(rho') alone.
__device__ __forceinline__ void loss_eval(int kind, double a, double s, double& rho, double& rho1) {
  const double b = a * a;
  if (kind == LORB_LOSS_HUBER) {
    if (s > b) {
      const double r = sqrt(s);
      rho = 2.0 * a * r - b;
      rho1 = fmax(DBL_MIN, a / r);
    } else {
      rho = s;
      rho1 = 1.0;
    }
  } else if (kind == LORB_LOSS_SOFTLONE) {
    const double t = sqrt(1.0 + s * (1.0 / b));
    rho = 2.0 * s / (t + 1.0);  // = 2b (t - 1)
    rho1 = fmax(DBL_MIN, 1.0 / t);
  } else if (kind == LORB_LOSS_CAUCHY) {
    const double sum = 1.0 + s * (1.0 / b);
    rho = b * log1p(s * (1.0 / b));
    rho1 = fmax(DBL_MIN, 1.0 / sum);
  } else {
    rho = s;
    rho1 = 1.0;
  }
}

// Corrector of one observation: r and its Jacobian blocks (Jc: 12, Jp: 6; each may be null) are
// scaled by sqrt(rho'(|r|^2)); returns rho(|r|^2), the observation's share of 2 * cost.
__device__ __forceinline__ double robust_correct(int kind, double a, double r[2], double* Jc, double* Jp) {
  double rho, rho1;
  loss_eval(kind, a, r[0] * r[0] + r[1] * r[1], rho, rho1);
  const double w = sqrt(rho1);
  r[0] *= w;
  r[1] *= w;
  if (Jc) {
#pragma unroll
    for (int k = 0; k < 12; k++) Jc[k] *= w;
  }
  if (Jp) {
#pragma unroll
    for (int k = 0; k < 6; k++) Jp[k] *= w;
  }
  return rho;
}

// residual only (candidate cost)
__device__ __forceinline__ double obs_cost(const double* __restrict__ R, const double t[3],
                                           const double X[3], const Intr& K, double u, double v) {
  const double q0 = R[0] * X[0] + R[1] * X[1] + R[2] * X[2] + t[0];
  const double q1 = R[3] * X[0] + R[4] * X[1] + R[5] * X[2] + t[1];
  const double q2 = R[6] * X[0] + R[7] * X[1] + R[8] * X[2] + t[2];
  const double iz = 1.0 / q2;
  const double r0 = q0 * iz * K.fu + K.cx - u;
  const double r1 = q1 * iz * K.fv + K.cy - v;
  return r0 * r0 + r1 * r1;
}

// inverse of a symmetric positive definite 3x3 given as (h00,h01,h02,h11,h12,h22);
// returns false when a Cholesky pivot is not positive.  The three pivots go through rsqrt (one
// MUFU seed + Newton steps each) instead of three square roots and six divisions: this function
// runs once per point and pass in every build kernel, where it was 8 % of the issue slots.
// il (optional): the inverse Cholesky factor L^-1 = [i00 0 0; i10 i11 0; i20 i21 i22] as
// (i00, i10, i11, i20, i21, i22), H^-1 = L^-T L^-1.
__device__ __forceinline__ bool inv3_spd(const double h[6], double hi[6], double* il = nullptr) {
  const double l00s = h[0];
  if (!(l00s > 0.0)) return false;
  const double i00 = rsqrt(l00s);
  const double l10 = h[1] * i00, l20 = h[2] * i00;
  const double l11s = h[3] - l10 * l10;
  if (!(l11s > 0.0)) return false;
  const double i11 = rsqrt(l11s);
  const double l21 = (h[4] - l20 * l10) * i11;
  const double l22s = h[5] - l20 * l20 - l21 * l21;
  if (!(l22s > 0.0)) return false;
  const double i22 = rsqrt(l22s);
  // inverse of L (lower)
  const double i10 = -l10 * i00 * i11;
  const double i21 = -l21 * i11 * i22;
  const double i20 = -(l20 * i00 + l21 * i10) * i22;
  // H^-1 = L^-T L^-1
  hi[0] = i00 * i00 + i10 * i10 + i20 * i20;
  hi[1] = i10 * i11 + i20 * i21;
  hi[2] = i20 * i22;
  hi[3] = i11 * i11 + i21 * i21;
  hi[4] = i21 * i22;
  hi[5] = i22 * i22;
  if (il) {
    il[0] = i00; il[1] = i10; il[2] = i11;
    il[3] = i20; il[4] = i21; il[5] = i22;
  }
  return true;
}

__device__ __forceinline__ double clamp_diag(double d, double lo, double hi) {
  return fmin(fmax(d, lo), hi);
}

// atomic max on non-negative doubles through their bit pattern
__device__ __forceinline__ void atomic_max_nonneg(double* addr, double v) {
  atomicMax(reinterpret_cast<unsigned long long*>(addr),
            (unsigned long long)__double_as_longlong(v));
}

// LM bookkeeping shared by every BA kernel family (Ceres TrustRegionMinimizer +
// LevenbergMarquardtStrategy; SURVEY §8(a) row a12).
struct LMState {
  // accumulators, zeroed before every attempt
  double acc_cost2;   // sum r^2 at the candidate
  double acc_model;   // sum m.(r + m/2),  m = J*step
  double acc_step2;   // |delta|^2
  double acc_xcand2;  // |x + delta|^2
  double acc_cur2;    // sum r^2 at the current point (build pass)
  double acc_xcur2;   // |x|^2 (init pass)
  double acc_gmax;    // max |J^T r| (unscaled), bit-pattern max
  // trust-region state
  double cost, radius, decrease_factor, x_norm, gmax, initial_cost;
  int iteration, n_success, n_fail, invalid_run;
  int termination, done, solve_ok, cur;  // cur: which parameter buffer is current (0/1)
  int check_gradient;  // a step was just accepted: test gradient tolerance after the next build
  int pad;
  int blocks_done;     // CTAs of this window that finished the back-substitution pass
  int pad2;
};

__device__ __forceinline__ void lm_zero_acc(LMState* s) {
  s->acc_cost2 = s->acc_model = s->acc_step2 = s->acc_xcand2 = s->acc_cur2 = 0.0;
  s->acc_gmax = 0.0;
}

// One trust-region decision (after the candidate has been evaluated).
// Returns 1 if the step is accepted.
__device__ __forceinline__ int lm_decide(LMState* s, const lorb_ba_options& o) {
  s->iteration++;
  const bool finite_ok = s->solve_ok && isfinite(s->acc_model) && isfinite(s->acc_step2);
  const double model_cost_change = -s->acc_model;
  int accepted = 0;
  if (!finite_ok || !(model_cost_change > 0.0)) {
    // HandleInvalidStep
    s->invalid_run++;
    s->n_fail++;
    if (s->invalid_run >= o.max_consecutive_invalid_steps) {
      s->termination = LORB_BA_FAILURE;
      s->done = 1;
      return 0;
    }
    s->radius = s->radius / s->decrease_factor;
    s->decrease_factor *= 2.0;
  } else {
    s->invalid_run = 0;
    const double cand_cost = 0.5 * s->acc_cost2;
    const double step_norm = sqrt(s->acc_step2);
    if (step_norm <= o.parameter_tolerance * (s->x_norm + o.parameter_tolerance)) {
      s->termination = LORB_BA_CONV_PARAMETER;
      s->done = 1;
      return 0;
    }
    const double cost_change = s->cost - cand_cost;
    if (fabs(cost_change) <= o.function_tolerance * s->cost) {
      s->termination = LORB_BA_CONV_FUNCTION;
      s->done = 1;
      return 0;
    }
    const double rho = cost_change / model_cost_change;
    if (rho > o.min_relative_decrease) {
      accepted = 1;
      s->cost = cand_cost;
      s->x_norm = sqrt(s->acc_xcand2);
      s->n_success++;
      s->check_gradient = 1;
      const double t = 2.0 * rho - 1.0;
      s->radius = s->radius / fmax(1.0 / 3.0, 1.0 - t * t * t);
      s->radius = fmin(o.max_trust_region_radius, s->radius);
      s->decrease_factor = 2.0;
    } else {
      s->n_fail++;
      s->radius = s->radius / s->decrease_factor;
      s->decrease_factor *= 2.0;
    }
  }
  if (s->iteration >= o.max_num_iterations) {
    s->done = 1;  // termination stays NO_CONVERGENCE unless the gradient test fires
  } else if (s->radius < o.min_trust_region_radius) {
    s->termination = LORB_BA_CONV_RADIUS;
    s->done = 1;
  }
  return accepted;
}

}  // namespace lorb
