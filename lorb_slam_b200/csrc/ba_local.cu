// ba_local.cu — local bundle adjustment on sm_100a (general multi-CTA path).
//
// Replaces the Ceres solve inside BA::LocalPoseOptimization (reference
// src/bundle_adjust.cpp:207-330): PoseMPCost / MPCost residuals, trust-region
// Levenberg-Marquardt with Jacobi scaling, DENSE_SCHUR (SURVEY §8(a) a9-a12).
//
// Data layout in HBM (DESIGN.md §4): observations sorted by point (CSR
// pt_ptr), 12 B each (camera index, u, v); parameters fp64 SoA-by-block
// (cams[C][6], pts[P][3]) double-buffered (current / candidate); per camera a
// 36-double rotation block (R, dR/dw) rebuilt per linearisation.
// Off-diagonal blocks W = Jc^T Jp are never stored: the Schur products are
// formed from recomputed Jacobians (the 48 B/obs/iteration design of
// SURVEY §8(d)).
//
// One LM attempt = build (Jacobians, H_pp, g_p, H_cc, g_c, Schur products)
//                -> [allreduce when sharded] -> finish (damping, mirror, rhs)
//                -> dense Cholesky + solve -> candidate cameras
//                -> back-substitution + model decrease + candidate cost
//                -> [allreduce] -> control (accept / reject, radius update).
// The trust-region state lives on the device; the host only enqueues.
#include <stdlib.h>

#include <omp.h>

#include <algorithm>
#include <chrono>
#include <new>
#include <vector>

#include <cub/cub.cuh>

#include "ba_math.cuh"
#include "dist.cuh"

namespace lorb {

constexpr int BA_THREADS = 256;
constexpr int HCC = 21;  // upper triangle of a 6x6 block

struct BADev {
  int C, P, n;  // n = 6C
  double* cams[2];
  double* pts[2];
  double* camrot[2];     // C x 36
  const int* pt_ptr;     // P+1
  const int* obs_cam;    // >=0 window camera; <0: fixed observation -1-f
  const float2* obs_uv;
  const double* fixrt;   // F x 12: R (9) + t (3) of out-of-window observers
  Intr K;
  double* scale_c;       // 6C
  double* scale_p;       // 3P
  double* lin;           // [S n*n (or Sp, packed) | Hcc 21C | gc 6C | rhs_corr 6C | tail 8 | gslot 16]
  double* S;             // dense n x n reduced camera system (what the Cholesky factorises)
  double* Sp;            // large path: packed upper block triangle the Schur products accumulate into
                         // (block row ci: 6 rows of 6 (C - ci) doubles); nullptr = S lives in lin
  double* gslot;         // [16] per-rank gradient maxima of a sharded solve (one sum all-reduce gathers them)
  int rank, world;       // of the sharded solve (0, 1 otherwise)
  double* Hcc;
  double* gc;
  double* rhs_corr;
  double* tail;          // acc_cur2, acc_xcur2, bad, spare
  double* rhs;           // n (becomes y_c after the solve)
  double* dinv;          // 1/L_jj of the Cholesky factor, padded to ceil(n/32)*32 (blocked path)
  double* pt_hinv;       // P x 6
  double* pt_gp;         // P x 3
  LMState* st;
  // large path only: camera-major / block-pair-major work lists (host built)
  const int* obs_pt;      // point of each observation (point-sorted observation order)
  const int2* cam_obs;    // (observation, its point) grouped by camera
  const int4* cam_items;  // (camera, start in cam_obs, length, 0)
  const int4* pairs;      // (point, observation i, observation j, 0) grouped by camera block
  const int4* pair_items; // (ci, cj, start in pairs, length)
  int n_cam_items, n_pair_items;
  int loss_kind;         // LORB_LOSS_* of the solve (read by the ROBUST kernel instantiations only)
  double loss_scale;
};

__device__ __forceinline__ int upper_idx(int a, int b) {  // a <= b, 6x6
  return a * 6 - (a * (a - 1)) / 2 + (b - a);
}

// Packed upper block triangle of the reduced camera system: element (a, b) of block (ci, cj), ci <= cj.
__device__ __forceinline__ size_t packed_idx(int C, int ci, int a, int cj, int b) {
  const size_t base = 36 * ((size_t)ci * C - (size_t)ci * (ci - 1) / 2);
  return base + (size_t)a * (6 * (C - ci)) + 6 * (cj - ci) + b;
}

// Largest |gradient| entry of the point side: this rank's own maximum, or, in a sharded solve,
// the maximum over the per-rank slots that the sum all-reduce of `lin` has gathered.
__device__ __forceinline__ double point_gmax(const BADev& p, const LMState* st) {
  double g = st->acc_gmax;
  if (p.world > 1)
    for (int r = 0; r < p.world && r < 16; r++) g = fmax(g, p.gslot[r]);
  return g;
}

// Sharded solve: publish this rank's maximum in its slot before the all-reduce.
__global__ void ba_gslot_kernel(const BADev* __restrict__ probs) {
  const BADev p = probs[0];
  if (p.world > 1 && p.rank < 16) p.gslot[p.rank] = p.st->acc_gmax;
}

__global__ void ba_camrot_kernel(const BADev* __restrict__ probs, int which /*0 = current, 1 = candidate*/, int force) {
  const BADev p = probs[blockIdx.y];
  LMState* st = p.st;
  if (st->done && !force) return;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= p.C) return;
  const int buf = st->cur ^ which;
  cam_rotation(p.cams[buf] + 6 * c, p.camrot[buf] + CAMROT * c, true);
}

// Observation of point X by window camera `cam` (>= 0) at pixel uv, with scaled Jacobians.
// ROBUST: r and the Jacobians come out corrected by the solve's loss (robust_correct) and *rho, when
// given, receives rho(|r|^2); the kernels are instantiated with ROBUST = false for plain least
// squares, which keeps that path exactly the code it was.
template <bool ROBUST = false>
__device__ __forceinline__ void eval_obs_cam(const BADev& p, const double* __restrict__ cams,
                                             const double* __restrict__ camrot, int cam, float2 uv,
                                             const double X[3], const double sp[3], double r[2], double Jc[12],
                                             double Jp[6], double* rho = nullptr) {
  const double* t = cams + 6 * cam + 3;
  const double tt[3] = {t[0], t[1], t[2]};
  obs_eval<true, true>(camrot + CAMROT * cam, tt, X, p.K, (double)uv.x, (double)uv.y, r, Jc, Jp);
  const double* sc = p.scale_c + 6 * cam;
#pragma unroll
  for (int a = 0; a < 6; a++) {
    Jc[a] *= sc[a];
    Jc[6 + a] *= sc[a];
  }
#pragma unroll
  for (int a = 0; a < 3; a++) {
    Jp[a] *= sp[a];
    Jp[3 + a] *= sp[a];
  }
  if (ROBUST) {
    const double q = robust_correct(p.loss_kind, p.loss_scale, r, Jc, Jp);
    if (rho) *rho = q;
  }
}

// Evaluate observation `o` of point X with scaled Jacobians (ROBUST, rho: as eval_obs_cam).
template <bool ROBUST = false>
__device__ __forceinline__ int eval_obs(const BADev& p, const double* __restrict__ cams,
                                        const double* __restrict__ camrot, int o, const double X[3],
                                        const double sp[3], double r[2], double Jc[12],
                                        double Jp[6], double* rho = nullptr) {
  const int cam = p.obs_cam[o];
  const float2 uv = p.obs_uv[o];
  if (cam >= 0) {
    eval_obs_cam<ROBUST>(p, cams, camrot, cam, uv, X, sp, r, Jc, Jp, rho);
    return cam;
  }
  const double* f = p.fixrt + 12 * (size_t)(-1 - cam);
  const double tt[3] = {f[9], f[10], f[11]};
  obs_eval<false, true>(f, tt, X, p.K, (double)uv.x, (double)uv.y, r, Jc, Jp);
#pragma unroll
  for (int a = 0; a < 3; a++) {
    Jp[a] *= sp[a];
    Jp[3 + a] *= sp[a];
  }
  if (ROBUST) {
    const double q = robust_correct(p.loss_kind, p.loss_scale, r, nullptr, Jp);
    if (rho) *rho = q;
  }
  return cam;
}

// Small windows keep their cameras in shared memory: the lanes of a warp evaluate observations of
// up to 32 different (point, camera) pairs, so every load of camera data from global memory costs
// one L1 wavefront per distinct camera (ncu: l1tex 50 % busy on 45 such loads per observation).
// Layout per camera, CS_BUILD doubles: [0,36) R and dR, [36,39) t, [39,45) Jacobi scale; the
// back-substitution appends [45,51) the camera step, [51,60) R and [60,63) t of the candidate.  Both
// strides are odd, so 16 consecutive cameras start on distinct even banks: a warp-wide load of a
// window of <= 16 cameras is conflict free (lanes on the same camera broadcast).  The dense build
// has at most 10 cameras; the back-substitution takes any window whose cameras fit twice per SM
// (config 5: 200 cameras, 100 KB, a few-way bank conflict instead of one L1 wavefront per camera).
constexpr int CS_BUILD = 45, CS_BACKSUB = 63, CS_MAX_CAMS = 16;

__device__ __forceinline__ void cs_fill(const BADev& p, const double* __restrict__ cams,
                                        const double* __restrict__ camrot, double* __restrict__ cs, int stride,
                                        int tid, int nthreads) {
  for (int i = tid; i < p.C * CS_BUILD; i += nthreads) {
    const int c = i / CS_BUILD, k = i - c * CS_BUILD;
    cs[c * stride + k] = k < 36 ? camrot[CAMROT * c + k] : k < 39 ? cams[6 * c + 3 + (k - 36)] : p.scale_c[6 * c + (k - 39)];
  }
}

// eval_obs with the window's cameras in shared memory (same arithmetic, same order).
template <bool ROBUST = false>
__device__ __forceinline__ int eval_obs_cs(const BADev& p, const double* __restrict__ cs, int stride, int o,
                                           const double X[3], const double sp[3], double r[2], double Jc[12],
                                           double Jp[6], double* rho = nullptr) {
  const int cam = p.obs_cam[o];
  const float2 uv = p.obs_uv[o];
  if (cam >= 0) {
    const double* cc = cs + cam * stride;
    const double tt[3] = {cc[36], cc[37], cc[38]};
    obs_eval<true, true>(cc, tt, X, p.K, (double)uv.x, (double)uv.y, r, Jc, Jp);
#pragma unroll
    for (int a = 0; a < 6; a++) {
      Jc[a] *= cc[39 + a];
      Jc[6 + a] *= cc[39 + a];
    }
  } else {
    const double* f = p.fixrt + 12 * (size_t)(-1 - cam);
    const double tt[3] = {f[9], f[10], f[11]};
    obs_eval<false, true>(f, tt, X, p.K, (double)uv.x, (double)uv.y, r, Jc, Jp);
  }
#pragma unroll
  for (int a = 0; a < 3; a++) {
    Jp[a] *= sp[a];
    Jp[3 + a] *= sp[a];
  }
  if (ROBUST) {
    const double q = robust_correct(p.loss_kind, p.loss_scale, r, cam >= 0 ? Jc : nullptr, Jp);
    if (rho) *rho = q;
  }
  return cam;
}

// Candidate cost of one observation with squared residual norm s: rho(s) under the solve's loss.
template <bool ROBUST>
__device__ __forceinline__ double obs_rho(const BADev& p, double s) {
  if (!ROBUST) return s;
  double rho, rho1;
  loss_eval(p.loss_kind, p.loss_scale, s, rho, rho1);
  return rho;
}

// |g_a / s_a| of the unscaled point gradient, coordinate a = lane of the point's group: the three
// divisions run on three lanes at once (the maximum over lanes is taken at the end of the kernel).
__device__ __forceinline__ double point_grad_abs(const double g[3], const double sp[3], int a) {
  const double ga = a == 0 ? g[0] : a == 1 ? g[1] : g[2];
  const double sa = a == 0 ? sp[0] : a == 1 ? sp[1] : sp[2];
  return fabs(ga / sa);
}

// Start a line on its way into L1 without holding a register for it (the consumer is a few
// hundred instructions later and the kernels below sit at their register cap).
__device__ __forceinline__ void prefetch_l1(const void* ptr) {
  asm volatile("prefetch.global.L1 [%0];" ::"l"(ptr));
}

__device__ __forceinline__ double group_sum8(double v) {
  v += __shfl_xor_sync(0xffffffffu, v, 4, 8);
  v += __shfl_xor_sync(0xffffffffu, v, 2, 8);
  v += __shfl_xor_sync(0xffffffffu, v, 1, 8);
  return v;
}

__device__ __forceinline__ double block_sum(double v, double* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double t = 0;
  if (threadIdx.x == 0)
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) t += red[w];
  return t;  // valid on thread 0
}

__device__ __forceinline__ double block_max(double v, double* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double t = 0;
  if (threadIdx.x == 0)
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) t = fmax(t, red[w]);
  return t;
}

// Build pass.  Eight lanes per point, one observation per lane per round.
// FULL = false: initial pass (scales are 1): cost, H_cc / g_c, point column
// norms -> scale_p, |x|^2, gradient max.  FULL = true: one LM attempt.
// Accumulation strategy of the build pass (template ACC):
//   0  global fp64 atomics straight into `lin` (many cameras: addresses are spread)
//   1  windows with n = 6C <= 96: every block of such a window hits the same few
//      hundred H_cc / S addresses and same-address fp64 atomics serialise in L2
//      (profiles/r01_ba_local_launches_before_opt.csv), so each CTA accumulates
//      into a private copy of `lin` in shared memory and flushes it once
//   3  many cameras (n > 96, BASELINE config 5): this kernel only does the
//      point side (H_pp, g_p, damped inverse, cost); the camera side runs in
//      ba_cam_rows_kernel and the Schur products in ba_schur_pairs_kernel, both
//      segmented reductions in registers over host-built lists - no atomics in
//      any inner loop
//   (n <= 64 with unique (point, camera) pairs - the 10-keyframe windows of BASELINE
//   configs 3/4 - do not come here: ba_build_dense_kernel below.)
constexpr int DENSE_N = 64;   // padded reduced-system size of the dense path
constexpr int DENSE_DS = 68;  // row stride (doubles) of the Y / W tiles: == 4 mod 16, so the four k-rows of
                              // a DMMA fragment load (lanes: k = lane % 4, row = lane / 4) hit 16 distinct banks
constexpr int DENSE_RC = 16;  // padded camera count of the residual tile

// D (8x8, fp64) += A (8x4, row) * B (4x8, col) on the tensor cores (SASS DMMA).  Fragments:
// a = A[lane/4][lane%4], b = B[lane%4][lane/4], c0/c1 = C[lane/4][2*(lane%4) + 0/1].
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

template <bool FULL, int ACC, bool ROBUST = false>
__global__ void __launch_bounds__(BA_THREADS)
    ba_build_kernel(const BADev* __restrict__ probs, lorb_ba_options opt, int force) {
  const BADev p = probs[blockIdx.y];
  LMState* st = p.st;
  if (st->done && !force) return;
  __shared__ int Csm[BA_THREADS];
  __shared__ double red[BA_THREADS / 32];
  extern __shared__ __align__(16) double dsm[];
  // dynamic shared memory carve-up
  //   ACC 0: [Wsm 256x18]   ACC 1: [lin copy][Wsm 256x18]
  const int lin_n = p.n * p.n + (HCC + 12) * p.C;
  double* slin = dsm;
  double (*Wsm)[18] = reinterpret_cast<double (*)[18]>(ACC == 1 ? dsm + lin_n : dsm);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, gl = lane & 7, gw = lane >> 3;
  if (ACC == 1) {
    for (int i = tid; i < lin_n; i += BA_THREADS) slin[i] = 0.0;
    __syncthreads();
  }
  double* const accS = ACC == 1 ? slin : p.S;
  double* const accH = ACC == 1 ? slin + (size_t)p.n * p.n : p.Hcc;
  double* const accG = accH + HCC * p.C;
  double* const accR = accG + 6 * p.C;
  const int cur = st->cur;
  const double* cams = p.cams[cur];
  const double* pts = p.pts[cur];
  const double* camrot = p.camrot[cur];
  const double radius = st->radius, inv_radius = 1.0 / radius;  // one division per kernel, not three per point
  const int n = p.n;
  double cost_acc = 0, gmax_acc = 0, xn_acc = 0, bad_acc = 0;
  for (int blk = blockIdx.x * (BA_THREADS / 8); blk < p.P; blk += gridDim.x * (BA_THREADS / 8)) {
    const int pt = blk + warp * 4 + gw;
    const int slot = warp * 4 + gw;
    const bool pv = pt < p.P;
    int s = 0, e = 0;
    double X[3] = {0, 0, 0}, sp[3] = {1, 1, 1};
    if (pv) {
      s = p.pt_ptr[pt];
      e = p.pt_ptr[pt + 1];
#pragma unroll
      for (int a = 0; a < 3; a++) {
        X[a] = pts[3 * (size_t)pt + a];
        sp[a] = p.scale_p[3 * (size_t)pt + a];
      }
    }
    const int rounds = __reduce_max_sync(0xffffffffu, (e - s + 7) >> 3);
    // ---- phase 1: H_pp, g_p, H_cc, g_c, cost
    double h[6] = {0, 0, 0, 0, 0, 0}, g[3] = {0, 0, 0};
    double r[2], Jc[12], Jp[6];
    int cam = -1;
    bool has = false;
    for (int rd = 0; rd < rounds; rd++) {
      const int o = s + rd * 8 + gl;
      has = o < e;
      if (has) {
        double rho;
        cam = eval_obs<ROBUST>(p, cams, camrot, o, X, sp, r, Jc, Jp, &rho);
        cost_acc += ROBUST ? rho : r[0] * r[0] + r[1] * r[1];
        h[0] += Jp[0] * Jp[0] + Jp[3] * Jp[3];
        h[1] += Jp[0] * Jp[1] + Jp[3] * Jp[4];
        h[2] += Jp[0] * Jp[2] + Jp[3] * Jp[5];
        h[3] += Jp[1] * Jp[1] + Jp[4] * Jp[4];
        h[4] += Jp[1] * Jp[2] + Jp[4] * Jp[5];
        h[5] += Jp[2] * Jp[2] + Jp[5] * Jp[5];
#pragma unroll
        for (int a = 0; a < 3; a++) g[a] += Jp[a] * r[0] + Jp[3 + a] * r[1];
        if (ACC != 3 && cam >= 0) {
          double* H = accH + HCC * (size_t)cam;
          int k = 0;
#pragma unroll
          for (int a = 0; a < 6; a++) {
#pragma unroll
            for (int c2 = a; c2 < 6; c2++) atomicAdd(&H[k++], Jc[a] * Jc[c2] + Jc[6 + a] * Jc[6 + c2]);
            atomicAdd(&accG[6 * cam + a], Jc[a] * r[0] + Jc[6 + a] * r[1]);
          }
        }
      }
    }
#pragma unroll
    for (int a = 0; a < 6; a++) h[a] = group_sum8(h[a]);
#pragma unroll
    for (int a = 0; a < 3; a++) g[a] = group_sum8(g[a]);
    if (!FULL) {
      if (pv && gl == 0) {
        if (opt.jacobi_scaling && force == 1) {
          p.scale_p[3 * (size_t)pt + 0] = 1.0 / (1.0 + sqrt(h[0]));
          p.scale_p[3 * (size_t)pt + 1] = 1.0 / (1.0 + sqrt(h[3]));
          p.scale_p[3 * (size_t)pt + 2] = 1.0 / (1.0 + sqrt(h[5]));
        }
        xn_acc += X[0] * X[0] + X[1] * X[1] + X[2] * X[2];
      }
      // gradient of the unscaled problem (this pass may run with scales already set)
      if (pv && gl < 3) gmax_acc = fmax(gmax_acc, point_grad_abs(g, sp, gl));
      continue;
    }
    if (pv && gl < 3) gmax_acc = fmax(gmax_acc, point_grad_abs(g, sp, gl));
    // LM diagonal on the scaled columns, clamped (LevenbergMarquardtStrategy)
    double hd[6] = {h[0], h[1], h[2], h[3], h[4], h[5]}, hi[6];
    hd[0] += clamp_diag(h[0], opt.min_lm_diagonal, opt.max_lm_diagonal) * inv_radius;
    hd[3] += clamp_diag(h[3], opt.min_lm_diagonal, opt.max_lm_diagonal) * inv_radius;
    hd[5] += clamp_diag(h[5], opt.min_lm_diagonal, opt.max_lm_diagonal) * inv_radius;
    const bool ok = inv3_spd(hd, hi);
    if (pv && gl == 0) {
      if (!ok) bad_acc += 1.0;
#pragma unroll
      for (int a = 0; a < 6; a++) p.pt_hinv[6 * (size_t)pt + a] = ok ? hi[a] : 0.0;
#pragma unroll
      for (int a = 0; a < 3; a++) p.pt_gp[3 * (size_t)pt + a] = g[a];
    }
    if (!ok) {
#pragma unroll
      for (int a = 0; a < 6; a++) hi[a] = 0.0;
    }
    // ---- phase 2: Schur products  S -= W_i Hinv W_j^T ,  rhs_corr += W_i Hinv g_p
    if (ACC == 3) continue;  // done by ba_cam_rows_kernel / ba_schur_pairs_kernel
    for (int ri = 0; ri < rounds; ri++) {
      const int oi = s + ri * 8 + gl;
      const bool has_i = oi < e;
      int ci = -1;
      double Wi[18], Yi[18];
      if (rounds > 1 || ri > 0) {
        if (has_i) ci = eval_obs<ROBUST>(p, cams, camrot, oi, X, sp, r, Jc, Jp);
      } else {
        ci = has ? cam : -1;  // single round: Jacobians of phase 1 are still live
      }
      const bool act_i = has_i && ci >= 0;
      if (act_i) {
#pragma unroll
        for (int a = 0; a < 6; a++)
#pragma unroll
          for (int c2 = 0; c2 < 3; c2++) Wi[3 * a + c2] = Jc[a] * Jp[c2] + Jc[6 + a] * Jp[3 + c2];
#pragma unroll
        for (int a = 0; a < 6; a++) {
          const double w0 = Wi[3 * a], w1 = Wi[3 * a + 1], w2 = Wi[3 * a + 2];
          Yi[3 * a + 0] = w0 * hi[0] + w1 * hi[1] + w2 * hi[2];
          Yi[3 * a + 1] = w0 * hi[1] + w1 * hi[3] + w2 * hi[4];
          Yi[3 * a + 2] = w0 * hi[2] + w1 * hi[4] + w2 * hi[5];
          atomicAdd(&accR[6 * ci + a],
                    Yi[3 * a] * g[0] + Yi[3 * a + 1] * g[1] + Yi[3 * a + 2] * g[2]);
        }
      }
      for (int rj = 0; rj < rounds; rj++) {
        if (rj == ri) {
          Csm[tid] = act_i ? ci : -1;
          if (act_i) {
#pragma unroll
            for (int a = 0; a < 18; a++) Wsm[tid][a] = Wi[a];
          }
        } else {
          const int oj = s + rj * 8 + gl;
          int cj = -1;
          if (oj < e) {
            double r2[2], Jc2[12], Jp2[6];
            cj = eval_obs<ROBUST>(p, cams, camrot, oj, X, sp, r2, Jc2, Jp2);
            if (cj >= 0) {
#pragma unroll
              for (int a = 0; a < 6; a++)
#pragma unroll
                for (int c2 = 0; c2 < 3; c2++)
                  Wsm[tid][3 * a + c2] = Jc2[a] * Jp2[c2] + Jc2[6 + a] * Jp2[3 + c2];
            }
          }
          Csm[tid] = cj;
        }
        __syncwarp();
        for (int j = 0; j < 8; j++) {
          const int src = (tid & ~7) + j;
          const int cj = Csm[src];
          // upper block triangle only (finish mirrors); equal cameras keep both orders
          if (act_i && cj >= ci) {
            const double* Wj = Wsm[src];
            double* Sblk = accS + (size_t)(6 * ci) * n + 6 * cj;
#pragma unroll
            for (int a = 0; a < 6; a++)
#pragma unroll
              for (int c2 = 0; c2 < 6; c2++) {
                const double v = Yi[3 * a] * Wj[3 * c2] + Yi[3 * a + 1] * Wj[3 * c2 + 1] +
                                 Yi[3 * a + 2] * Wj[3 * c2 + 2];
                atomicAdd(&Sblk[(size_t)a * n + c2], -v);
              }
          }
        }
        __syncwarp();
      }
    }
  }
  if (ACC == 1) {
    __syncthreads();
    for (int i = tid; i < lin_n; i += BA_THREADS) {
      const double v = slin[i];
      if (v != 0.0) atomicAdd(&p.lin[i], v);
    }
  }
  double t = block_sum(cost_acc, red);
  if (tid == 0 && t != 0.0) atomicAdd(&p.tail[0], t);
  t = block_sum(xn_acc, red);
  if (tid == 0 && t != 0.0) atomicAdd(&p.tail[1], t);
  t = block_sum(bad_acc, red);
  if (tid == 0 && t != 0.0) atomicAdd(&p.tail[2], t);
  t = block_max(gmax_acc, red);
  if (tid == 0 && t > 0.0) atomic_max_nonneg(&st->acc_gmax, t);
}

// ---- dense path, n = 6C <= 64 and unique (point, camera) pairs (BASELINE configs 3 / 4).
// H_cc, g_c, the Schur right-hand side and the Schur products of a window are dense contractions
// over its points.  The CTA is three independent GROUPS of four warps; a group owns 16 points per
// round and keeps private dense tiles of them in shared memory:
//     J  [32 x 64]  rows (point slot, residual component), columns camera parameters
//     R  [32 x 16]  residual of that row per camera
//     Z = L^-1 W^T  [48 x 64]  rows (point slot, point coordinate), H_pp^-1 = L^-T L^-1
// After one 128-thread named barrier the group contracts its own tiles on the fp64 tensor cores
// (DMMA m8n8k4): S_group += Z^T Z (= W H_pp^-1 W^T) as 36 upper 8x8 tiles (10 / 10 / 8 / 8 per
// warp, compile-time lists; both fragments of a tile pair come from the same loads: 4 or 6 per
// k-step) and H_cc += J^T J on the 13 tiles that meet a 6x6 diagonal block; g_c is a column dot
// product per thread, the Schur right-hand side comes out of the same contraction (L^-1 g_p sits in
// a spare column of Z).  Four warps per group instead of two (round 2): a warp carries 24-26
// accumulator doubles instead of 50, which brings the kernel from 255 registers and 8 warps per SM
// to <= 168 and 12.  A second group
// barrier, then every lane clears exactly what it stored.  No block-wide barrier and no atomic
// in the round loop; the pairs are reduced through shared memory once at the end and the CTA
// flushes one partial result.
constexpr int DENSE_RHS_COL = 60;         // 6C <= 64 means C <= 10: columns 60..63 of the tiles are never a camera's
static_assert(DENSE_N == 64 && DENSE_RHS_COL >= (DENSE_N / 6) * 6 && DENSE_RHS_COL < DENSE_N, "spare column");
constexpr int DP_GW = 4;                  // warps per point group
constexpr int DP_PTS = 4 * DP_GW;         // points per group and round
constexpr int DP_KW = 3 * DP_PTS;         // rows of the Z tile
constexpr int DP_KJ = 2 * DP_PTS;         // rows of the J / R tiles
constexpr int DP_GROUP = DP_KW * DENSE_DS + DP_KJ * DENSE_DS + DP_KJ * DENSE_RC;  // doubles
constexpr int DP_THREADS = 384;           // 3 groups of 4 warps: 12 warps per SM at <= 168 registers
constexpr int DP_NGROUP = DP_THREADS / (32 * DP_GW);
constexpr int DP_SMEM_DOUBLES = DP_NGROUP * DP_GROUP;
static_assert(DP_GROUP % 2 == 0 && DENSE_DS % 2 == 0 && (DP_KW * DENSE_DS) % 2 == 0, "128-bit tile stores stay aligned");
static_assert(DP_SMEM_DOUBLES >= DENSE_N * DENSE_N + HCC * 10 + 2 * DENSE_N + 16, "reduction buffer fits");

__device__ __forceinline__ void group_barrier(int grp) {
  asm volatile("bar.sync %0, %1;" ::"r"(grp + 1), "n"(32 * DP_GW) : "memory");
}

// Upper 8x8 tiles of the 64x64 product, split between the four warps of a group: the two diagonal
// 4x4 tile blocks (10 upper tiles each, 4 distinct fragments per k-step) and the two halves of the
// off-diagonal block (8 tiles, 6 fragments); the 13 tiles of J^T J that meet a 6x6 diagonal block
// (block boundaries 24 and 48 are tile aligned) go 2 / 2 / 5 / 4, which evens out the DMMA counts.
template <int Q>
struct DenseTiles {
  static constexpr int NS = Q < 2 ? 10 : 8;
  static constexpr int NH = Q < 2 ? 2 : (Q == 2 ? 5 : 4);
  __device__ static constexpr int si(int t) {
    constexpr int a[4][10] = {{0, 0, 0, 0, 1, 1, 1, 2, 2, 3}, {4, 4, 4, 4, 5, 5, 5, 6, 6, 7},
                              {0, 0, 0, 0, 1, 1, 1, 1, 0, 0}, {2, 2, 2, 2, 3, 3, 3, 3, 0, 0}};
    return a[Q][t];
  }
  __device__ static constexpr int sj(int t) {
    constexpr int a[4][10] = {{0, 1, 2, 3, 1, 2, 3, 2, 3, 3}, {4, 5, 6, 7, 5, 6, 7, 6, 7, 7},
                              {4, 5, 6, 7, 4, 5, 6, 7, 0, 0}, {4, 5, 6, 7, 4, 5, 6, 7, 0, 0}};
    return a[Q][t];
  }
  __device__ static constexpr int hi(int t) {
    constexpr int a[4][5] = {{0, 1, 0, 0, 0}, {4, 5, 0, 0, 0}, {0, 1, 2, 3, 3}, {4, 6, 6, 7, 0}};
    return a[Q][t];
  }
  __device__ static constexpr int hj(int t) {
    constexpr int a[4][5] = {{0, 1, 0, 0, 0}, {4, 5, 0, 0, 0}, {1, 2, 2, 3, 4}, {5, 6, 7, 7, 0}};
    return a[Q][t];
  }
};
constexpr int DP_NS_MAX = 10, DP_NH_MAX = 5;

template <int Q, bool FULL>
__device__ __forceinline__ void dense_contract(const double* __restrict__ Zt,
                                               const double* __restrict__ Jt, int lane,
                                               double (&sacc)[DP_NS_MAX][2], double (&hacc)[DP_NH_MAX][2]) {
  using T = DenseTiles<Q>;
  const int fo = (lane & 3) * DENSE_DS + (lane >> 2);
#pragma unroll
  for (int k0 = 0; k0 < DP_KJ; k0 += 4) {
    double f[8];
#pragma unroll
    for (int i = 0; i < 8; i++) f[i] = Jt[fo + k0 * DENSE_DS + 8 * i];  // unused ones are eliminated
#pragma unroll
    for (int t = 0; t < T::NH; t++) dmma884(hacc[t][0], hacc[t][1], f[T::hi(t)], f[T::hj(t)]);
  }
  if (FULL) {
#pragma unroll
    for (int k0 = 0; k0 < DP_KW; k0 += 4) {
      double z[8];  // Z^T Z: the A and the B fragment of a tile pair are the same loads
#pragma unroll
      for (int i = 0; i < 8; i++) z[i] = Zt[fo + k0 * DENSE_DS + 8 * i];
#pragma unroll
      for (int t = 0; t < T::NS; t++) dmma884(sacc[t][0], sacc[t][1], z[T::si(t)], z[T::sj(t)]);
    }
  }
}

// Adds this warp's accumulators into the CTA's reduction buffers (called by one group at a time;
// the four warps of a group own disjoint tiles).
template <int Q, bool FULL>
__device__ __forceinline__ void dense_reduce(double* __restrict__ Sbuf, double* __restrict__ Hbuf, int lane,
                                             int n, const double (&sacc)[DP_NS_MAX][2],
                                             const double (&hacc)[DP_NH_MAX][2]) {
  using T = DenseTiles<Q>;
#pragma unroll
  for (int t = 0; t < T::NH; t++)
#pragma unroll
    for (int q = 0; q < 2; q++) {
      const int row = 8 * T::hi(t) + (lane >> 2), col = 8 * T::hj(t) + 2 * (lane & 3) + q;
      if (col < n && row / 6 == col / 6 && row <= col)
        Hbuf[HCC * (row / 6) + upper_idx(row % 6, col % 6)] += hacc[t][q];
    }
  if (FULL) {
#pragma unroll
    for (int t = 0; t < T::NS; t++)
#pragma unroll
      for (int q = 0; q < 2; q++) {
        const int row = 8 * T::si(t) + (lane >> 2), col = 8 * T::sj(t) + 2 * (lane & 3) + q;
        Sbuf[row * DENSE_N + col] += sacc[t][q];
      }
  }
}

template <bool FULL, bool ROBUST = false>
__global__ void __launch_bounds__(DP_THREADS)
    ba_build_dense_kernel(const BADev* __restrict__ probs, lorb_ba_options opt, int force) {
  const BADev p = probs[blockIdx.y];
  LMState* st = p.st;
  if (st->done && !force) return;
  __shared__ double red[DP_THREADS / 32];
  __shared__ double cs[CS_MAX_CAMS * CS_BUILD];  // the window's cameras (6C <= 64: at most 10)
  extern __shared__ __align__(16) double dsm[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, gl = lane & 7, gw = lane >> 3;
  const int grp = warp / DP_GW, q = warp % DP_GW, gtid = tid % (32 * DP_GW);
  double* const Zt = dsm + grp * DP_GROUP;
  double* const Jt = Zt + DP_KW * DENSE_DS;
  double* const Rt = Jt + DP_KJ * DENSE_DS;
  for (int i = tid; i < DP_SMEM_DOUBLES; i += DP_THREADS) dsm[i] = 0.0;
  __syncthreads();
  const int cur = st->cur;
  const double* cams = p.cams[cur];
  const double* pts = p.pts[cur];
  const double* camrot = p.camrot[cur];
  const double radius = st->radius, inv_radius = 1.0 / radius;  // one division per kernel, not three per point
  const int n = p.n;
  cs_fill(p, cams, camrot, cs, CS_BUILD, tid, DP_THREADS);
  __syncthreads();
  double cost_acc = 0, gmax_acc = 0, xn_acc = 0, bad_acc = 0;
  double sacc[DP_NS_MAX][2], hacc[DP_NH_MAX][2], gown = 0.0;
#pragma unroll
  for (int t = 0; t < DP_NS_MAX; t++) sacc[t][0] = sacc[t][1] = 0.0;
#pragma unroll
  for (int t = 0; t < DP_NH_MAX; t++) hacc[t][0] = hacc[t][1] = 0.0;
  const int ps = q * 4 + gw;  // point slot inside the group
  const int gcol = gtid & 63, grow0 = (gtid >> 6) * (DP_KJ / 2);  // g_c: a column and half of the J rows per thread
  // block-uniform trip count (group barriers inside)
  for (int blk = blockIdx.x * (DP_THREADS / 8); blk < p.P; blk += gridDim.x * (DP_THREADS / 8)) {
    const int pt = blk + warp * 4 + gw;
    const bool pv = pt < p.P;
    int s = 0, e = 0;
    double X[3] = {0, 0, 0}, sp[3] = {1, 1, 1};
    if (pv) {
      s = p.pt_ptr[pt];
      e = p.pt_ptr[pt + 1];
#pragma unroll
      for (int a = 0; a < 3; a++) {
        X[a] = pts[3 * (size_t)pt + a];
        sp[a] = p.scale_p[3 * (size_t)pt + a];
      }
    }
    const int rounds = __reduce_max_sync(0xffffffffu, (e - s + 7) >> 3);
    // ---- phase 1: Jacobians -> J / R tiles, H_pp, g_p, cost
    double h[6] = {0, 0, 0, 0, 0, 0}, g[3] = {0, 0, 0};
    double r[2], Jc[12], Jp[6];
    int cam = -1;
    bool has = false;
    for (int rd = 0; rd < rounds; rd++) {
      const int o = s + rd * 8 + gl;
      has = o < e;
      if (has) {
        double rho;
        cam = eval_obs_cs<ROBUST>(p, cs, CS_BUILD, o, X, sp, r, Jc, Jp, &rho);
        cost_acc += ROBUST ? rho : r[0] * r[0] + r[1] * r[1];
        h[0] += Jp[0] * Jp[0] + Jp[3] * Jp[3];
        h[1] += Jp[0] * Jp[1] + Jp[3] * Jp[4];
        h[2] += Jp[0] * Jp[2] + Jp[3] * Jp[5];
        h[3] += Jp[1] * Jp[1] + Jp[4] * Jp[4];
        h[4] += Jp[1] * Jp[2] + Jp[4] * Jp[5];
        h[5] += Jp[2] * Jp[2] + Jp[5] * Jp[5];
#pragma unroll
        for (int a = 0; a < 3; a++) g[a] += Jp[a] * r[0] + Jp[3 + a] * r[1];
        if (cam >= 0) {
#pragma unroll
          for (int comp = 0; comp < 2; comp++) {
#pragma unroll
            for (int a = 0; a < 6; a += 2)  // a camera's six columns start 16-byte aligned: 128-bit stores
              *reinterpret_cast<double2*>(&Jt[(ps * 2 + comp) * DENSE_DS + 6 * cam + a]) =
                  make_double2(Jc[6 * comp + a], Jc[6 * comp + a + 1]);
            Rt[(ps * 2 + comp) * DENSE_RC + cam] = r[comp];
          }
        }
      }
    }
#pragma unroll
    for (int a = 0; a < 6; a++) h[a] = group_sum8(h[a]);
#pragma unroll
    for (int a = 0; a < 3; a++) g[a] = group_sum8(g[a]);
    if (pv && gl < 3) gmax_acc = fmax(gmax_acc, point_grad_abs(g, sp, gl));
    if (!FULL) {
      if (pv && gl == 0) {
        if (opt.jacobi_scaling && force == 1) {
          p.scale_p[3 * (size_t)pt + 0] = 1.0 / (1.0 + sqrt(h[0]));
          p.scale_p[3 * (size_t)pt + 1] = 1.0 / (1.0 + sqrt(h[3]));
          p.scale_p[3 * (size_t)pt + 2] = 1.0 / (1.0 + sqrt(h[5]));
        }
        xn_acc += X[0] * X[0] + X[1] * X[1] + X[2] * X[2];
      }
    } else {
      // LM diagonal on the scaled columns, clamped (LevenbergMarquardtStrategy)
      double hd[6] = {h[0], h[1], h[2], h[3], h[4], h[5]}, hi[6];
      hd[0] += clamp_diag(h[0], opt.min_lm_diagonal, opt.max_lm_diagonal) * inv_radius;
      hd[3] += clamp_diag(h[3], opt.min_lm_diagonal, opt.max_lm_diagonal) * inv_radius;
      hd[5] += clamp_diag(h[5], opt.min_lm_diagonal, opt.max_lm_diagonal) * inv_radius;
      double il[6];
      const bool ok = inv3_spd(hd, hi, il);
      if (pv && gl == 0) {
        if (!ok) bad_acc += 1.0;
#pragma unroll
        for (int a = 0; a < 6; a++) p.pt_hinv[6 * (size_t)pt + a] = ok ? hi[a] : 0.0;
#pragma unroll
        for (int a = 0; a < 3; a++) p.pt_gp[3 * (size_t)pt + a] = g[a];
      }
      if (!ok) {
#pragma unroll
        for (int a = 0; a < 6; a++) il[a] = 0.0;
      }
      // ---- phase 2: Z_i = L^-1 W_i^T into the group's tile (H_pp^-1 = L^-T L^-1, so the Schur
      // product W H_pp^-1 W^T of the point is Z^T Z: one tile, contracted with itself).
      // L^-1 g_p rides in the spare column DENSE_RHS_COL: the contraction then leaves the Schur
      // right-hand side W H_pp^-1 g_p in that column of the product (rewritten every round: never cleared)
      if (gl == 0) {
        const double g0 = pv ? g[0] : 0.0, g1 = pv ? g[1] : 0.0, g2 = pv ? g[2] : 0.0;
        Zt[(ps * 3 + 0) * DENSE_DS + DENSE_RHS_COL] = il[0] * g0;
        Zt[(ps * 3 + 1) * DENSE_DS + DENSE_RHS_COL] = il[1] * g0 + il[2] * g1;
        Zt[(ps * 3 + 2) * DENSE_DS + DENSE_RHS_COL] = il[3] * g0 + il[4] * g1 + il[5] * g2;
      }
      for (int ri = 0; ri < rounds; ri++) {
        const int oi = s + ri * 8 + gl;
        const bool has_i = oi < e;
        int ci = -1;
        if (rounds > 1) {
          if (has_i) ci = eval_obs_cs<ROBUST>(p, cs, CS_BUILD, oi, X, sp, r, Jc, Jp);
        } else {
          ci = has ? cam : -1;  // single round: the Jacobians of phase 1 are still live
        }
        if (has_i && ci >= 0) {
#pragma unroll
          for (int a = 0; a < 6; a += 2) {  // two columns at a time: 128-bit stores
            double w[2][3];
#pragma unroll
            for (int q = 0; q < 2; q++) {
              w[q][0] = Jc[a + q] * Jp[0] + Jc[6 + a + q] * Jp[3];
              w[q][1] = Jc[a + q] * Jp[1] + Jc[6 + a + q] * Jp[4];
              w[q][2] = Jc[a + q] * Jp[2] + Jc[6 + a + q] * Jp[5];
            }
            const int col = 6 * ci + a;
            *reinterpret_cast<double2*>(&Zt[(ps * 3 + 0) * DENSE_DS + col]) =
                make_double2(il[0] * w[0][0], il[0] * w[1][0]);
            *reinterpret_cast<double2*>(&Zt[(ps * 3 + 1) * DENSE_DS + col]) =
                make_double2(il[1] * w[0][0] + il[2] * w[0][1], il[1] * w[1][0] + il[2] * w[1][1]);
            *reinterpret_cast<double2*>(&Zt[(ps * 3 + 2) * DENSE_DS + col]) =
                make_double2(il[3] * w[0][0] + il[4] * w[0][1] + il[5] * w[0][2],
                             il[3] * w[1][0] + il[4] * w[1][1] + il[5] * w[1][2]);
          }
        }
      }
    }
    group_barrier(grp);
    // ---- contractions over the group's 16 points
    switch (q) {
      case 0: dense_contract<0, FULL>(Zt, Jt, lane, sacc, hacc); break;
      case 1: dense_contract<1, FULL>(Zt, Jt, lane, sacc, hacc); break;
      case 2: dense_contract<2, FULL>(Zt, Jt, lane, sacc, hacc); break;
      default: dense_contract<3, FULL>(Zt, Jt, lane, sacc, hacc); break;
    }
    if (gcol < n) {  // g_c: one column and half of the rows per thread of the group
      const int c2 = gcol / 6;
      double a2 = 0;
#pragma unroll
      for (int k2 = 0; k2 < DP_KJ / 2; k2++)
        a2 += Jt[(grow0 + k2) * DENSE_DS + gcol] * Rt[(grow0 + k2) * DENSE_RC + c2];
      gown += a2;
    }
    group_barrier(grp);
    // ---- clear exactly what this lane stored
    for (int ri = 0; ri < rounds; ri++) {
      const int oi = s + ri * 8 + gl;
      if (oi < e) {
        const int ci = p.obs_cam[oi];
        if (ci >= 0) {
#pragma unroll
          for (int a = 0; a < 6; a += 2) {
            const double2 z = make_double2(0.0, 0.0);
            *reinterpret_cast<double2*>(&Jt[(ps * 2 + 0) * DENSE_DS + 6 * ci + a]) = z;
            *reinterpret_cast<double2*>(&Jt[(ps * 2 + 1) * DENSE_DS + 6 * ci + a]) = z;
            if (FULL) {
#pragma unroll
              for (int c2 = 0; c2 < 3; c2++)
                *reinterpret_cast<double2*>(&Zt[(ps * 3 + c2) * DENSE_DS + 6 * ci + a]) = z;
            }
          }
          Rt[(ps * 2 + 0) * DENSE_RC + ci] = 0.0;
          Rt[(ps * 2 + 1) * DENSE_RC + ci] = 0.0;
        }
      }
    }
  }
  // ---- reduce the four pairs through shared memory, flush once per CTA
  __syncthreads();
  double* const Sbuf = dsm;                        // 64 x 64
  double* const Hbuf = Sbuf + DENSE_N * DENSE_N;   // 21 per camera
  double* const Gbuf = Hbuf + HCC * 10 + 6;        // g_c
  for (int i = tid; i < DENSE_N * DENSE_N + HCC * 10 + 6 + 2 * DENSE_N; i += DP_THREADS) dsm[i] = 0.0;
  __syncthreads();
  for (int pp = 0; pp < 2 * DP_NGROUP; pp++) {  // (group, row half of the g_c partials)
    if (grp == (pp >> 1)) {
      if ((pp & 1) == 0) {
        switch (q) {
          case 0: dense_reduce<0, FULL>(Sbuf, Hbuf, lane, n, sacc, hacc); break;
          case 1: dense_reduce<1, FULL>(Sbuf, Hbuf, lane, n, sacc, hacc); break;
          case 2: dense_reduce<2, FULL>(Sbuf, Hbuf, lane, n, sacc, hacc); break;
          default: dense_reduce<3, FULL>(Sbuf, Hbuf, lane, n, sacc, hacc); break;
        }
      }
      if (gcol < n && (gtid >> 6) == (pp & 1)) Gbuf[gcol] += gown;
    }
    __syncthreads();
  }
  for (int i = tid; i < HCC * p.C; i += DP_THREADS)
    if (Hbuf[i] != 0.0) atomicAdd(&p.Hcc[i], Hbuf[i]);
  if (tid < n) {
    if (Gbuf[tid] != 0.0) atomicAdd(&p.gc[tid], Gbuf[tid]);
    const double rc = FULL ? Sbuf[tid * DENSE_N + DENSE_RHS_COL] : 0.0;
    if (FULL && rc != 0.0) atomicAdd(&p.rhs_corr[tid], rc);
  }
  if (FULL) {
    for (int i = tid; i < DENSE_N * DENSE_N; i += DP_THREADS) {
      const int row = i / DENSE_N, col = i % DENSE_N;
      const double v = Sbuf[i];
      if (row >= n || col >= n || v == 0.0) continue;
      // diagonal and upper camera blocks only (the solve mirrors the rest).  Only upper TILES were
      // computed: a tile that cuts through a 6x6 diagonal block supplies that block's lower
      // entries by symmetry of W H^-1 W^T.
      if (col / 6 >= row / 6) atomicAdd(&p.S[(size_t)row * n + col], -v);
      if (row / 8 != col / 8 && col / 6 == row / 6) atomicAdd(&p.S[(size_t)col * n + row], -v);
    }
  }
  double t = block_sum(cost_acc, red);
  if (tid == 0 && t != 0.0) atomicAdd(&p.tail[0], t);
  t = block_sum(xn_acc, red);
  if (tid == 0 && t != 0.0) atomicAdd(&p.tail[1], t);
  t = block_sum(bad_acc, red);
  if (tid == 0 && t != 0.0) atomicAdd(&p.tail[2], t);
  t = block_max(gmax_acc, red);
  if (tid == 0 && t > 0.0) atomic_max_nonneg(&st->acc_gmax, t);
}

// ---- large path, camera side.  Work item = (camera, slice of its observation
// list): one warp accumulates H_cc (21), g_c (6) and the Schur right-hand side
// W H_pp^-1 g_p (6) of its slice in registers, reduces by shuffles and issues 33
// atomics per item.
template <bool ROBUST = false>
__global__ void __launch_bounds__(256)
    ba_cam_rows_kernel(const BADev* __restrict__ probs, int full, int force) {
  const BADev p = probs[blockIdx.y];
  LMState* st = p.st;
  if (st->done && !force) return;
  const int lane = threadIdx.x & 31;
  const int item = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (item >= p.n_cam_items) return;
  const int4 it = p.cam_items[item];  // camera, start, length
  const int cur = st->cur;
  const double* cams = p.cams[cur];
  const double* pts = p.pts[cur];
  const double* camrot = p.camrot[cur];
  double acc[33];
#pragma unroll
  for (int a = 0; a < 33; a++) acc[a] = 0.0;
  // records are streamed one step ahead so that only one gather level (the point's data) is exposed
  int2 rec = lane < it.z ? p.cam_obs[it.y + lane] : make_int2(0, 0);
  for (int e = lane; e < it.z; e += 32) {
    const int o = rec.x, pt = rec.y;
    if (e + 32 < it.z) rec = p.cam_obs[it.y + e + 32];
    const float2 uv = p.obs_uv[o];
    double X[3], sp[3], r[2], Jc[12], Jp[6];
#pragma unroll
    for (int a = 0; a < 3; a++) {
      X[a] = pts[3 * (size_t)pt + a];
      sp[a] = p.scale_p[3 * (size_t)pt + a];
    }
    eval_obs_cam<ROBUST>(p, cams, camrot, it.x, uv, X, sp, r, Jc, Jp);
    int k = 0;
#pragma unroll
    for (int a = 0; a < 6; a++) {
#pragma unroll
      for (int c2 = a; c2 < 6; c2++) acc[k++] += Jc[a] * Jc[c2] + Jc[6 + a] * Jc[6 + c2];
      acc[21 + a] += Jc[a] * r[0] + Jc[6 + a] * r[1];
    }
    if (full) {
      const double* hi = p.pt_hinv + 6 * (size_t)pt;
      const double* gp = p.pt_gp + 3 * (size_t)pt;
      // t = Hinv g_p ; rhs_corr += W t = Jc^T (Jp t)
      const double t0 = hi[0] * gp[0] + hi[1] * gp[1] + hi[2] * gp[2];
      const double t1 = hi[1] * gp[0] + hi[3] * gp[1] + hi[4] * gp[2];
      const double t2 = hi[2] * gp[0] + hi[4] * gp[1] + hi[5] * gp[2];
      const double q0 = Jp[0] * t0 + Jp[1] * t1 + Jp[2] * t2;
      const double q1 = Jp[3] * t0 + Jp[4] * t1 + Jp[5] * t2;
#pragma unroll
      for (int a = 0; a < 6; a++) acc[27 + a] += Jc[a] * q0 + Jc[6 + a] * q1;
    }
  }
#pragma unroll
  for (int a = 0; a < 33; a++) {
    double v = acc[a];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    acc[a] = v;
  }
  if (lane == 0) {
    const int cam = it.x;
#pragma unroll
    for (int a = 0; a < 21; a++) atomicAdd(&p.Hcc[HCC * (size_t)cam + a], acc[a]);
#pragma unroll
    for (int a = 0; a < 6; a++) {
      atomicAdd(&p.gc[6 * cam + a], acc[21 + a]);
      if (full) atomicAdd(&p.rhs_corr[6 * cam + a], acc[27 + a]);
    }
  }
}

// ---- large path, Schur products.  Work item = (camera block (ci,cj), slice of
// the pair records of that block); a record is (observation i, observation j)
// of one point with camera(i) = ci, camera(j) = cj.  One warp accumulates
// sum Y_i W_j^T (6x6) in registers over its slice, reduces by shuffles and
// subtracts it from S with 36 atomics per item (an item is <= 2048 records).
template <bool ROBUST = false>
__global__ void __launch_bounds__(256)
    ba_schur_pairs_kernel(const BADev* __restrict__ probs) {
  const BADev p = probs[blockIdx.y];
  LMState* st = p.st;
  if (st->done) return;
  const int lane = threadIdx.x & 31;
  const int item = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (item >= p.n_pair_items) return;
  const int4 it = p.pair_items[item];  // ci, cj, start, length
  const int cur = st->cur;
  const double* cams = p.cams[cur];
  const double* pts = p.pts[cur];
  const double* camrot = p.camrot[cur];
  double acc[36];
#pragma unroll
  for (int a = 0; a < 36; a++) acc[a] = 0.0;
  // records are streamed one step ahead: only the gathers of the point's data and the two pixels
  // (one level, all independent) are exposed per step
  int4 rec = lane < it.w ? p.pairs[it.z + lane] : make_int4(0, 0, 0, 0);
  for (int e = lane; e < it.w; e += 32) {
    const int pt = rec.x, oi = rec.y, oj = rec.z;
    if (e + 32 < it.w) rec = p.pairs[it.z + e + 32];
    const float2 uvi = p.obs_uv[oi], uvj = p.obs_uv[oj];
    double X[3], sp[3], r[2], Jc[12], Jp[6], Y[18];
#pragma unroll
    for (int a = 0; a < 3; a++) {
      X[a] = pts[3 * (size_t)pt + a];
      sp[a] = p.scale_p[3 * (size_t)pt + a];
    }
    const double* hi = p.pt_hinv + 6 * (size_t)pt;
    const double h0 = hi[0], h1 = hi[1], h2 = hi[2], h3 = hi[3], h4 = hi[4], h5 = hi[5];
    eval_obs_cam<ROBUST>(p, cams, camrot, it.x, uvi, X, sp, r, Jc, Jp);
#pragma unroll
    for (int a = 0; a < 6; a++) {
      const double w0 = Jc[a] * Jp[0] + Jc[6 + a] * Jp[3];
      const double w1 = Jc[a] * Jp[1] + Jc[6 + a] * Jp[4];
      const double w2 = Jc[a] * Jp[2] + Jc[6 + a] * Jp[5];
      Y[3 * a + 0] = w0 * h0 + w1 * h1 + w2 * h2;
      Y[3 * a + 1] = w0 * h1 + w1 * h3 + w2 * h4;
      Y[3 * a + 2] = w0 * h2 + w1 * h4 + w2 * h5;
    }
    if (oj != oi) eval_obs_cam<ROBUST>(p, cams, camrot, it.y, uvj, X, sp, r, Jc, Jp);
#pragma unroll
    for (int b = 0; b < 6; b++) {
      const double w0 = Jc[b] * Jp[0] + Jc[6 + b] * Jp[3];
      const double w1 = Jc[b] * Jp[1] + Jc[6 + b] * Jp[4];
      const double w2 = Jc[b] * Jp[2] + Jc[6 + b] * Jp[5];
#pragma unroll
      for (int a = 0; a < 6; a++) acc[6 * a + b] += Y[3 * a] * w0 + Y[3 * a + 1] * w1 + Y[3 * a + 2] * w2;
    }
  }
#pragma unroll
  for (int a = 0; a < 36; a++) {
    double v = acc[a];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    acc[a] = v;
  }
  if (lane == 0) {
    // block (ci, cj), ci <= cj, of the packed upper block triangle (or of the dense matrix)
    double* Sblk = p.Sp ? p.Sp + packed_idx(p.C, it.x, 0, it.y, 0) : p.S + (size_t)(6 * it.x) * p.n + 6 * it.y;
    const size_t ld = p.Sp ? (size_t)6 * (p.C - it.x) : (size_t)p.n;
#pragma unroll
    for (int a = 0; a < 6; a++)
#pragma unroll
      for (int b = 0; b < 6; b++) atomicAdd(&Sblk[(size_t)a * ld + b], -acc[6 * a + b]);
  }
}

// After the initial pass: camera column scales, |x|, cost, gradient test.
__global__ void ba_init_finish_kernel(const BADev* __restrict__ probs, lorb_ba_options opt) {
  const BADev p = probs[blockIdx.y];
  LMState* st = p.st;
  __shared__ double red[32];
  double xn = 0, gm = 0;
  for (int i = threadIdx.x; i < p.n; i += blockDim.x) {
    const int c = i / 6, a = i % 6;
    const double d = p.Hcc[HCC * (size_t)c + upper_idx(a, a)];
    gm = fmax(gm, fabs(p.gc[i]));
    if (opt.jacobi_scaling) p.scale_c[i] = 1.0 / (1.0 + sqrt(d));
    const double x = p.cams[st->cur][i];
    xn += x * x;
  }
  const double xs = block_sum(xn, red);
  const double gmx = block_max(gm, red);
  if (threadIdx.x == 0) {
    st->x_norm = sqrt(xs + p.tail[1]);
    st->cost = 0.5 * p.tail[0];
    st->initial_cost = st->cost;
    st->gmax = fmax(gmx, point_gmax(p, st));
    st->radius = opt.initial_trust_region_radius;
    st->decrease_factor = 2.0;
    st->iteration = st->n_success = st->n_fail = st->invalid_run = 0;
    st->termination = LORB_BA_NO_CONVERGENCE;
    st->done = 0;
    st->check_gradient = 0;
    st->solve_ok = 1;
    if (st->gmax <= opt.gradient_tolerance) {
      st->termination = LORB_BA_CONV_GRADIENT;
      st->done = 1;
    }
    if (opt.max_num_iterations <= 0) st->done = 1;
    lm_zero_acc(st);
  }
}

// Gradient-tolerance test of the point accepted by the previous attempt
// (Ceres checks it right after HandleSuccessfulStep; here the gradient only
// exists after the next build pass).  One CTA.
__global__ void ba_gradcheck_kernel(const BADev* __restrict__ probs, lorb_ba_options opt, int force) {
  const BADev p = probs[blockIdx.y];
  LMState* st = p.st;
  if (st->done && !force) return;
  __shared__ double red[32];
  double gm = 0;
  for (int i = threadIdx.x; i < p.n; i += blockDim.x) gm = fmax(gm, fabs(p.gc[i] / p.scale_c[i]));
  const double gmx = block_max(gm, red);
  if (threadIdx.x == 0 && st->check_gradient) {
    st->gmax = fmax(gmx, point_gmax(p, st));
    st->check_gradient = 0;
    if (st->gmax <= opt.gradient_tolerance) {
      st->termination = LORB_BA_CONV_GRADIENT;
      st->done = 1;
    }
  }
}

// S <- blockdiag(H_cc + D_c^2) + (Schur part, upper blocks mirrored); rhs = g_c - corr.
__global__ void ba_finish_kernel(const BADev* __restrict__ probs, lorb_ba_options opt) {
  const BADev p = probs[blockIdx.y];
  LMState* st = p.st;
  if (st->done) return;
  const int n = p.n;
  const double radius = st->radius, inv_radius = 1.0 / radius;  // one division per kernel, not three per point
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < (size_t)n * n;
       idx += (size_t)gridDim.x * blockDim.x) {
    const int i = (int)(idx / n), j = (int)(idx % n);
    const int ci = i / 6, cj = j / 6;
    if (p.Sp) {  // unpack (and mirror) the packed upper block triangle into the dense matrix
      const int a = i % 6, b = j % 6;
      double v = ci <= cj ? p.Sp[packed_idx(p.C, ci, a, cj, b)] : p.Sp[packed_idx(p.C, cj, b, ci, a)];
      if (ci == cj) {
        double h = p.Hcc[HCC * (size_t)ci + (a <= b ? upper_idx(a, b) : upper_idx(b, a))];
        if (a == b) h += clamp_diag(h, opt.min_lm_diagonal, opt.max_lm_diagonal) * inv_radius;
        v += h;
      }
      p.S[idx] = v;
    } else if (ci == cj) {
      const int a = i % 6, b = j % 6;
      double v = p.Hcc[HCC * (size_t)ci + (a <= b ? upper_idx(a, b) : upper_idx(b, a))];
      if (a == b) v += clamp_diag(v, opt.min_lm_diagonal, opt.max_lm_diagonal) * inv_radius;
      p.S[idx] += v;
    } else if (ci > cj) {
      p.S[idx] = p.S[(size_t)j * n + i];  // mirror the upper block triangle
    }
    if (j == 0) p.rhs[i] = p.gc[i] - p.rhs_corr[i];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) st->solve_ok = (p.tail[2] == 0.0) ? 1 : 0;
}

// ---- dense Cholesky (lower, in place) + solve.  Small systems: one CTA, matrix in smem.
__global__ void __launch_bounds__(256) ba_chol_small_kernel(const BADev* __restrict__ probs) {
  const BADev p = probs[blockIdx.y];
  LMState* st = p.st;
  if (st->done) return;
  extern __shared__ double A[];  // n*n + n
  __shared__ int s_ok;
  const int n = p.n, tid = threadIdx.x;
  double* b = A + (size_t)n * n;
  for (int i = tid; i < n * n; i += blockDim.x) A[i] = p.S[i];
  for (int i = tid; i < n; i += blockDim.x) b[i] = p.rhs[i];
  if (tid == 0) s_ok = 1;
  __syncthreads();
  for (int j = 0; j < n; j++) {
    if (tid == 0) {
      const double d = A[j * n + j];
      if (!(d > 0.0)) s_ok = 0;
      A[j * n + j] = sqrt(d > 0.0 ? d : 1.0);
    }
    __syncthreads();
    const double dj = A[j * n + j];
    for (int i = j + 1 + tid; i < n; i += blockDim.x) A[i * n + j] /= dj;
    __syncthreads();
    // trailing update of the lower triangle
    const int m = n - j - 1;
    for (int e = tid; e < m * m; e += blockDim.x) {
      const int i = j + 1 + e / m, k = j + 1 + e % m;
      if (k <= i) A[i * n + k] -= A[i * n + j] * A[k * n + j];
    }
    __syncthreads();
  }
  // forward / backward substitution by warp 0
  if (tid < 32) {
    for (int i = 0; i < n; i++) {
      double sacc = 0;
      for (int k = tid; k < i; k += 32) sacc += A[i * n + k] * b[k];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, o);
      if (tid == 0) b[i] = (b[i] - sacc) / A[i * n + i];
      __syncwarp();
    }
    for (int i = n - 1; i >= 0; i--) {
      double sacc = 0;
      for (int k = i + 1 + tid; k < n; k += 32) sacc += A[k * n + i] * b[k];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sacc += __shfl_xor_sync(0xffffffffu, sacc, o);
      if (tid == 0) b[i] = (b[i] - sacc) / A[i * n + i];
      __syncwarp();
    }
  }
  __syncthreads();
  for (int i = tid; i < n; i += blockDim.x) p.rhs[i] = b[i];
  if (tid == 0 && !s_ok) st->solve_ok = 0;
}

constexpr int NB = 32;  // tile size of the dense factorisations

// The same two warp-level tile operations on a shared-memory matrix with leading dimension ld that
// keeps L transposed in its upper triangle (L_ij, i > j, at M[j*ld + i]; dg[j] = 1 / L_jj): the
// layout of ba_solve_small_kernel.  kn / rn < 32 pad with identity / zero rows.
__device__ __forceinline__ void potrf_tile_ld(double* M, int ld, int k0, int kn, double* dg, int* s_ok, int lane) {
  double a[NB];
#pragma unroll
  for (int c = 0; c < NB; c++)
    a[c] = (lane < kn && c < kn) ? M[(size_t)(k0 + lane) * ld + k0 + c] : (c == lane ? 1.0 : 0.0);
#pragma unroll
  for (int c = 0; c < NB; c++) {
    double d = __shfl_sync(0xffffffffu, a[c], c);
    if (!(d > 0.0)) {
      if (lane == 0) *s_ok = 0;
      d = 1.0;
    }
    const double is = rsqrt(d);
    const double l = a[c] * is;
    a[c] = l;
    if (lane == c && c < kn) dg[k0 + c] = is;
#pragma unroll
    for (int q = c + 1; q < NB; q++) {
      const double lq = __shfl_sync(0xffffffffu, l, q);
      a[q] -= l * lq;
    }
  }
#pragma unroll
  for (int c = 0; c < NB; c++)
    if (lane > c && lane < kn) M[(size_t)(k0 + c) * ld + k0 + lane] = a[c];
}

// rows r0 .. r0+rn of the panel below the diagonal tile at k0: X L_kk^T = A_rk
__device__ __forceinline__ void trsm_tile_ld(double* M, int ld, int r0, int rn, int k0, int kn, const double* dg,
                                             int lane) {
  double a[NB];
#pragma unroll
  for (int c = 0; c < NB; c++) a[c] = (lane < rn && c < kn) ? M[(size_t)(r0 + lane) * ld + k0 + c] : 0.0;
#pragma unroll
  for (int m = 0; m < NB; m++) {
    if (m < kn) {  // uniform
      const double x = a[m] * dg[k0 + m];
      a[m] = x;
#pragma unroll
      for (int c = m + 1; c < NB; c++)
        if (c < kn) a[c] -= x * M[(size_t)(k0 + m) * ld + k0 + c];  // L_cm, broadcast
    }
  }
#pragma unroll
  for (int c = 0; c < NB; c++)
    if (lane < rn && c < kn) M[(size_t)(k0 + c) * ld + r0 + lane] = a[c];
}

// Small windows: one CTA does everything between the build pass and the
// back-substitution: gradient-tolerance test, assembly of the damped reduced
// camera system in shared memory, Cholesky, both triangular solves, candidate
// cameras and their rotation blocks.  L is kept transposed in the (unused) upper
// triangle so a column step needs a single barrier.
__global__ void __launch_bounds__(256)
    ba_solve_small_kernel(const BADev* __restrict__ probs, lorb_ba_options opt) {
  const BADev p = probs[blockIdx.y];
  LMState* st = p.st;
  if (st->done) return;
  extern __shared__ double A[];  // n*n | b[n] | diag[n] | tmp[32] | Linv[nb][32][33]
  __shared__ double red[8];
  __shared__ int s_ok, s_done;
  const int n = p.n, tid = threadIdx.x;
  double* b = A + (size_t)n * n;
  double* dg = b + n;
  double* tmp = dg + n;
  double* Linv = tmp + NB;  // inverses of the diagonal tiles of L (lower triangular, [tile][r][c], stride 33)
  // gradient tolerance of the point accepted by the previous attempt
  double gm = 0;
  for (int i = tid; i < n; i += blockDim.x) gm = fmax(gm, fabs(p.gc[i] / p.scale_c[i]));
  const double gmx = block_max(gm, red);
  if (tid == 0) {
    s_done = 0;
    s_ok = (p.tail[2] == 0.0) ? 1 : 0;
    if (st->check_gradient) {
      st->gmax = fmax(gmx, point_gmax(p, st));
      st->check_gradient = 0;
      if (st->gmax <= opt.gradient_tolerance) {
        st->termination = LORB_BA_CONV_GRADIENT;
        st->done = 1;
        s_done = 1;
      }
    }
  }
  __syncthreads();
  if (s_done) return;
  const double radius = st->radius, inv_radius = 1.0 / radius;  // one division per kernel, not three per point
  // (the loads of four elements per thread are issued together: the loop was one exposed L2
  //  round trip per element, 8.5 us of the 50 us this kernel took)
  for (int base = 0; base < n * n; base += 4 * 256) {
    double vs[4], vh[4];
    int dcase[4];  // 0 off-diagonal block, 1 diagonal block, 2 diagonal element
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const int idx = base + tid + 256 * q;
      vs[q] = vh[q] = 0.0;
      dcase[q] = -1;
      if (idx < n * n) {
        const int i = idx / n, j = idx % n;
        const int ci = i / 6, cj = j / 6;
        if (ci == cj) {
          const int a2 = i % 6, c2 = j % 6;
          vh[q] = p.Hcc[HCC * (size_t)ci + (a2 <= c2 ? upper_idx(a2, c2) : upper_idx(c2, a2))];
          vs[q] = p.S[idx];
          dcase[q] = a2 == c2 ? 2 : 1;
        } else {
          vs[q] = ci < cj ? p.S[idx] : p.S[(size_t)j * n + i];
          dcase[q] = 0;
        }
      }
    }
#pragma unroll
    for (int q = 0; q < 4; q++) {
      const int idx = base + tid + 256 * q;
      if (dcase[q] < 0) continue;
      double v = vs[q] + vh[q];
      if (dcase[q] == 2) v += clamp_diag(vh[q], opt.min_lm_diagonal, opt.max_lm_diagonal) * inv_radius;
      A[idx] = v;
    }
  }
  for (int i = tid; i < n; i += blockDim.x) b[i] = p.gc[i] - p.rhs_corr[i];
  __syncthreads();
  // Blocked right-looking Cholesky on 32-wide tiles: the diagonal tile by warp 0 and each panel
  // tile by one warp, both with the tile in registers (no barrier inside), then the trailing
  // update by the whole CTA: 3 block barriers per tile column instead of one per column.
  {
    const int lane = tid & 31, warp = tid >> 5;
    const int nb = (n + NB - 1) / NB;
    for (int kb = 0; kb < nb; kb++) {
      const int k0 = kb * NB, kn = min(NB, n - k0);
      if (warp == 0) potrf_tile_ld(A, n, k0, kn, dg, &s_ok, lane);
      __syncthreads();
      const int rb = kb + warp;  // warps 1.. take the panel tiles below
      if (warp >= 1 && rb < nb) trsm_tile_ld(A, n, rb * NB, min(NB, n - rb * NB), k0, kn, dg, lane);
      __syncthreads();
      const int t0 = k0 + NB, tn = max(0, n - t0);  // trailing block (lower triangle incl. diagonal)
      for (int idx = tid; idx < tn * tn; idx += 256) {
        const int r = idx / tn, q = idx % tn;
        if (q > r) continue;
        double acc = 0;
#pragma unroll 8
        for (int m = 0; m < kn; m++) acc += A[(k0 + m) * n + t0 + r] * A[(k0 + m) * n + t0 + q];
        A[(t0 + r) * n + t0 + q] -= acc;
      }
      __syncthreads();
    }
  }
  // Triangular solves without a per-column dependency chain: warps 0..nb-1 invert the diagonal
  // tiles of L (lane c solves L x = e_c with the column in registers; L_rm is a shared-memory
  // broadcast), then warp 0 runs both substitutions block-wise as matrix-vector products:
  // y_k = Linv_kk (b_k - sum_{j<k} L_kj y_j),  x_k = Linv_kk^T (y_k - sum_{i>k} L_ik^T x_i).
  // (The register-vector column sweep this replaces took 24 k cycles of the kernel's 98 k.)
  {
    const int lane = tid & 31, warp = tid >> 5;
    const int nb = (n + NB - 1) / NB;
    if (warp < nb) {
      const int k0 = warp * NB, kn = min(NB, n - k0);
      double x[NB];
#pragma unroll
      for (int r = 0; r < NB; r++) {
        double acc = (r == lane) ? 1.0 : 0.0;
        if (r < kn) {
#pragma unroll
          for (int m = 0; m < r; m++) acc -= A[(size_t)(k0 + m) * n + k0 + r] * x[m];  // L_rm
          x[r] = acc * dg[k0 + r];
        } else {
          x[r] = 0.0;
        }
      }
#pragma unroll
      for (int r = 0; r < NB; r++) Linv[(warp * NB + r) * (NB + 1) + lane] = x[r];
    }
    __syncthreads();
    if (warp == 0) {
      for (int kb = 0; kb < nb; kb++) {  // forward
        const int k0 = kb * NB, kn = min(NB, n - k0);
        double t = 0.0;
        if (lane < kn) {
          t = b[k0 + lane];
          for (int j = 0; j < k0; j++) t -= A[(size_t)j * n + k0 + lane] * b[j];  // L_{k0+lane, j} y_j
        }
        tmp[lane] = t;
        __syncwarp();
        double y = 0.0;
#pragma unroll 8
        for (int c2 = 0; c2 < NB; c2++) y += Linv[(kb * NB + lane) * (NB + 1) + c2] * tmp[c2];
        __syncwarp();
        if (lane < kn) b[k0 + lane] = y;
        __syncwarp();
      }
      for (int kb = nb - 1; kb >= 0; kb--) {  // backward
        const int k0 = kb * NB, kn = min(NB, n - k0);
        double t = 0.0;
        if (lane < kn) {
          t = b[k0 + lane];
          for (int i = k0 + NB; i < n; i++) t -= A[(size_t)(k0 + lane) * n + i] * b[i];  // L_{i, k0+lane} x_i
        }
        tmp[lane] = t;
        __syncwarp();
        double xv = 0.0;
#pragma unroll 8
        for (int c2 = 0; c2 < NB; c2++) xv += Linv[(kb * NB + c2) * (NB + 1) + lane] * tmp[c2];
        __syncwarp();
        if (lane < kn) b[k0 + lane] = xv;
        __syncwarp();
      }
    }
  }
  __syncthreads();
  // candidate cameras + rotation blocks
  const int cur = st->cur;
  double step2 = 0, xc2 = 0;
  for (int i = tid; i < n; i += blockDim.x) {
    p.rhs[i] = b[i];
    const double dlt = -b[i] * p.scale_c[i];
    const double x = p.cams[cur][i] + dlt;
    p.cams[cur ^ 1][i] = x;
    step2 += dlt * dlt;
    xc2 += x * x;
  }
  const double s2 = block_sum(step2, red);
  const double x2 = block_sum(xc2, red);
  if (tid == 0) {
    p.tail[3] = s2;
    p.tail[4] = x2;
    st->solve_ok = s_ok;
  }
  __syncthreads();
  for (int c = tid; c < p.C; c += blockDim.x)
    cam_rotation(p.cams[cur ^ 1] + 6 * c, p.camrot[cur ^ 1] + CAMROT * c, true);
}

// Large systems: right-looking blocked Cholesky in global memory, NB = 32.

// Panel: every CTA factors the 32x32 diagonal block in shared memory with all
// 256 threads (one barrier per column, rsqrt instead of sqrt + divides; L_ij,
// i>j, is kept transposed at D[j][i]); CTA 0 writes L_kk and 1/L_jj, CTA b>0
// solves its 32-row block  X L_kk^T = A_ik  with 8 threads per row.
__global__ void __launch_bounds__(NB * NB / 4)
    ba_chol_panel_kernel(const BADev* __restrict__ probs, int kb) {
  const BADev p = probs[blockIdx.y];
  LMState* st = p.st;
  if (st->done) return;
  __shared__ double D[NB][NB + 1];
  __shared__ double X[NB][NB + 1];
  __shared__ double idg[NB];  // 1 / L_jj
  __shared__ int s_ok;
  const int n = p.n, tid = threadIdx.x;
  const int k0 = kb * NB, kn = min(NB, n - k0);
  if (k0 >= n || (kb + (int)blockIdx.x) * NB >= n) return;
  const int ib = kb + blockIdx.x;
  const int i0 = ib * NB, in = min(NB, n - i0);
  for (int e = tid; e < NB * NB; e += blockDim.x) {
    const int i = e / NB, j = e % NB;
    D[i][j] = (i < kn && j < kn) ? p.S[(size_t)(k0 + i) * n + k0 + j] : (i == j ? 1.0 : 0.0);
    X[i][j] = (blockIdx.x > 0 && i < in && j < kn) ? p.S[(size_t)(i0 + i) * n + k0 + j] : 0.0;
  }
  if (tid == 0) s_ok = 1;
  __syncthreads();
  const int ty = tid >> 4, tx = tid & 15;
  for (int j = 0; j < NB; j++) {
    double d = D[j][j];
    if (!(d > 0.0)) {
      if (tid == 0) s_ok = 0;
      d = 1.0;
    }
    const double is = rsqrt(d), inv_d = is * is;
    if (tid == 0) idg[j] = is;
    if (tid > j && tid < NB) D[j][tid] = D[tid][j] * is;  // L_ij at [j][i]
    for (int i = j + 1 + ty; i < NB; i += 16) {
      const double aij = D[i][j] * inv_d;
      for (int k = j + 1 + tx; k <= i; k += 16) D[i][k] -= aij * D[k][j];
    }
    __syncthreads();
  }
  if (blockIdx.x == 0) {
    for (int e = tid; e < NB * NB; e += blockDim.x) {
      const int i = e / NB, j = e % NB;
      if (i < kn && j < i) p.S[(size_t)(k0 + i) * n + k0 + j] = D[j][i];
    }
    if (tid < NB) {
      if (tid < kn) p.S[(size_t)(k0 + tid) * n + k0 + tid] = 1.0 / idg[tid];
      p.dinv[(size_t)kb * NB + tid] = idg[tid];
    }
    if (tid == 0 && !s_ok) st->solve_ok = 0;
    return;
  }
  // row r (8 threads): x_c = (a_c - sum_{m<c} x_m L_cm) / L_cc ,  L_cm = D[m][c]
  {
    const int r = tid >> 3, sub = tid & 7;
    for (int c = 0; c < NB; c++) {
      double part = 0;
      for (int m = sub; m < c; m += 8) part += X[r][m] * D[m][c];
      part += __shfl_xor_sync(0xffffffffu, part, 4);
      part += __shfl_xor_sync(0xffffffffu, part, 2);
      part += __shfl_xor_sync(0xffffffffu, part, 1);
      if (sub == 0) X[r][c] = (X[r][c] - part) * idg[c];
      __syncwarp();
    }
  }
  __syncthreads();
  for (int e = tid; e < NB * NB; e += blockDim.x) {
    const int i = e / NB, j = e % NB;
    if (i < in && j < kn) p.S[(size_t)(i0 + i) * n + k0 + j] = X[i][j];
  }
}

// 32x32 POTRF by ONE warp with the tile in registers (lane = row, fully unrolled): per column one
// broadcast of the pivot, rsqrt, and 31-c shuffle + FMA pairs; no barriers.  The 256-thread
// shared-memory version took 11.3 us per tile on the critical path of the dataflow factorisation
// (globaltimer trace, profiles/README.md); this one is bound by ~150 dependent cycles per column.
// In: A[r][c] (lower part valid).  Out: L_rc (r > c) at A[c][r], idg[c] = 1 / L_cc.
__device__ __forceinline__ void potrf32_warp(double (*A)[NB + 1], double* idg, int* s_ok, int lane) {
  double a[NB];
#pragma unroll
  for (int c = 0; c < NB; c++) a[c] = A[lane][c];
#pragma unroll
  for (int c = 0; c < NB; c++) {
    double d = __shfl_sync(0xffffffffu, a[c], c);
    if (!(d > 0.0)) {
      if (lane == 0) *s_ok = 0;
      d = 1.0;
    }
    const double is = rsqrt(d);
    const double l = a[c] * is;  // L_rc for r >= c
    a[c] = l;
    if (lane == c) idg[c] = is;
#pragma unroll
    for (int q = c + 1; q < NB; q++) {
      const double lq = __shfl_sync(0xffffffffu, l, q);  // L_qc
      a[q] -= l * lq;  // meaningful for r >= q; the unused upper part may hold anything
    }
  }
#pragma unroll
  for (int c = 0; c < NB; c++)
    if (lane > c) A[c][lane] = a[c];
}

// X L^T = A for one 32x32 tile by ONE warp (lane = row of X, registers, right-looking):
// B[m][c] = L_cm (m < c) is read as a shared-memory broadcast, idg[m] = 1 / L_mm.
__device__ __forceinline__ void trsm32_warp(double (*A)[NB + 1], const double (*B)[NB + 1], const double* idg,
                                            int lane) {
  double a[NB];
#pragma unroll
  for (int c = 0; c < NB; c++) a[c] = A[lane][c];
#pragma unroll
  for (int m = 0; m < NB; m++) {
    const double x = a[m] * idg[m];
    a[m] = x;
#pragma unroll
    for (int c = m + 1; c < NB; c++) a[c] -= x * B[m][c];
  }
#pragma unroll
  for (int c = 0; c < NB; c++) A[lane][c] = a[c];
}

__device__ __forceinline__ void flag_wait(const int* flag) {
  if (threadIdx.x == 0) {
    while (*reinterpret_cast<const volatile int*>(flag) == 0) {
    }
    __threadfence();
  }
  __syncthreads();
}

// ---- dataflow tiled Cholesky, chain form (n > 143, one window): ONE cooperative launch.
// The factorisation's critical path is POTRF(j) -> TRSM(j+1, j) -> last update of (j+1, j+1) ->
// POTRF(j+1).  With 32x32 tiles dealt round-robin to CTAs those three steps belong to three
// different CTAs, so a block column costs two publish / consume hops through global memory and two
// tile reloads on top of the arithmetic.  Here CTA 0 walks the whole chain with L_jj and L_(j+1)j
// staying in its shared memory, and every other CTA is a helper working through a list of items in
// column order:
//   * normal tiles (i, j), i >= j + 2: left-looking accumulation A_ij -= sum_{k<j} L_ik L_jk^T as
//     soon as both source tiles are flagged ready, then TRSM against L_jj;
//   * the "sub partial" of column j: S(j+1, j) - sum_{k<j} L(j+1, k) L(j, k)^T, left in place for
//     the chain CTA, which only has to apply L_jj^-T;
//   * the "diagonal partial" of block d = j + 1: S(d, d) - sum_{k<=d-2} L(d, k) L(d, k)^T and the
//     forward-substitution partial b_d - sum_{k<=d-2} L(d, k) y_k; the chain CTA subtracts the
//     k = d - 1 term, whose tile it has just produced itself.
// Item numbers grow with the column; an item depends only on smaller items and on chain output of
// earlier columns, the chain on partials of smaller items: no deadlock while all CTAs are resident.
__global__ void __launch_bounds__(256)
    ba_chol_chain_kernel(const BADev* __restrict__ probs, int* __restrict__ flags, int* __restrict__ yflag,
                         int* __restrict__ pflag /* [2T]: sub partial of column j, diagonal partial of block j */,
                         double* __restrict__ ypart /* [T][32] */, int T) {
  const BADev p = probs[0];
  LMState* st = p.st;
  if (st->done) return;
  __shared__ double A[NB][NB + 1];
  __shared__ double B[NB][NB + 1];
  __shared__ double X[NB][NB + 1];
  __shared__ double idg[NB];
  __shared__ double sk[NB], vec[NB];
  __shared__ int s_ok;
  const int n = p.n, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int ty = tid >> 4, tx = tid & 15;
  int* sflag = pflag;
  int* dflag = pflag + T;
  if (tid == 0) s_ok = 1;
  __syncthreads();
  auto publish = [&](int* f) {  // every thread has written its part: fence, barrier, one flag store
    __threadfence();
    __syncthreads();
    if (tid == 0) atomicExch(f, 1);
  };
  if (blockIdx.x == 0) {
    // ================= the chain
    __shared__ double Dn[NB][NB + 1];  // next diagonal partial, fetched by idle warps during POTRF
    __shared__ double skn[NB];
    __shared__ int have_next;  // halves of Dn fetched: warp 2 rows 0-15 and skn, warp 3 rows 16-31
    if (tid == 0) have_next = 0;
    __syncthreads();
    for (int j = 0; j < T; j++) {
      const int j0 = j * NB, s0 = (j + 1) * NB;
      // uniform: written before the last barrier of the previous column.  Warps 2 and 3 read the
      // partial's flag each on their own, so the prefetched tile is complete only when both counted in.
      const bool pre = have_next == 2;
      if (j >= 2 && !pre) flag_wait(&dflag[j]);
      // diagonal tile (partial) minus this CTA's own last term X X^T (X = L_j(j-1), still in X)
      double acc[2][2];
#pragma unroll
      for (int a = 0; a < 2; a++)
#pragma unroll
        for (int b = 0; b < 2; b++) {
          const int r = j0 + 2 * ty + a, c = j0 + 2 * tx + b;
          if (pre)
            acc[a][b] = Dn[2 * ty + a][2 * tx + b];
          else
            acc[a][b] = (r < n && c < n) ? __ldcg(&p.S[(size_t)r * n + c]) : (r == c ? 1.0 : 0.0);
        }
      {
        // running right-hand side of the forward substitution: (partial) - X y_(j-1), 8 lanes per row
        const int r = tid >> 3, sub8 = tid & 7;
        double a2 = 0;
        if (j >= 1) {
#pragma unroll
          for (int m = sub8; m < NB; m += 8) a2 += X[r][m] * vec[m];  // vec = y_(j-1)
        }
        a2 += __shfl_xor_sync(0xffffffffu, a2, 4);
        a2 += __shfl_xor_sync(0xffffffffu, a2, 2);
        a2 += __shfl_xor_sync(0xffffffffu, a2, 1);
        if (sub8 == 0) {
          double b0;
          if (pre)
            b0 = skn[r];
          else
            b0 = j0 + r < n ? (j >= 2 ? __ldcg(&ypart[j * NB + r]) : __ldcg(&p.rhs[j0 + r])) : 0.0;
          sk[r] = b0 - a2;
        }
      }
      if (j >= 1) {
#pragma unroll 8
        for (int m = 0; m < NB; m++) {
          const double a0 = X[2 * ty][m], a1 = X[2 * ty + 1][m];
          const double b0 = X[2 * tx][m], b1 = X[2 * tx + 1][m];
          acc[0][0] -= a0 * b0;
          acc[0][1] -= a0 * b1;
          acc[1][0] -= a1 * b0;
          acc[1][1] -= a1 * b1;
        }
      }
      __syncthreads();  // X, vec, Dn, skn and have_next have been read
      if (tid == 0) have_next = 0;
#pragma unroll
      for (int a = 0; a < 2; a++)
#pragma unroll
        for (int b = 0; b < 2; b++) A[2 * ty + a][2 * tx + b] = acc[a][b];
      // meanwhile: the sub partial of this column into registers (needed right after POTRF)
      const bool sub = j + 1 < T;
      __syncthreads();
      if (tid < 32) {
        potrf32_warp(A, idg, &s_ok, tid);
      } else if (warp == 2 || warp == 3) {
        // if the next diagonal partial is already there, take it now (no waiting here: these warps
        // are needed again as soon as the factorisation is done)
        if (sub) {
          const int jn = j + 1, jn0 = jn * NB;
          int ready = 1;
          if (jn >= 2) ready = *reinterpret_cast<const volatile int*>(&dflag[jn]);
          ready = __shfl_sync(0xffffffffu, ready, 0);
          if (ready) {
            __threadfence();
            for (int q = 0; q < 16; q++) {
              const int r = (warp - 2) * 16 + q;
              const int gr = jn0 + r, gc = jn0 + lane;
              Dn[r][lane] = (gr < n && gc < n) ? __ldcg(&p.S[(size_t)gr * n + gc]) : (gr == gc ? 1.0 : 0.0);
            }
            if (warp == 2)
              skn[lane] = jn0 + lane < n ? (jn >= 2 ? __ldcg(&ypart[jn * NB + lane]) : __ldcg(&p.rhs[jn0 + lane])) : 0.0;
            if (lane == 0) atomicAdd(&have_next, 1);
          }
        }
      } else if (sub && warp >= 4) {
        // warps 4..7 fetch the sub partial while warp 0 factorises (lane = column, 8 rows per warp)
        if (j >= 1 && lane == 0) {
          while (*reinterpret_cast<const volatile int*>(&sflag[j]) == 0) {
          }
          __threadfence();
        }
        __syncwarp();
        for (int q = 0; q < 8; q++) {
          const int r = (warp - 4) * 8 + q;
          X[r][lane] = (s0 + r < n && j0 + lane < n) ? __ldcg(&p.S[(size_t)(s0 + r) * n + j0 + lane]) : 0.0;
        }
      }
      __syncthreads();
      // L_jj is final: warp 0 goes on to X L_jj^T = (sub partial), warp 1 finishes y_j, the others publish L_jj
      if (tid < 32) {
        if (sub) trsm32_warp(X, A, idg, tid);
      } else if (warp == 1) {
        double v = sk[lane];
#pragma unroll 8
        for (int c = 0; c < NB; c++) {
          const double yc = __shfl_sync(0xffffffffu, v, c) * idg[c];
          if (lane == c) v = yc;
          if (lane > c) v -= A[c][lane] * yc;
        }
        vec[lane] = v;  // y_j, used by the next column
        if (j0 + lane < n) p.rhs[j0 + lane] = v;
        __threadfence();
        __syncwarp();
        if (lane == 0) atomicExch(&yflag[j], 1);
      } else {
        for (int e = tid - 64; e < NB * NB; e += 192) {
          const int r = e >> 5, c = e & 31;
          if (j0 + r < n && c < r) p.S[(size_t)(j0 + r) * n + j0 + c] = A[c][r];
        }
        if (tid - 64 < NB) {
          const int d = tid - 64;
          if (j0 + d < n) p.S[(size_t)(j0 + d) * n + j0 + d] = 1.0 / idg[d];
          p.dinv[(size_t)j * NB + d] = idg[d];
        }
        __threadfence();
      }
      __syncthreads();
      if (tid == 0) atomicExch(&flags[j * T + j], 1);
      if (sub) {
        for (int e = tid; e < NB * NB; e += 256) {
          const int r = e >> 5, c = e & 31;
          if (s0 + r < n && j0 + c < n) p.S[(size_t)(s0 + r) * n + j0 + c] = X[r][c];
        }
        publish(&flags[(j + 1) * T + j]);
      }
    }
    __syncthreads();
    if (tid == 0 && !s_ok) st->solve_ok = 0;
    return;
  }
  // ================= helpers: items in column order, dealt round-robin to CTAs 1 .. gridDim.x - 1
  const int n_help = (int)gridDim.x - 1;
  int g = 0, g_start = 0;  // column group of the current item and the number of its first item
  auto group_items = [&](int gg) {
    const int extra = (gg >= 1 && gg + 1 < T) ? 2 : 0;  // sub partial (gg+1, gg) and diagonal partial of block gg+1
    return extra + max(0, T - gg - 2);
  };
  int total = 0;
  for (int gg = 0; gg < T; gg++) total += group_items(gg);
  for (int t = (int)blockIdx.x - 1; t < total; t += n_help) {
    while (t >= g_start + group_items(g)) {
      g_start += group_items(g);
      g++;
    }
    const int local = t - g_start;
    const bool has_extra = g >= 1 && g + 1 < T;
    // kind 0: normal tile (i, g); 1: sub partial (g+1, g); 2: diagonal partial of block g+1
    int kind = 0, i = 0, j = g, kmax = g;
    if (has_extra && local == 0) {
      kind = 1;
      i = g + 1;
    } else if (has_extra && local == 1) {
      kind = 2;
      i = j = g + 1;
      kmax = g;  // k <= (g+1) - 2 = g - 1, i.e. k < g
    } else {
      i = g + 2 + (local - (has_extra ? 2 : 0));
    }
    const int i0 = i * NB, j0 = j * NB;
    const bool ywarp = kind == 2 && warp == 1;
    double skreg = (ywarp && i0 + lane < n) ? __ldcg(&p.rhs[i0 + lane]) : 0.0, yreg = 0.0;
    double acc[2][2];
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
      for (int b = 0; b < 2; b++) {
        const int r = i0 + 2 * ty + a, c = j0 + 2 * tx + b;
        acc[a][b] = (r < n && c < n) ? __ldcg(&p.S[(size_t)r * n + c]) : (r == c ? 1.0 : 0.0);
      }
    for (int k = 0; k < kmax; k++) {
      flag_wait(&flags[i * T + k]);
      if (i != j) flag_wait(&flags[j * T + k]);
      const int k0 = k * NB;
      if (ywarp) {
        if (lane == 0) {
          while (*reinterpret_cast<const volatile int*>(&yflag[k]) == 0) {
          }
          __threadfence();
        }
        __syncwarp();
        yreg = __ldcg(&p.rhs[k0 + lane]);
      }
      {
        double ta[4], tb[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
          const int e = tid + 256 * q, r = e >> 5, c = e & 31;
          ta[q] = (i0 + r < n) ? __ldcg(&p.S[(size_t)(i0 + r) * n + k0 + c]) : 0.0;
          tb[q] = (j0 + r < n) ? __ldcg(&p.S[(size_t)(j0 + r) * n + k0 + c]) : 0.0;
        }
#pragma unroll
        for (int q = 0; q < 4; q++) {
          const int e = tid + 256 * q, r = e >> 5, c = e & 31;
          A[r][c] = ta[q];
          B[r][c] = tb[q];
        }
      }
      __syncthreads();
      if (ywarp) {
        vec[lane] = yreg;
        __syncwarp();
        double a2 = 0;
#pragma unroll 8
        for (int m = 0; m < NB; m++) a2 += A[lane][m] * vec[m];
        skreg -= a2;
        __syncwarp();
      }
#pragma unroll 8
      for (int m = 0; m < NB; m++) {
        const double a0 = A[2 * ty][m], a1 = A[2 * ty + 1][m];
        const double b0 = B[2 * tx][m], b1 = B[2 * tx + 1][m];
        acc[0][0] -= a0 * b0;
        acc[0][1] -= a0 * b1;
        acc[1][0] -= a1 * b0;
        acc[1][1] -= a1 * b1;
      }
      __syncthreads();
    }
    if (kind != 0) {
      // partials go back in place (the chain CTA finishes them)
#pragma unroll
      for (int a = 0; a < 2; a++)
#pragma unroll
        for (int b = 0; b < 2; b++) {
          const int r = i0 + 2 * ty + a, c = j0 + 2 * tx + b;
          if (r < n && c < n && (kind == 1 || c <= r)) p.S[(size_t)r * n + c] = acc[a][b];
        }
      if (ywarp) ypart[i * NB + lane] = skreg;
      publish(kind == 1 ? &sflag[g] : &dflag[i]);
      continue;
    }
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
      for (int b = 0; b < 2; b++) A[2 * ty + a][2 * tx + b] = acc[a][b];
    flag_wait(&flags[j * T + j]);
    for (int e = tid; e < NB * NB; e += 256) {
      const int r = e >> 5, c = e & 31;  // B[m][c] = L_cm for m < c
      B[c][r] = (r > c && j0 + r < n) ? __ldcg(&p.S[(size_t)(j0 + r) * n + j0 + c]) : 0.0;
    }
    if (tid < NB) idg[tid] = __ldcg(&p.dinv[(size_t)j * NB + tid]);
    __syncthreads();
    if (tid < 32) trsm32_warp(A, B, idg, tid);
    __syncthreads();
    for (int e = tid; e < NB * NB; e += 256) {
      const int r = e >> 5, c = e & 31;
      if (i0 + r < n && j0 + c < n) p.S[(size_t)(i0 + r) * n + j0 + c] = A[r][c];
    }
    publish(&flags[i * T + j]);
    __syncthreads();
  }
}

// ---- dataflow triangular solves (one cooperative launch, one CTA per block row).
// Forward: CTA k accumulates b_k - sum_{j<k} L_kj y_j as the y_j are flagged ready
// (tile loads are issued before the flag wait: the factor is complete), solves its
// diagonal block with one warp (vector in registers) and publishes y_k.  Backward
// likewise from the last block row up with the transposed tiles.  The chain is
// T sequential publish/consume hops instead of 2T block steps of a single CTA.
__global__ void __launch_bounds__(256)
    ba_trisolve_dataflow_kernel(const BADev* __restrict__ probs, int* __restrict__ flags, int T, int fwd_done) {
  const BADev p = probs[0];
  LMState* st = p.st;
  if (st->done) return;
  __shared__ double Lt[3][NB][NB + 1];  // two streaming buffers + the diagonal tile (loaded once, up front)
  __shared__ double vec[NB];   // the consumed y_j / x_i
  __shared__ double part[8][NB];
  __shared__ double sk[NB];    // running right-hand side of this block row
  __shared__ double idg[NB];
  const int n = p.n, tid = threadIdx.x;
  const int k = blockIdx.x, k0 = k * NB;
  if (k >= T) return;
  const int kn = min(NB, n - k0);
  int* yflag = flags;
  int* xflag = flags + T;
  double* yv = p.rhs;  // y overwrites b block by block; x overwrites y
  auto load_tile = [&](int buf, int rb, int cb) {  // Lt[buf][r][c] = L[rb*32 + r][cb*32 + c]
    for (int e = tid; e < NB * NB; e += 256) {
      const int r = e >> 5, c = e & 31;
      const int gr = rb * NB + r, gc = cb * NB + c;
      Lt[buf][r][c] = (gr < n && gc < n && gc <= gr) ? __ldcg(&p.S[(size_t)gr * n + gc]) : 0.0;
    }
  };
  if (tid < NB) {
    sk[tid] = tid < kn ? __ldcg(&p.rhs[k0 + tid]) : 0.0;
    idg[tid] = __ldcg(&p.dinv[(size_t)k * NB + tid]);
  }
  load_tile(2, k, k);
  // ---------------- forward: L y = b (already done inside ba_chol_chain_kernel when fwd_done)
  if (!fwd_done && k > 0) load_tile(0, k, 0);
  __syncthreads();
  for (int j = 0; j < (fwd_done ? 0 : k); j++) {
    if (j + 1 < k) load_tile((j + 1) & 1, k, j + 1);
    flag_wait(&yflag[j]);
    if (tid < NB) vec[tid] = __ldcg(&yv[j * NB + tid]);
    __syncthreads();
    {
      const int r = tid & 31, q = tid >> 5;  // 8 column slices of 4
      double a = 0;
#pragma unroll
      for (int c = 0; c < 4; c++) a += Lt[j & 1][r][4 * q + c] * vec[4 * q + c];
      part[q][r] = a;
    }
    __syncthreads();
    if (tid < NB) {
      double a = 0;
#pragma unroll
      for (int q = 0; q < 8; q++) a += part[q][tid];
      sk[tid] -= a;
    }
    __syncthreads();
  }
  if (!fwd_done) {
    if (tid < 32) {
      double v = sk[tid];
      for (int j = 0; j < kn; j++) {
        const double yj = __shfl_sync(0xffffffffu, v, j) * idg[j];
        if (tid == j) v = yj;
        if (tid > j) v -= Lt[2][tid][j] * yj;
      }
      if (tid < kn) yv[k0 + tid] = v;
      sk[tid] = tid < kn ? v : 0.0;
      __threadfence();
      __syncwarp();
      if (tid == 0) atomicExch(&yflag[k], 1);
    }
    __syncthreads();
  }
  // ---------------- backward: L^T x = y   (sk holds y_k)
  if (k + 1 < T) load_tile(1, T - 1, k);
  __syncthreads();
  for (int i = T - 1; i > k; i--) {
    const int buf = (T - i) & 1;  // T-1 -> 1, T-2 -> 0, ...
    if (i - 1 > k) load_tile(buf ^ 1, i - 1, k);
    flag_wait(&xflag[i]);
    if (tid < NB) vec[tid] = (i * NB + tid < n) ? __ldcg(&yv[i * NB + tid]) : 0.0;
    __syncthreads();
    {
      const int c = tid & 31, q = tid >> 5;  // (L_ik^T x_i)[c] = sum_r L_ik[r][c] x_i[r]
      double a = 0;
#pragma unroll
      for (int r = 0; r < 4; r++) a += Lt[buf][4 * q + r][c] * vec[4 * q + r];
      part[q][c] = a;
    }
    __syncthreads();
    if (tid < NB) {
      double a = 0;
#pragma unroll
      for (int q = 0; q < 8; q++) a += part[q][tid];
      sk[tid] -= a;
    }
    __syncthreads();
  }
  if (tid < 32) {
    double v = sk[tid];
    for (int j = kn - 1; j >= 0; j--) {
      const double xj = __shfl_sync(0xffffffffu, v, j) * idg[j];
      if (tid == j) v = xj;
      if (tid < j) v -= Lt[2][j][tid] * xj;
    }
    if (tid < kn) yv[k0 + tid] = v;
    __threadfence();
    __syncwarp();
    if (tid == 0) atomicExch(&xflag[k], 1);
  }
}

// Trailing update A_ij -= L_ik L_jk^T for block pairs i >= j > kb (lower triangle).
__global__ void __launch_bounds__(256) ba_chol_update_kernel(const BADev* __restrict__ probs, int kb, int nblk) {
  const BADev p = probs[blockIdx.y];
  LMState* st = p.st;
  if (st->done) return;
  __shared__ double Li[NB][NB + 1];
  __shared__ double Lj[NB][NB + 1];
  const int n = p.n, tid = threadIdx.x;
  nblk = (n + NB - 1) / NB;
  // decode (bi, bj) from the linear block id over the lower triangle of the trailing part
  const int m = nblk - kb - 1;
  if (m <= 0) return;
  int t = blockIdx.x, bi = 0;
  while (t >= bi + 1) {
    t -= bi + 1;
    bi++;
  }
  const int bj = t;
  if (bi >= m) return;
  const int i0 = (kb + 1 + bi) * NB, j0 = (kb + 1 + bj) * NB, k0 = kb * NB;
  const int in = min(NB, n - i0), jn = min(NB, n - j0), kn = min(NB, n - k0);
  for (int e = tid; e < NB * NB; e += blockDim.x) {
    const int i = e / NB, k = e % NB;
    Li[i][k] = (i < in && k < kn) ? p.S[(size_t)(i0 + i) * n + k0 + k] : 0.0;
    Lj[i][k] = (i < jn && k < kn) ? p.S[(size_t)(j0 + i) * n + k0 + k] : 0.0;
  }
  __syncthreads();
  for (int e = tid; e < NB * NB; e += blockDim.x) {
    const int i = e / NB, j = e % NB;
    if (i < in && j < jn) {
      double acc = 0;
#pragma unroll 8
      for (int k = 0; k < NB; k++) acc += Li[i][k] * Lj[j][k];
      p.S[(size_t)(i0 + i) * n + j0 + j] -= acc;
    }
  }
}

// Triangular solves with the factor in global memory; one CTA, vector in smem.
// Per 32-wide block: the diagonal block is staged in shared memory and solved by
// one warp with the vector in registers (one shuffle + one FMA per column, the
// stored 1/L_jj instead of divides); then all threads update the remaining rows
// with register-staged loads.
__global__ void __launch_bounds__(1024) ba_chol_solve_kernel(const BADev* __restrict__ probs) {
  const BADev p = probs[blockIdx.y];
  LMState* st = p.st;
  if (st->done) return;
  extern __shared__ double y[];
  __shared__ double Lb[NB][NB + 1];
  __shared__ double yk[NB];
  __shared__ double idg[NB];
  const int n = p.n, tid = threadIdx.x;
  const int nblk = (n + NB - 1) / NB;
  for (int i = tid; i < n; i += blockDim.x) y[i] = p.rhs[i];
  __syncthreads();
  for (int kb = 0; kb < nblk; kb++) {  // L y = b
    const int k0 = kb * NB, kn = min(NB, n - k0);
    {
      const int i = tid >> 5, j = tid & 31;
      Lb[i][j] = (i < kn && j < i) ? p.S[(size_t)(k0 + i) * n + k0 + j] : 0.0;
      if (tid < NB) idg[tid] = p.dinv[(size_t)kb * NB + tid];
    }
    __syncthreads();
    if (tid < 32) {
      double v = tid < kn ? y[k0 + tid] : 0.0;
      for (int j = 0; j < kn; j++) {
        const double yj = __shfl_sync(0xffffffffu, v, j) * idg[j];
        if (tid == j) v = yj;
        if (tid > j) v -= Lb[tid][j] * yj;
      }
      yk[tid] = tid < kn ? v : 0.0;
      if (tid < kn) y[k0 + tid] = v;
    }
    __syncthreads();
    {
      // rows below the block: one warp per row, lane = column (coalesced 256 B),
      // four rows in flight per warp
      const int lane = tid & 31, warp = tid >> 5;
      const double ykl = yk[lane];
      for (int i = k0 + kn + warp; i < n; i += 32 * 4) {
        double a[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
          const int r = i + 32 * q;
          a[q] = (r < n && lane < kn) ? p.S[(size_t)r * n + k0 + lane] * ykl : 0.0;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
          for (int q = 0; q < 4; q++) a[q] += __shfl_xor_sync(0xffffffffu, a[q], o);
        }
        if (lane < 4) {
          const int r = i + 32 * lane;
          const double v = lane == 0 ? a[0] : (lane == 1 ? a[1] : (lane == 2 ? a[2] : a[3]));
          if (r < n) y[r] -= v;
        }
      }
    }
    __syncthreads();
  }
  for (int kb = nblk - 1; kb >= 0; kb--) {  // L^T x = y
    const int k0 = kb * NB, kn = min(NB, n - k0);
    {
      const int i = tid >> 5, j = tid & 31;
      Lb[i][j] = (i < kn && j < i) ? p.S[(size_t)(k0 + i) * n + k0 + j] : 0.0;
      if (tid < NB) idg[tid] = p.dinv[(size_t)kb * NB + tid];
    }
    __syncthreads();
    if (tid < 32) {
      double v = tid < kn ? y[k0 + tid] : 0.0;
      for (int j = kn - 1; j >= 0; j--) {
        const double xj = __shfl_sync(0xffffffffu, v, j) * idg[j];
        if (tid == j) v = xj;
        if (tid < j) v -= Lb[j][tid] * xj;  // (L^T)_{tid,j} = L_{j,tid}
      }
      yk[tid] = tid < kn ? v : 0.0;
      if (tid < kn) y[k0 + tid] = v;
    }
    __syncthreads();
    for (int i = tid; i < k0; i += blockDim.x) {
      double v[NB];
#pragma unroll
      for (int m = 0; m < NB; m++) v[m] = m < kn ? p.S[(size_t)(k0 + m) * n + i] : 0.0;
      double acc = 0;
#pragma unroll
      for (int m = 0; m < NB; m++) acc += v[m] * yk[m];
      y[i] -= acc;
    }
    __syncthreads();
  }
  for (int i = tid; i < n; i += blockDim.x) p.rhs[i] = y[i];
}

// Candidate cameras x_c - y_c * scale_c (+ their rotation blocks).  One CTA per window: the
// camera parts of |step|^2 and |x + step|^2 are summed in a fixed order (strided per thread,
// then a fixed shuffle / shared-memory tree), so that every rank of a sharded solve -- cameras
// are replicated there -- gets the same bits and takes the same trust-region decision.
__global__ void __launch_bounds__(128) ba_candcam_kernel(const BADev* __restrict__ probs) {
  const BADev p = probs[blockIdx.y];
  LMState* st = p.st;
  if (st->done) return;
  __shared__ double red[32];
  const int cur = st->cur;
  double step2 = 0, xc2 = 0;
  for (int c = threadIdx.x; c < p.C; c += blockDim.x) {
#pragma unroll
    for (int a = 0; a < 6; a++) {
      const double d = -p.rhs[6 * c + a] * p.scale_c[6 * c + a];
      const double x = p.cams[cur][6 * c + a] + d;
      p.cams[cur ^ 1][6 * c + a] = x;
      step2 += d * d;
      xc2 += x * x;
    }
    cam_rotation(p.cams[cur ^ 1] + 6 * c, p.camrot[cur ^ 1] + CAMROT * c, true);
  }
  const double s2 = block_sum(step2, red);
  const double x2 = block_sum(xc2, red);
  // camera parts are replicated on every rank: kept apart from the all-reduced sums
  if (threadIdx.x == 0) {
    p.tail[3] = s2;
    p.tail[4] = x2;
  }
}

// Back-substitution, model decrease, candidate points and candidate cost.
__device__ __forceinline__ void lm_control(const BADev& p, const lorb_ba_options& opt, int* n_active) {
  // volatile copy: accumulators were written by other CTAs through L2 atomics
  LMState loc;
  {
    const volatile long long* src = reinterpret_cast<const volatile long long*>(p.st);
    long long* dst = reinterpret_cast<long long*>(&loc);
    for (int i = 0; i < (int)(sizeof(LMState) / 8); i++) dst[i] = src[i];
  }
  const volatile double* tail = p.tail;
  loc.acc_step2 += tail[3];
  loc.acc_xcand2 += tail[4];
  const int acc = lm_decide(&loc, opt);
  if (acc) loc.cur ^= 1;
  lm_zero_acc(&loc);
  loc.blocks_done = 0;
  if (!loc.done) atomicAdd(n_active, 1);
  *p.st = loc;
}

// CS: every window of the launch has <= CS_MAX_CAMS cameras, kept in shared memory
template <bool CS, bool ROBUST = false>
__global__ void __launch_bounds__(BA_THREADS, 2)  // latency-bound gathers: two CTAs per SM (ncu: long_scoreboard)
    ba_backsub_kernel(const BADev* __restrict__ probs, lorb_ba_options opt, int fuse_control,
                      int* __restrict__ n_active) {
  const BADev p = probs[blockIdx.y];
  LMState* st = p.st;
  if (st->done) return;
  __shared__ double red[BA_THREADS / 32];
  extern __shared__ __align__(16) double cs[];  // CS: maxC * CS_BACKSUB doubles
  const int cur = st->cur;
  const double* cams = p.cams[cur];
  const double* pts = p.pts[cur];
  const double* camrot = p.camrot[cur];
  const double* cams_c = p.cams[cur ^ 1];
  const double* camrot_c = p.camrot[cur ^ 1];
  double* pts_c = p.pts[cur ^ 1];
  const double* yc = p.rhs;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, gl = lane & 7, gw = lane >> 3;
  if (CS) {
    cs_fill(p, cams, camrot, cs, CS_BACKSUB, tid, BA_THREADS);
    for (int i = tid; i < p.C * 18; i += BA_THREADS) {
      const int c = i / 18, k = i - c * 18;
      cs[c * CS_BACKSUB + CS_BUILD + k] = k < 6 ? yc[6 * c + k] : k < 15 ? camrot_c[CAMROT * c + (k - 6)] : cams_c[6 * c + 3 + (k - 15)];
    }
    __syncthreads();
  }
  double model_acc = 0, cost_acc = 0, step_acc = 0, xn_acc = 0;
  for (int base = (blockIdx.x * (BA_THREADS / 32) + warp) * 4; base < p.P;
       base += gridDim.x * (BA_THREADS / 8)) {
    const int pt = base + gw;
    const bool pv = pt < p.P;
    int s = 0, e = 0;
    double X[3] = {0, 0, 0}, sp[3] = {1, 1, 1};
    if (pv) {
      s = p.pt_ptr[pt];
      e = p.pt_ptr[pt + 1];
#pragma unroll
      for (int a = 0; a < 3; a++) {
        X[a] = pts[3 * (size_t)pt + a];
        sp[a] = p.scale_p[3 * (size_t)pt + a];
      }
    }
    // ncu: a third of this kernel's stall samples waited on three dependent global loads (the point
    // header of the next iteration, the observation's camera index, H_pp^-1 / g_p after the loop)
    if (pv && gl == 0) {
      prefetch_l1(p.pt_hinv + 6 * (size_t)pt);
      prefetch_l1(p.pt_gp + 3 * (size_t)pt);
    }
    {
      const int ptn = pt + (int)gridDim.x * (BA_THREADS / 8);
      if (ptn < p.P && gl == 1) {
        prefetch_l1(p.pt_ptr + ptn);
        prefetch_l1(pts + 3 * (size_t)ptn);
        prefetch_l1(p.scale_p + 3 * (size_t)ptn);
      }
    }
    const int rounds = __reduce_max_sync(0xffffffffu, (e - s + 7) >> 3);
    double bsum[3] = {0, 0, 0};
    double r[2], Jc[12], Jp[6];
    int cam = -1;
    bool has = false;
    double jcy[2] = {0, 0};
    for (int rd = 0; rd < rounds; rd++) {
      const int o = s + rd * 8 + gl;
      has = o < e;
      if (has) {
        cam = CS ? eval_obs_cs<ROBUST>(p, cs, CS_BACKSUB, o, X, sp, r, Jc, Jp)
                 : eval_obs<ROBUST>(p, cams, camrot, o, X, sp, r, Jc, Jp);
        jcy[0] = jcy[1] = 0;
        if (cam >= 0) {
          const double* ycam = CS ? cs + cam * CS_BACKSUB + CS_BUILD : yc + 6 * cam;
#pragma unroll
          for (int a = 0; a < 6; a++) {
            jcy[0] += Jc[a] * ycam[a];
            jcy[1] += Jc[6 + a] * ycam[a];
          }
#pragma unroll
          for (int a = 0; a < 3; a++) bsum[a] += Jp[a] * jcy[0] + Jp[3 + a] * jcy[1];
        }
      }
    }
#pragma unroll
    for (int a = 0; a < 3; a++) bsum[a] = group_sum8(bsum[a]);
    double yp[3] = {0, 0, 0}, Xc[3] = {0, 0, 0};
    if (pv) {
      const double* hi = p.pt_hinv + 6 * (size_t)pt;
      const double* gp = p.pt_gp + 3 * (size_t)pt;
      const double b0 = gp[0] - bsum[0], b1 = gp[1] - bsum[1], b2 = gp[2] - bsum[2];
      yp[0] = hi[0] * b0 + hi[1] * b1 + hi[2] * b2;
      yp[1] = hi[1] * b0 + hi[3] * b1 + hi[4] * b2;
      yp[2] = hi[2] * b0 + hi[4] * b1 + hi[5] * b2;
#pragma unroll
      for (int a = 0; a < 3; a++) Xc[a] = X[a] - yp[a] * sp[a];
      if (gl == 0) {
#pragma unroll
        for (int a = 0; a < 3; a++) {
          const double d = yp[a] * sp[a];
          pts_c[3 * (size_t)pt + a] = Xc[a];
          step_acc += d * d;
          xn_acc += Xc[a] * Xc[a];
        }
      }
    }
    // model residual m = J*step = -(Jc yc + Jp yp); candidate cost
    for (int rd = 0; rd < rounds; rd++) {
      const int o = s + rd * 8 + gl;
      if (o < e) {
        if (rounds > 1) {
          cam = CS ? eval_obs_cs<ROBUST>(p, cs, CS_BACKSUB, o, X, sp, r, Jc, Jp)
                 : eval_obs<ROBUST>(p, cams, camrot, o, X, sp, r, Jc, Jp);
          jcy[0] = jcy[1] = 0;
          if (cam >= 0) {
            const double* ycam = CS ? cs + cam * CS_BACKSUB + CS_BUILD : yc + 6 * cam;
#pragma unroll
            for (int a = 0; a < 6; a++) {
              jcy[0] += Jc[a] * ycam[a];
              jcy[1] += Jc[6 + a] * ycam[a];
            }
          }
        }
        const double m0 = -(jcy[0] + Jp[0] * yp[0] + Jp[1] * yp[1] + Jp[2] * yp[2]);
        const double m1 = -(jcy[1] + Jp[3] * yp[0] + Jp[4] * yp[1] + Jp[5] * yp[2]);
        model_acc += m0 * (r[0] + 0.5 * m0) + m1 * (r[1] + 0.5 * m1);
        const float2 uv = p.obs_uv[o];
        if (cam >= 0) {
          const double* rc = CS ? cs + cam * CS_BACKSUB + 51 : camrot_c + CAMROT * cam;
          const double* t = CS ? cs + cam * CS_BACKSUB + 60 : cams_c + 6 * cam + 3;
          const double tt[3] = {t[0], t[1], t[2]};
          cost_acc += obs_rho<ROBUST>(p, obs_cost(rc, tt, Xc, p.K, (double)uv.x, (double)uv.y));
        } else {
          const double* f = p.fixrt + 12 * (size_t)(-1 - cam);
          const double tt[3] = {f[9], f[10], f[11]};
          cost_acc += obs_rho<ROBUST>(p, obs_cost(f, tt, Xc, p.K, (double)uv.x, (double)uv.y));
        }
      }
    }
  }
  double t = block_sum(model_acc, red);
  if (tid == 0 && t != 0.0) atomicAdd(&st->acc_model, t);
  t = block_sum(cost_acc, red);
  if (tid == 0 && t != 0.0) atomicAdd(&st->acc_cost2, t);
  t = block_sum(step_acc, red);
  if (tid == 0 && t != 0.0) atomicAdd(&st->acc_step2, t);
  t = block_sum(xn_acc, red);
  if (tid == 0 && t != 0.0) atomicAdd(&st->acc_xcand2, t);
  if (fuse_control && tid == 0) {
    __threadfence();
    const int prev = atomicAdd(&st->blocks_done, 1);
    if (prev == (int)gridDim.x - 1) {
      __threadfence();
      lm_control(p, opt, n_active);
    }
  }
}

// End of a solve: windows whose current parameters sit in buffer 1 copy them to buffer 0 (where
// download and the next solve expect them).  One launch for the whole batch.
__global__ void __launch_bounds__(256) ba_make_current_kernel(const BADev* __restrict__ probs) {
  const BADev p = probs[blockIdx.y];
  if (p.st->cur != 1) return;
  const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gsize = gridDim.x * blockDim.x;
  for (int i = gtid; i < p.n; i += gsize) p.cams[0][i] = p.cams[1][i];
  for (int i = gtid; i < 3 * p.P; i += gsize) p.pts[0][i] = p.pts[1][i];
}

__global__ void ba_control_kernel(const BADev* __restrict__ probs, lorb_ba_options opt, int* __restrict__ n_active) {
  const BADev p = probs[blockIdx.x];
  LMState* st = p.st;
  if (st->done) return;
  lm_control(p, opt, n_active);
}

}  // namespace lorb

using namespace lorb;


// ------------------------------------------------------------------ host side
// A lorb_ba_problem is a batch of nw >= 1 independent windows resident in HBM
// (nw = 1 for lorb_ba_local / the sharded large solve).
struct lorb_ba_problem {
  lorb_ctx* ctx = nullptr;
  int nw = 0;
  std::vector<lorb::BADev> h_dev;     // host copies of the per-window descriptors
  std::vector<int> h_cam_off, h_pt_off;
  lorb::Buf params, topo, work, descs, hstate, counter, lists, stage;
  lorb::Buf list_scratch, list_scratch2;  // device scratch of the work-list builder (grow-only)
  double *h_cams_stage = nullptr, *h_pts_stage = nullptr;  // pinned staging of the parameters (up and down)
  int max_cam_items = 0, max_pair_items = 0;
  bool has_dup = false;  // some point is observed twice by the same window camera
  double *cams0 = nullptr, *pts0 = nullptr;  // initial parameters of all windows
  size_t cam_doubles = 0, pt_doubles = 0;
  int maxC = 0, maxP = 0;
  size_t lin_doubles_max = 0, lin_bytes_total = 0;
  double* lin_base = nullptr;
  lorb::LMState* d_states = nullptr;
};

namespace lorb {

static size_t al(size_t bytes) { return (bytes + 255) & ~(size_t)255; }

struct WindowSpec {  // host view of one window's inputs
  int C, P, O, F;
  const double* cams;
  const double* pts;
  const int* obs_cam;
  const int* obs_pt;
  const float* obs_uv;
  const int* fix_pt;
  const float* fix_uv;
  const float* fix_rt;
};

static void host_fix_rotation(const float* rt, double* R) {
  // float angle-axis widened to double (T(mRvec.at<float>(i)), reference
  // src/bundle_adjust.cpp:87), Rodrigues / small-angle as ceres::AngleAxisRotatePoint
  const double w0 = rt[0], w1 = rt[1], w2 = rt[2];
  const double th2 = w0 * w0 + w1 * w1 + w2 * w2;
  if (th2 > DBL_EPSILON) {
    const double th = sqrt(th2), s = sin(th), cth = cos(th), ith = 1.0 / th;
    const double k0 = w0 * ith, k1 = w1 * ith, k2 = w2 * ith, omc = 1.0 - cth;
    R[0] = cth + omc * k0 * k0; R[1] = -s * k2 + omc * k0 * k1; R[2] = s * k1 + omc * k0 * k2;
    R[3] = s * k2 + omc * k1 * k0; R[4] = cth + omc * k1 * k1; R[5] = -s * k0 + omc * k1 * k2;
    R[6] = -s * k1 + omc * k2 * k0; R[7] = s * k0 + omc * k2 * k1; R[8] = cth + omc * k2 * k2;
  } else {
    R[0] = 1; R[1] = -w2; R[2] = w1; R[3] = w2; R[4] = 1; R[5] = -w0; R[6] = -w1; R[7] = w0; R[8] = 1;
  }
  R[9] = rt[3];
  R[10] = rt[4];
  R[11] = rt[5];
}

// ---- work lists of the large path, built on the device -----------------------------------
// The large path (6C > 96) needs, per window, the observations grouped by camera (cam_obs /
// cam_items) and one record per pair of observations of the same point grouped by camera block
// (pairs / pair_items; 6.4 M records = 100 MB for 200 keyframes / 1.5 M observations).  They are
// derived from the point-major CSR that is uploaded anyway: building them on the host and
// uploading them took 15 of the 19 ms a cached lorb_ba_local call spends before the first LM
// iteration.  Order inside a group is the serial one (point, then observation ascending): records
// are generated point by point and grouped by a STABLE radix sort on the group key, so the fp64
// summation order of the consuming kernels does not depend on scheduling.
__global__ void __launch_bounds__(256)
    lists_count_kernel(int P, const int* __restrict__ ptr, const int* __restrict__ cam, int* __restrict__ obs_pt,
                       int* __restrict__ pcount) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const int a = ptr[p], b = ptr[p + 1];
  int n = 0;
  for (int e1 = a; e1 < b; e1++) {
    obs_pt[e1] = p;
    const int c1 = cam[e1];
    if (c1 < 0) continue;
    for (int e2 = a; e2 < b; e2++) n += cam[e2] >= c1;
  }
  pcount[p] = n;
}

__global__ void __launch_bounds__(256)
    lists_gen_pairs_kernel(int P, int C, const int* __restrict__ ptr, const int* __restrict__ cam,
                           const int* __restrict__ poff, uint32_t* __restrict__ key, uint32_t* __restrict__ idx,
                           int4* __restrict__ rec, int* __restrict__ kcnt) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const int a = ptr[p], b = ptr[p + 1];
  int i = poff[p];
  for (int e1 = a; e1 < b; e1++) {
    const int c1 = cam[e1];
    if (c1 < 0) continue;
    for (int e2 = a; e2 < b; e2++) {
      const int c2 = cam[e2];
      if (c2 < c1) continue;
      const uint32_t k = (uint32_t)c1 * C + c2;
      key[i] = k;
      idx[i] = i;
      rec[i] = make_int4(p, e1, e2, 0);
      atomicAdd(&kcnt[k], 1);
      i++;
    }
  }
}

__global__ void __launch_bounds__(256)
    lists_gather_pairs_kernel(int n, const uint32_t* __restrict__ idx, const int4* __restrict__ rec,
                              int4* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = rec[idx[i]];
}

__global__ void __launch_bounds__(256)
    lists_cam_keys_kernel(int OT, int C, const int* __restrict__ cam, uint32_t* __restrict__ key,
                          uint32_t* __restrict__ val, int* __restrict__ ccnt) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= OT) return;
  const int c1 = cam[e];
  key[e] = c1 >= 0 ? (uint32_t)c1 : (uint32_t)C;  // fixed observers sort behind every camera
  val[e] = e;
  if (c1 >= 0) atomicAdd(&ccnt[c1], 1);
}

__global__ void __launch_bounds__(256)
    lists_cam_obs_kernel(int n_valid, const uint32_t* __restrict__ val, const int* __restrict__ obs_pt,
                         int2* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_valid) out[i] = make_int2((int)val[i], obs_pt[val[i]]);
}

// nitems[k] = number of items of group k (chunks of `chunk` records)
__global__ void __launch_bounds__(256)
    lists_item_count_kernel(int n_groups, const int* __restrict__ cnt, int chunk, int* __restrict__ nitems) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n_groups) nitems[k] = (cnt[k] + chunk - 1) / chunk;
}

// items of group k: (a, b, start, length) with (a, b) = (k / C, k % C) for pair blocks (C > 0) or
// (k, start, length, 0) for cameras (C == 0)
__global__ void __launch_bounds__(256)
    lists_item_write_kernel(int n_groups, int C, const int* __restrict__ cnt, const int* __restrict__ start,
                            const int* __restrict__ ioff, int chunk, int4* __restrict__ items) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_groups) return;
  const int n = cnt[k], s0 = start[k];
  int o = ioff[k];
  for (int st = 0; st < n; st += chunk, o++) {
    const int len = min(chunk, n - st);
    items[o] = C > 0 ? make_int4(k / C, k % C, s0 + st, len) : make_int4(k, s0 + st, len, 0);
  }
}

struct DevListCounts {
  int n_cam_obs, n_cam_items, n_pair_items;
  long long n_pairs;
};

static int log2_ceil(unsigned v) {
  int b = 1;
  while (b < 32 && (1u << b) < v) b++;
  return b;
}

// Phase 1 of a window: obs_pt, the camera-major lists (sizes bounded by OT) and the number of
// pair records.  Phase 2: the pair records and their items into `pairs` / `pair_items`.
struct DevListBuilder {
  lorb_ctx* c;
  Buf* scratch;
  cudaStream_t s;

  static int nblocks(long long n) { return (int)std::max<long long>(1, (n + 255) / 256); }  // empty inputs still launch

  template <typename T>
  static T* carve(uint8_t*& p, size_t n) {
    T* r = reinterpret_cast<T*>(p);
    p += (n * sizeof(T) + 255) & ~(size_t)255;
    return r;
  }

  int phase1(int C, int P, int OT, const int* d_ptr, const int* d_cam, int* obs_pt, int2* cam_obs, int4* cam_items,
             int cam_items_cap, int** poff_out, DevListCounts* out) {
    // scratch: pcount / poff [P+1], keys / vals x2 [OT], ccnt / cstart / nitems / ioff [C+2], cub temp
    size_t tmp_sort = 0, tmp_scan = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp_sort, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr,
                                    (uint32_t*)nullptr, OT, 0, log2_ceil(C + 1), s);
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_scan, (int*)nullptr, (int*)nullptr, std::max(P, C) + 2, s);
    const size_t tmp = std::max(tmp_sort, tmp_scan);
    const size_t need = 2 * al((size_t)(P + 2) * 4) + 4 * al((size_t)std::max(OT, 1) * 4) + 4 * al((size_t)(C + 2) * 4) +
                        al(tmp) + 1024;
    LORB_TRY(scratch->reserve(need));
    uint8_t* q = scratch->as<uint8_t>();
    int* pcount = carve<int>(q, P + 2);
    int* poff = carve<int>(q, P + 2);
    uint32_t* k0 = carve<uint32_t>(q, std::max(OT, 1));
    uint32_t* k1 = carve<uint32_t>(q, std::max(OT, 1));
    uint32_t* v0 = carve<uint32_t>(q, std::max(OT, 1));
    uint32_t* v1 = carve<uint32_t>(q, std::max(OT, 1));
    int* ccnt = carve<int>(q, C + 2);
    int* cstart = carve<int>(q, C + 2);
    int* nitems = carve<int>(q, C + 2);
    int* ioff = carve<int>(q, C + 2);
    void* cub_tmp = q;
    LORB_CUDA_TRY(cudaMemsetAsync(pcount, 0, (size_t)(P + 2) * 4, s));
    LORB_CUDA_TRY(cudaMemsetAsync(ccnt, 0, (size_t)(C + 2) * 4, s));
    LORB_LAUNCH(c, lists_count_kernel, nblocks(P), 256, 0, P, d_ptr, d_cam, obs_pt, pcount);
    size_t t1 = tmp;
    LORB_CUDA_TRY(cub::DeviceScan::ExclusiveSum(cub_tmp, t1, pcount, poff, P + 1, s));
    // observations grouped by camera
    LORB_LAUNCH(c, lists_cam_keys_kernel, nblocks(OT), 256, 0, OT, C, d_cam, k0, v0, ccnt);
    t1 = tmp;
    LORB_CUDA_TRY(cub::DeviceRadixSort::SortPairs(cub_tmp, t1, k0, k1, v0, v1, OT, 0, log2_ceil(C + 1), s));
    t1 = tmp;
    LORB_CUDA_TRY(cub::DeviceScan::ExclusiveSum(cub_tmp, t1, ccnt, cstart, C + 1, s));
    LORB_LAUNCH(c, lists_item_count_kernel, nblocks(C), 256, 0, C, ccnt, 1024, nitems);
    t1 = tmp;
    LORB_CUDA_TRY(cub::DeviceScan::ExclusiveSum(cub_tmp, t1, nitems, ioff, C + 1, s));
    int h[3];
    LORB_CUDA_TRY(cudaMemcpyAsync(&h[0], poff + P, 4, cudaMemcpyDeviceToHost, s));
    LORB_CUDA_TRY(cudaMemcpyAsync(&h[1], cstart + C, 4, cudaMemcpyDeviceToHost, s));
    LORB_CUDA_TRY(cudaMemcpyAsync(&h[2], ioff + C, 4, cudaMemcpyDeviceToHost, s));
    LORB_CUDA_TRY(cudaStreamSynchronize(s));
    LORB_REQUIRE(h[0] >= 0 && h[1] >= 0 && h[1] <= OT && h[2] <= cam_items_cap, "work list sizes (internal)");
    LORB_LAUNCH(c, lists_cam_obs_kernel, nblocks(h[1]), 256, 0, h[1], v1, obs_pt, cam_obs);
    LORB_LAUNCH(c, lists_item_write_kernel, nblocks(C), 256, 0, C, 0, ccnt, cstart, ioff, 1024, cam_items);
    out->n_pairs = h[0];
    out->n_cam_obs = h[1];
    out->n_cam_items = h[2];
    *poff_out = poff;  // stays valid until the next phase1 call
    return LORB_OK;
  }

  // pairs [n_pairs], pair_items [<= n_pairs / 2048 + C*(C+1)/2]; scratch2 holds keys, indices, records
  int phase2(int C, int P, int n_pairs, const int* d_ptr, const int* d_cam, const int* poff, Buf* scratch2,
             int4* pairs, int4* pair_items, int pair_items_cap, int* n_pair_items) {
    *n_pair_items = 0;
    if (n_pairs == 0) return LORB_OK;
    const int nblk = C * C;
    size_t tmp_sort = 0, tmp_scan = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp_sort, (uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr,
                                    (uint32_t*)nullptr, n_pairs, 0, log2_ceil(nblk), s);
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_scan, (int*)nullptr, (int*)nullptr, nblk + 2, s);
    const size_t tmp = std::max(tmp_sort, tmp_scan);
    const size_t need = 4 * al((size_t)n_pairs * 4) + al((size_t)n_pairs * 16) + 4 * al((size_t)(nblk + 2) * 4) + al(tmp) + 1024;
    LORB_TRY(scratch2->reserve(need));
    uint8_t* q = scratch2->as<uint8_t>();
    uint32_t* k0 = carve<uint32_t>(q, n_pairs);
    uint32_t* k1 = carve<uint32_t>(q, n_pairs);
    uint32_t* v0 = carve<uint32_t>(q, n_pairs);
    uint32_t* v1 = carve<uint32_t>(q, n_pairs);
    int4* rec = carve<int4>(q, n_pairs);
    int* kcnt = carve<int>(q, nblk + 2);
    int* kstart = carve<int>(q, nblk + 2);
    int* nitems = carve<int>(q, nblk + 2);
    int* ioff = carve<int>(q, nblk + 2);
    void* cub_tmp = q;
    LORB_CUDA_TRY(cudaMemsetAsync(kcnt, 0, (size_t)(nblk + 2) * 4, s));
    LORB_LAUNCH(c, lists_gen_pairs_kernel, nblocks(P), 256, 0, P, C, d_ptr, d_cam, poff, k0, v0, rec, kcnt);
    size_t t1 = tmp;
    LORB_CUDA_TRY(cub::DeviceRadixSort::SortPairs(cub_tmp, t1, k0, k1, v0, v1, n_pairs, 0, log2_ceil(nblk), s));
    LORB_LAUNCH(c, lists_gather_pairs_kernel, nblocks(n_pairs), 256, 0, n_pairs, v1, rec, pairs);
    t1 = tmp;
    LORB_CUDA_TRY(cub::DeviceScan::ExclusiveSum(cub_tmp, t1, kcnt, kstart, nblk + 1, s));
    LORB_LAUNCH(c, lists_item_count_kernel, nblocks(nblk), 256, 0, nblk, kcnt, 2048, nitems);
    t1 = tmp;
    LORB_CUDA_TRY(cub::DeviceScan::ExclusiveSum(cub_tmp, t1, nitems, ioff, nblk + 1, s));
    int h = 0;
    LORB_CUDA_TRY(cudaMemcpyAsync(&h, ioff + nblk, 4, cudaMemcpyDeviceToHost, s));
    LORB_CUDA_TRY(cudaStreamSynchronize(s));
    LORB_REQUIRE(h >= 0 && h <= pair_items_cap, "pair item count (internal)");
    LORB_LAUNCH(c, lists_item_write_kernel, nblocks(nblk), 256, 0, nblk, C, kcnt, kstart, ioff, 2048, pair_items);
    *n_pair_items = h;
    return LORB_OK;
  }
};

// LORB_BA_TRACE=1: host timeline of problem_build on stderr (microseconds since it started)
struct BuildTrace {
  bool on;
  std::chrono::steady_clock::time_point t0;
  BuildTrace() : on(getenv("LORB_BA_TRACE") != nullptr), t0(std::chrono::steady_clock::now()) {}
  void mark(const char* what) const {
    if (!on) return;
    fprintf(stderr, "[ba build %9.1f us] %s\n",
            std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count(), what);
  }
};

static int problem_build(lorb_ba_problem* pb, lorb_ctx* c, const std::vector<WindowSpec>& ws,
                         const float* K) {
  const BuildTrace btr;
  pb->ctx = c;
  const int nw = (int)ws.size();
  pb->nw = nw;
  pb->maxC = pb->maxP = 0;
  pb->lin_doubles_max = 0;
  pb->h_dev.resize(nw);
  pb->h_cam_off.assign(nw + 1, 0);
  pb->h_pt_off.assign(nw + 1, 0);
  size_t tot_obs = 0, tot_fix = 0, tot_ptr = 0, tot_lin = 0, tot_rot = 0, tot_dinv = 0, tot_sfull = 0;
  for (int w = 0; w < nw; w++) {
    const WindowSpec& W = ws[w];
    LORB_REQUIRE(W.C > 0 && W.P >= 0 && W.O >= 0 && W.F >= 0, "window sizes");
    pb->h_cam_off[w + 1] = pb->h_cam_off[w] + W.C;
    pb->h_pt_off[w + 1] = pb->h_pt_off[w] + W.P;
    pb->maxC = std::max(pb->maxC, W.C);
    pb->maxP = std::max(pb->maxP, W.P);
    const int n = 6 * W.C;
    // the large path accumulates the Schur products into the packed upper block triangle (half the
    // memset and, sharded, half the all-reduce); its dense matrix is a separate buffer
    const bool packed = n > 96;
    const size_t lin = (packed ? (size_t)18 * W.C * (W.C + 1) : (size_t)n * n) + (size_t)HCC * W.C +
                       12 * (size_t)W.C + 24;
    pb->lin_doubles_max = std::max(pb->lin_doubles_max, lin);
    tot_lin += lin;
    if (packed) tot_sfull += (size_t)n * n;
    tot_obs += (size_t)W.O + W.F;
    tot_fix += W.F;
    tot_ptr += (size_t)W.P + 1;
    tot_rot += (size_t)W.C * CAMROT;
    tot_dinv += (size_t)((n + NB - 1) / NB) * NB;
  }
  const size_t totC = pb->h_cam_off[nw], totP = pb->h_pt_off[nw];
  pb->cam_doubles = totC * 6;
  pb->pt_doubles = totP * 3;
  // ---- host staging of the topology (CSR by point per window)
  // staged in pinned memory owned by the problem (grow-only): the uploads below are
  // true async DMA and a cached problem allocates nothing in steady state
  const size_t sb_ptr = al(tot_ptr * 4), sb_cam = al(std::max<size_t>(tot_obs, 1) * 4),
               sb_uv = al(std::max<size_t>(tot_obs, 1) * 8), sb_fix = al(std::max<size_t>(tot_fix, 1) * 96),
               sb_cams = al(std::max<size_t>(pb->cam_doubles, 1) * 8),
               sb_pts = al(std::max<size_t>(pb->pt_doubles, 1) * 8);
  pb->stage.pinned = true;
  LORB_TRY(pb->stage.reserve(sb_ptr + sb_cam + sb_uv + sb_fix + sb_cams + sb_pts));
  uint8_t* sg = pb->stage.as<uint8_t>();
  int* h_ptr = reinterpret_cast<int*>(sg);
  int* h_cam = reinterpret_cast<int*>(sg + sb_ptr);
  float2* h_uv = reinterpret_cast<float2*>(sg + sb_ptr + sb_cam);
  double* h_fix = reinterpret_cast<double*>(sg + sb_ptr + sb_cam + sb_uv);
  double* h_cams = reinterpret_cast<double*>(sg + sb_ptr + sb_cam + sb_uv + sb_fix);
  double* h_pts = reinterpret_cast<double*>(sg + sb_ptr + sb_cam + sb_uv + sb_fix + sb_cams);
  pb->h_cams_stage = h_cams;
  pb->h_pts_stage = h_pts;
  std::vector<size_t> o_ptr(nw), o_obs(nw), o_fix(nw);
  // large-path work lists (windows with 6C > 96), concatenated over windows
  struct ListOff {
    size_t obs_pt, cam_obs, cam_items, pairs, pair_items;
    int n_cam_items, n_pair_items, large;
    long long n_pairs;
  };
  std::vector<ListOff> lo(nw, ListOff{0, 0, 0, 0, 0, 0, 0, 0, 0});
  pb->max_cam_items = pb->max_pair_items = 0;
  pb->has_dup = false;
  {
    bool any_large = false;
    {
      size_t a = 0, b = 0, f = 0;
      for (int w = 0; w < nw; w++) {
        o_ptr[w] = a;
        o_obs[w] = b;
        o_fix[w] = f;
        a += (size_t)ws[w].P + 1;
        b += (size_t)ws[w].O + ws[w].F;
        f += ws[w].F;
        any_large = any_large || 6 * ws[w].C > 96;
      }
    }
    // Staging one window touches only its own slices, so a batch of small windows is staged by
    // all host threads; windows that need the large-path work lists (shared vectors) go serially.
    int bad_obs = 0, bad_fix = 0, dup_any = 0;
#pragma omp parallel for schedule(dynamic, 1) reduction(| : bad_obs, bad_fix, dup_any) if (nw > 3 && !any_large)
    for (int w = 0; w < nw; w++) {
      const WindowSpec& W = ws[w];
      const size_t a = o_ptr[w], b = o_obs[w], f = o_fix[w];
      int* ptr = &h_ptr[a];
      for (int i = 0; i <= W.P; i++) ptr[i] = 0;
      bool sorted = W.F == 0;  // fast path: window observations already grouped by ascending point
      bool bad = false;
      const bool big = W.O > 200000;  // a large window is staged alone: its loops use the host threads
      if (big) {
        int bad_i = 0, unsorted_i = 0;
#pragma omp parallel for schedule(static) reduction(| : bad_i, unsorted_i)
        for (int i = 0; i < W.O; i++) {
          if (!(W.obs_pt[i] >= 0 && W.obs_pt[i] < W.P && W.obs_cam[i] >= 0 && W.obs_cam[i] < W.C)) {
            bad_i |= 1;
            continue;
          }
#pragma omp atomic
          ptr[W.obs_pt[i] + 1]++;
          if (i > 0 && W.obs_pt[i] < W.obs_pt[i - 1]) unsorted_i |= 1;
        }
        bad = bad_i != 0;
        if (unsorted_i) sorted = false;
      } else {
        for (int i = 0; i < W.O; i++) {
          if (!(W.obs_pt[i] >= 0 && W.obs_pt[i] < W.P && W.obs_cam[i] >= 0 && W.obs_cam[i] < W.C)) {
            bad = true;
            break;
          }
          ptr[W.obs_pt[i] + 1]++;
          if (i > 0 && W.obs_pt[i] < W.obs_pt[i - 1]) sorted = false;
        }
      }
      if (bad) {
        bad_obs |= 1;
        continue;
      }
      for (int i = 0; i < W.F; i++) {
        if (!(W.fix_pt[i] >= 0 && W.fix_pt[i] < W.P)) {
          bad = true;
          break;
        }
        ptr[W.fix_pt[i] + 1]++;
      }
      if (bad) {
        bad_fix |= 1;
        continue;
      }
      for (int i = 0; i < W.P; i++) ptr[i + 1] += ptr[i];
      std::vector<int> fill;
      if (sorted) {  // the CSR order is the input order: two block copies
        if (W.O && big) {
          const int nchunk = 64;
#pragma omp parallel for schedule(static)
          for (int ch = 0; ch < nchunk; ch++) {
            const size_t i0 = (size_t)W.O * ch / nchunk, i1 = (size_t)W.O * (ch + 1) / nchunk;
            memcpy(&h_cam[b + i0], W.obs_cam + i0, (i1 - i0) * 4);
            memcpy(&h_uv[b + i0], W.obs_uv + 2 * i0, (i1 - i0) * 8);
          }
        } else if (W.O) {
          memcpy(&h_cam[b], W.obs_cam, (size_t)W.O * 4);
          memcpy(&h_uv[b], W.obs_uv, (size_t)W.O * 8);
        }
      } else {
        fill.assign(ptr, ptr + W.P);
        for (int i = 0; i < W.O; i++) {
          const int d = fill[W.obs_pt[i]]++;
          h_cam[b + d] = W.obs_cam[i];
          h_uv[b + d] = make_float2(W.obs_uv[2 * i], W.obs_uv[2 * i + 1]);
        }
      }
      for (int i = 0; i < W.F; i++) {
        const int d = fill[W.fix_pt[i]]++;
        h_cam[b + d] = -1 - i;
        h_uv[b + d] = make_float2(W.fix_uv[2 * i], W.fix_uv[2 * i + 1]);
        host_fix_rotation(W.fix_rt + 6 * (size_t)i, &h_fix[12 * (f + i)]);
      }
      if (6 * W.C <= DENSE_N) {
        // the atomic-free dense path stores (point, camera) tiles: needs unique pairs
        const int* cam2 = &h_cam[b];
        bool dup = false;
        for (int pp = 0; pp < W.P && !dup; pp++)
          for (int e1 = ptr[pp]; e1 < ptr[pp + 1] && !dup; e1++)
            for (int e2 = e1 + 1; e2 < ptr[pp + 1]; e2++)
              if (cam2[e1] >= 0 && cam2[e1] == cam2[e2]) {
                dup = true;
                break;
              }
        if (dup) dup_any |= 1;
      }
      if (any_large) {
        // large path: the work lists are built on the device from the CSR (DevListBuilder); the
        // host only counts the pair records so that every buffer can be sized before the uploads.
        // One window with 6C > 96 puts the whole batch on this path (the build kernels are chosen
        // per launch), so every window of such a batch gets its lists.
        btr.mark("csr staged");
        const int* cam = &h_cam[b];
        long long np = 0;
#pragma omp parallel for schedule(static) reduction(+ : np) if (big)
        for (int pp = 0; pp < W.P; pp++)
          for (int e1 = ptr[pp]; e1 < ptr[pp + 1]; e1++) {
            if (cam[e1] < 0) continue;
            for (int e2 = ptr[pp]; e2 < ptr[pp + 1]; e2++) np += cam[e2] >= cam[e1];
          }
        lo[w].large = 1;
        lo[w].n_pairs = np;
        btr.mark("pair records counted");
      }
      memcpy(&h_cams[6 * (size_t)pb->h_cam_off[w]], W.cams, (size_t)W.C * 48);
      if (W.P) memcpy(&h_pts[3 * (size_t)pb->h_pt_off[w]], W.pts, (size_t)W.P * 24);
    }
    LORB_REQUIRE(!bad_obs, "observation index out of range");
    LORB_REQUIRE(!bad_fix, "fixed observation point out of range");
    pb->has_dup = dup_any != 0;
  }
  btr.mark("staging done");
  // ---- device layout
  const size_t cb = al(pb->cam_doubles * 8), pbts = al(std::max<size_t>(pb->pt_doubles, 1) * 8);
  LORB_TRY(pb->params.reserve(3 * cb + 3 * pbts));
  uint8_t* q = pb->params.as<uint8_t>();
  double* d_cams[2] = {(double*)q, (double*)(q + cb)};
  pb->cams0 = (double*)(q + 2 * cb);
  double* d_pts[2] = {(double*)(q + 3 * cb), (double*)(q + 3 * cb + pbts)};
  pb->pts0 = (double*)(q + 3 * cb + 2 * pbts);
  const size_t t_ptr = al(tot_ptr * 4), t_cam = al(std::max<size_t>(tot_obs, 1) * 4),
               t_uv = al(std::max<size_t>(tot_obs, 1) * 8), t_fix = al(std::max<size_t>(tot_fix, 1) * 96);
  LORB_TRY(pb->topo.reserve(t_ptr + t_cam + t_uv + t_fix));
  uint8_t* t = pb->topo.as<uint8_t>();
  int* d_ptr = (int*)t;
  int* d_ocam = (int*)(t + t_ptr);
  float2* d_uv = (float2*)(t + t_ptr + t_cam);
  double* d_fix = (double*)(t + t_ptr + t_cam + t_uv);
  const size_t w_rot = al(tot_rot * 8), w_sc = cb, w_sp = pbts, w_lin = al(tot_lin * 8), w_rhs = cb,
               w_hinv = al(std::max<size_t>(totP, 1) * 48), w_gp = pbts,
               w_st = al(sizeof(LMState) * (size_t)nw), w_dinv = al(tot_dinv * 8), w_sfull = al(tot_sfull * 8);
  LORB_TRY(pb->work.reserve(2 * w_rot + w_sc + w_sp + w_lin + w_rhs + w_hinv + w_gp + w_st + w_dinv + w_sfull));
  uint8_t* wk = pb->work.as<uint8_t>();
  double* d_rot[2] = {(double*)wk, (double*)(wk + w_rot)};
  wk += 2 * w_rot;
  double* d_sc = (double*)wk;   wk += w_sc;
  double* d_sp = (double*)wk;   wk += w_sp;
  double* d_lin = (double*)wk;  wk += w_lin;
  double* d_rhs = (double*)wk;  wk += w_rhs;
  double* d_hinv = (double*)wk; wk += w_hinv;
  double* d_gp = (double*)wk;   wk += w_gp;
  pb->d_states = (LMState*)wk;  wk += w_st;
  double* d_dinv = (double*)wk; wk += w_dinv;
  double* d_sfull = (double*)wk;
  pb->lin_base = d_lin;
  pb->lin_bytes_total = tot_lin * 8;
  {
    size_t lin_off = 0, rot_off = 0, dinv_off = 0, sfull_off = 0;
    for (int w = 0; w < nw; w++) {
      const WindowSpec& W = ws[w];
      BADev& d = pb->h_dev[w];
      const size_t co = 6 * (size_t)pb->h_cam_off[w], po = 3 * (size_t)pb->h_pt_off[w];
      d.C = W.C;
      d.P = W.P;
      d.n = 6 * W.C;
      for (int b = 0; b < 2; b++) {
        d.cams[b] = d_cams[b] + co;
        d.pts[b] = d_pts[b] + po;
        d.camrot[b] = d_rot[b] + rot_off;
      }
      d.pt_ptr = d_ptr + o_ptr[w];
      d.obs_cam = d_ocam + o_obs[w];
      d.obs_uv = d_uv + o_obs[w];
      d.fixrt = d_fix + 12 * o_fix[w];
      d.K.fu = (double)K[0];
      d.K.fv = (double)K[1];
      d.K.cx = (double)K[2];
      d.K.cy = (double)K[3];
      d.scale_c = d_sc + co;
      d.scale_p = d_sp + po;
      d.lin = d_lin + lin_off;
      const bool packed = d.n > 96;
      const size_t s_doubles = packed ? (size_t)18 * W.C * (W.C + 1) : (size_t)d.n * d.n;
      d.Sp = packed ? d.lin : nullptr;
      d.S = packed ? d_sfull + sfull_off : d.lin;
      if (packed) sfull_off += (size_t)d.n * d.n;
      d.Hcc = d.lin + s_doubles;
      d.gc = d.Hcc + (size_t)HCC * W.C;
      d.rhs_corr = d.gc + 6 * (size_t)W.C;
      d.tail = d.rhs_corr + 6 * (size_t)W.C;
      d.gslot = d.tail + 8;
      d.rank = 0;
      d.world = 1;
      d.rhs = d_rhs + co;
      d.pt_hinv = d_hinv + 2 * po;
      d.pt_gp = d_gp + po;
      d.st = pb->d_states + w;
      d.dinv = d_dinv + dinv_off;
      dinv_off += (size_t)((d.n + NB - 1) / NB) * NB;
      lin_off += s_doubles + (size_t)HCC * W.C + 12 * (size_t)W.C + 24;
      rot_off += (size_t)W.C * CAMROT;
    }
  }
  cudaStream_t s = c->stream;
  // the CSR goes up first: the device list builder reads it
  LORB_CUDA_TRY(cudaMemcpyAsync(d_ptr, h_ptr, tot_ptr * 4, cudaMemcpyHostToDevice, s));
  LORB_CUDA_TRY(cudaMemcpyAsync(d_ocam, h_cam, tot_obs * 4, cudaMemcpyHostToDevice, s));
  pb->max_cam_items = pb->max_pair_items = 0;
  {
    // layout of the list buffer: every size is known on the host
    size_t n_obs_pt = 0, n_cam_obs = 0, n_cam_items = 0, n_pairs = 0, n_pair_items = 0;
    long long max_pairs = 0;
    for (int w = 0; w < nw; w++) {
      ListOff& L = lo[w];
      if (!L.large) continue;
      const WindowSpec& W = ws[w];
      const size_t OT = (size_t)W.O + W.F;
      LORB_REQUIRE(L.n_pairs < (1ll << 31), "more than 2^31 pair records in one window");
      LORB_REQUIRE(W.C <= 8192, "more than 8192 cameras in one window (camera-block keys are C*C)");
      L.obs_pt = n_obs_pt;
      L.cam_obs = n_cam_obs;
      L.cam_items = n_cam_items;
      L.pairs = n_pairs;
      L.pair_items = n_pair_items;
      n_obs_pt += OT;
      n_cam_obs += OT;
      n_cam_items += (size_t)W.C + OT / 1024 + 1;
      n_pairs += (size_t)L.n_pairs;
      n_pair_items += (size_t)(L.n_pairs / 2048) + (size_t)W.C * (W.C + 1) / 2 + 1;
      max_pairs = std::max(max_pairs, L.n_pairs);
    }
    const size_t b0 = al(n_obs_pt * 4), b1 = al(n_cam_obs * 8), b2 = al(n_cam_items * 16), b3 = al(n_pairs * 16),
                 b4 = al(n_pair_items * 16);
    LORB_TRY(pb->lists.reserve(b0 + b1 + b2 + b3 + b4 + 256));
    uint8_t* lb = pb->lists.as<uint8_t>();
    DevListBuilder bld{c, &pb->list_scratch, s};
    for (int w = 0; w < nw; w++) {
      BADev& d = pb->h_dev[w];
      ListOff& L = lo[w];
      d.obs_pt = nullptr;
      d.cam_obs = nullptr;
      d.cam_items = nullptr;
      d.pairs = nullptr;
      d.pair_items = nullptr;
      d.n_cam_items = d.n_pair_items = 0;
      if (!L.large) continue;
      const WindowSpec& W = ws[w];
      const int OT = W.O + W.F;
      int* obs_pt = reinterpret_cast<int*>(lb) + L.obs_pt;
      int2* cam_obs = reinterpret_cast<int2*>(lb + b0) + L.cam_obs;
      int4* cam_items = reinterpret_cast<int4*>(lb + b0 + b1) + L.cam_items;
      int4* pairs = reinterpret_cast<int4*>(lb + b0 + b1 + b2) + L.pairs;
      int4* pair_items = reinterpret_cast<int4*>(lb + b0 + b1 + b2 + b3) + L.pair_items;
      const int* w_ptr = d_ptr + o_ptr[w];
      const int* w_cam = d_ocam + o_obs[w];
      DevListCounts cnt{};
      int* poff = nullptr;
      LORB_TRY(bld.phase1(W.C, W.P, OT, w_ptr, w_cam, obs_pt, cam_obs, cam_items, W.C + OT / 1024 + 1, &poff, &cnt));
      LORB_REQUIRE(cnt.n_pairs == L.n_pairs, "pair record count differs between host and device (internal)");
      LORB_TRY(bld.phase2(W.C, W.P, (int)L.n_pairs, w_ptr, w_cam, poff, &pb->list_scratch2, pairs, pair_items,
                          (int)(L.n_pairs / 2048) + W.C * (W.C + 1) / 2 + 1, &L.n_pair_items));
      L.n_cam_items = cnt.n_cam_items;
      d.obs_pt = obs_pt;
      d.cam_obs = cam_obs;
      d.cam_items = cam_items;
      d.pairs = pairs;
      d.pair_items = pair_items;
      d.n_cam_items = L.n_cam_items;
      d.n_pair_items = L.n_pair_items;
      pb->max_cam_items = std::max(pb->max_cam_items, L.n_cam_items);
      pb->max_pair_items = std::max(pb->max_pair_items, L.n_pair_items);
    }
    btr.mark("device work lists");
  }
  LORB_TRY(pb->descs.reserve(sizeof(BADev) * (size_t)nw));
  LORB_TRY(pb->counter.reserve(256));
  pb->hstate.pinned = true;
  LORB_TRY(pb->hstate.reserve(sizeof(LMState) * (size_t)nw + 64));
  LORB_CUDA_TRY(cudaMemcpyAsync(pb->descs.p, pb->h_dev.data(), sizeof(BADev) * (size_t)nw, cudaMemcpyHostToDevice, s));
  LORB_CUDA_TRY(cudaMemcpyAsync(pb->cams0, h_cams, pb->cam_doubles * 8, cudaMemcpyHostToDevice, s));
  LORB_CUDA_TRY(cudaMemcpyAsync(pb->pts0, h_pts, pb->pt_doubles * 8, cudaMemcpyHostToDevice, s));
  LORB_CUDA_TRY(cudaMemcpyAsync(d_uv, h_uv, tot_obs * 8, cudaMemcpyHostToDevice, s));
  LORB_CUDA_TRY(cudaMemcpyAsync(d_fix, h_fix, tot_fix * 96, cudaMemcpyHostToDevice, s));
  btr.mark("uploads queued");
  LORB_CUDA_TRY(cudaStreamSynchronize(s));  // host staging vectors go out of scope
  btr.mark("uploads done");
  return LORB_OK;
}

__global__ void fill_ones_kernel(double* a, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    a[i] = 1.0;
}

static int problem_reset(lorb_ba_problem* pb) {
  lorb_ctx* c = pb->ctx;
  const BADev& d0 = pb->h_dev[0];
  LORB_CUDA_TRY(cudaMemcpyAsync(d0.cams[0], pb->cams0, pb->cam_doubles * 8, cudaMemcpyDeviceToDevice, c->stream));
  if (pb->pt_doubles)
    LORB_CUDA_TRY(cudaMemcpyAsync(d0.pts[0], pb->pts0, pb->pt_doubles * 8, cudaMemcpyDeviceToDevice, c->stream));
  return LORB_OK;
}

static int run_cholesky(lorb_ba_problem* pb) {
  lorb_ctx* c = pb->ctx;
  const BADev* dp = pb->descs.as<BADev>();
  const int n = 6 * pb->maxC, nw = pb->nw;
  const size_t small_bytes = ((size_t)n * n + n) * 8;
  if (small_bytes <= 160 * 1024) {
    LORB_CUDA_TRY(cudaFuncSetAttribute(ba_chol_small_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)small_bytes));
    LORB_LAUNCH(c, ba_chol_small_kernel, dim3(1, nw), 256, small_bytes, dp);
    return LORB_OK;
  }
  const int nblk = (n + NB - 1) / NB;
  if (c->chol_chain_blocks < 0) {  // per context (= per device and calling thread)
    int per_sm = 0;
    LORB_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ba_chol_chain_kernel, 256, 0));
    c->chol_chain_blocks = per_sm * c->sm_count;
  }
  // one window, one CTA per block row of the solve co-resident, and at least one helper beside the chain CTA
  if (nw == 1 && nblk <= c->sm_count && c->chol_chain_blocks >= 2) {
    const int n_tiles = nblk * (nblk + 1) / 2;
    // tile flags [T*T], y / x flags [2T], partial flags [2T], forward-substitution partials [T][32]
    const size_t flag_ints = (size_t)nblk * nblk + 4 * (size_t)nblk + 2;
    LORB_TRY(dev_reserve(c, 14, flag_ints * 4 + (size_t)nblk * NB * 8));
    int* flags = c->d[14].as<int>();
    LORB_CUDA_TRY(cudaMemsetAsync(flags, 0, flag_ints * 4, c->stream));
    int T = nblk;
    int* sflags = flags + (size_t)nblk * nblk;  // y flags [T], x flags [T]
    int* pflag = sflags + 2 * (size_t)nblk;
    double* ypart = reinterpret_cast<double*>(flags + (((size_t)nblk * nblk + 4 * (size_t)nblk + 1) & ~(size_t)1));
    void* cargs[] = {(void*)&dp, (void*)&flags, (void*)&sflags, (void*)&pflag, (void*)&ypart, (void*)&T};
    LORB_CUDA_TRY(cudaLaunchCooperativeKernel((void*)ba_chol_chain_kernel,
                                              dim3(std::min(n_tiles + 1, c->chol_chain_blocks)), dim3(256), cargs, 0,
                                              c->stream));
    c->launches++;
    int fwd_done = 1;  // the factorisation kernel also ran the forward substitution
    void* args2[] = {(void*)&dp, (void*)&sflags, (void*)&T, (void*)&fwd_done};
    LORB_CUDA_TRY(cudaLaunchCooperativeKernel((void*)ba_trisolve_dataflow_kernel, dim3(nblk),
                                              dim3(256), args2, 0, c->stream));
    c->launches++;
    return LORB_OK;
  }
  for (int kb = 0; kb < nblk; kb++) {
    LORB_LAUNCH(c, ba_chol_panel_kernel, dim3(nblk - kb, nw), NB * NB / 4, 0, dp, kb);
    const int m = nblk - kb - 1;
    if (m > 0) LORB_LAUNCH(c, ba_chol_update_kernel, dim3(m * (m + 1) / 2, nw), 256, 0, dp, kb, nblk);
  }
  LORB_REQUIRE((size_t)n * 8 <= 200 * 1024, "reduced camera system too large for the solve kernel");
  LORB_CUDA_TRY(cudaFuncSetAttribute(ba_chol_solve_kernel,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, n * 8));
  LORB_LAUNCH(c, ba_chol_solve_kernel, dim3(1, nw), 1024, (size_t)n * 8, dp);
  return LORB_OK;
}

static int problem_solve(lorb_ba_problem* pb, const lorb_ba_options* optp, int sharded,
                         lorb_ba_summary* sums) {
  lorb_ctx* c = pb->ctx;
  const BADev* dp = pb->descs.as<BADev>();
  const BADev& d0 = pb->h_dev[0];
  const int nw = pb->nw;
  lorb_ba_options opt = *optp;
  LORB_REQUIRE(!sharded || (dist_ready(c) && nw == 1), "sharded solve needs lorb_dist_init and one window");

  {
    // the descriptor carries rank / world of a sharded solve (per-rank gradient slots)
    BADev& h0 = pb->h_dev[0];
    const int w_ = sharded ? dist_world(c) : 1, r_ = sharded ? dist_rank(c) : 0;
    LORB_REQUIRE(w_ <= 16, "sharded solve supports up to 16 ranks");
    if (h0.world != w_ || h0.rank != r_) {
      h0.world = w_;
      h0.rank = r_;
      LORB_CUDA_TRY(cudaMemcpyAsync(pb->descs.p, &h0, sizeof(BADev), cudaMemcpyHostToDevice, c->stream));
    }
  }
  // the robust loss is the ctx's at solve time: every window's descriptor carries it
  const lorb_ba_loss loss = c->ba_loss;
  const bool robust = loss.kind != LORB_LOSS_TRIVIAL;
  {
    bool changed = false;
    for (BADev& d : pb->h_dev) {
      changed |= d.loss_kind != loss.kind || d.loss_scale != loss.scale;
      d.loss_kind = loss.kind;
      d.loss_scale = loss.scale;
    }
    if (changed)
      LORB_CUDA_TRY(cudaMemcpyAsync(pb->descs.p, pb->h_dev.data(), sizeof(BADev) * (size_t)nw,
                                    cudaMemcpyHostToDevice, c->stream));
  }
  // kernel instantiation for the loss: ROBUST = false is plain least squares, unchanged
#define LORB_BA_K(K_, ...) (robust ? K_<__VA_ARGS__, true> : K_<__VA_ARGS__, false>)
  const int gx_pts = std::max(1, std::min((pb->maxP + 31) / 32, std::max(1, c->sm_count * 8 / nw)));
  const dim3 grid_pts(gx_pts, nw);
  // back-substitution with the cameras in shared memory: two CTAs per SM must fit (C <= 203); a CTA
  // of a large window copies 100 KB, so such a launch is just the co-resident CTAs, grid-striding
  const size_t backsub_smem = (size_t)pb->maxC * CS_BACKSUB * 8;
  const bool backsub_cs = backsub_smem <= 100 * 1024;
  if (backsub_cs && backsub_smem > 40 * 1024)
    LORB_CUDA_TRY(cudaFuncSetAttribute(LORB_BA_K(ba_backsub_kernel, true), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)backsub_smem));
  const dim3 grid_backsub(backsub_smem > 16 * 1024 ? std::min(gx_pts, std::max(1, 2 * c->sm_count / nw)) : gx_pts, nw);
  const int ppc = DP_THREADS / 8;  // points per CTA round of the dense path
  // CTAs per window of the dense build: a CTA pays about two rounds' worth of prologue, reduction
  // and flush, and CTAs run in waves of one per SM -- minimise waves x (rounds per CTA + 2)
  int gx_dense = 1;
  {
    const int gx_hi = std::max(1, std::min((pb->maxP + ppc - 1) / ppc, std::max(1, c->sm_count * 8 / nw)));
    long long best = -1;
    for (int g = 1; g <= gx_hi; g++) {
      const long long waves = ((long long)nw * g + c->sm_count - 1) / c->sm_count;
      const long long cost = waves * ((pb->maxP + (long long)ppc * g - 1) / ((long long)ppc * g) + 2);
      if (best < 0 || cost < best) {
        best = cost;
        gx_dense = g;
      }
    }
  }
  const dim3 grid_dense(gx_dense, nw);
  const dim3 grid_cam((pb->maxC + 127) / 128, nw);
  const int nmax = 6 * pb->maxC;
  const dim3 grid_fin(std::max(1, std::min(c->sm_count * 2 / std::min(nw, c->sm_count) + 1, (nmax * nmax + 255) / 256)), nw);
  cudaStream_t s = c->stream;
  int* d_active = pb->counter.as<int>();
  int* h_active = reinterpret_cast<int*>(pb->hstate.as<uint8_t>() + sizeof(LMState) * (size_t)nw);
  // small windows: shared-memory privatised accumulation + one fused solve kernel
  const bool small = nmax <= 96;
  const int acc_mode = (nmax <= DENSE_N && !pb->has_dup) ? 2 : (small ? 1 : 3);
  const size_t wsm_bytes = (size_t)BA_THREADS * 18 * 8;
  const size_t lin_small = (size_t)(HCC + 12) * pb->maxC;
  const size_t smem_build_full =
      acc_mode == 2 ? (size_t)DP_SMEM_DOUBLES * 8
                    : (acc_mode == 1 ? ((size_t)nmax * nmax + lin_small) * 8 + wsm_bytes : 0);
  const size_t smem_build_init =
      acc_mode == 2 ? (size_t)DP_SMEM_DOUBLES * 8
                    : (acc_mode == 1 ? ((size_t)nmax * nmax + lin_small) * 8 + wsm_bytes : 0);
  const size_t smem_solve = ((size_t)nmax * nmax + 2 * (size_t)nmax + NB + (size_t)((nmax + NB - 1) / NB) * NB * (NB + 1)) * 8;
#define LORB_BUILD_ATTR(FULL_, ACC_, BYTES_)                                                  \
  LORB_CUDA_TRY(cudaFuncSetAttribute(LORB_BA_K(ba_build_kernel, FULL_, ACC_),                 \
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(BYTES_))); \
  LORB_CUDA_TRY(cudaFuncSetAttribute(LORB_BA_K(ba_build_kernel, FULL_, ACC_),                 \
                                     cudaFuncAttributePreferredSharedMemoryCarveout,           \
                                     (int)cudaSharedmemCarveoutMaxShared))
  if (acc_mode == 2) {
    LORB_CUDA_TRY(cudaFuncSetAttribute(LORB_BA_K(ba_build_dense_kernel, true), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)(DP_SMEM_DOUBLES * 8)));
    LORB_CUDA_TRY(cudaFuncSetAttribute(LORB_BA_K(ba_build_dense_kernel, false), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)(DP_SMEM_DOUBLES * 8)));
  } else if (acc_mode == 1) {
    LORB_BUILD_ATTR(true, 1, smem_build_full);
    LORB_BUILD_ATTR(false, 1, smem_build_init);
  }
#undef LORB_BUILD_ATTR
  if (small)
    LORB_CUDA_TRY(cudaFuncSetAttribute(ba_solve_small_kernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_solve));
  auto launch_build = [&](bool full, int force) -> int {
    const size_t sm = full ? smem_build_full : smem_build_init;
#define LORB_BUILD(FULL_, ACC_) \
  LORB_LAUNCH(c, LORB_BA_K(ba_build_kernel, FULL_, ACC_), grid_pts, BA_THREADS, sm, dp, opt, force)
    if (acc_mode == 2) {
      if (full) LORB_LAUNCH(c, LORB_BA_K(ba_build_dense_kernel, true), grid_dense, DP_THREADS, DP_SMEM_DOUBLES * 8, dp, opt, force);
      else      LORB_LAUNCH(c, LORB_BA_K(ba_build_dense_kernel, false), grid_dense, DP_THREADS, DP_SMEM_DOUBLES * 8, dp, opt, force);
    } else if (acc_mode == 1) {
      if (full) LORB_BUILD(true, 1); else LORB_BUILD(false, 1);
    } else {
      // large path: point side, then camera side and Schur products from the work lists
      if (full) LORB_LAUNCH(c, LORB_BA_K(ba_build_kernel, true, 3), grid_pts, BA_THREADS, 0, dp, opt, force);
      else      LORB_LAUNCH(c, LORB_BA_K(ba_build_kernel, false, 3), grid_pts, BA_THREADS, 0, dp, opt, force);
      // camera rows (H_cc, g_c, Schur rhs) and Schur pairs (S) both need only the point side and write
      // disjoint outputs; both are latency-bound gathers, so the camera rows run on a side stream
      // beside the (six times longer) pair pass
      const bool side = full && pb->max_cam_items > 0 && pb->max_pair_items > 0;
      if (side) {
        if (!c->ba_stream2) {
          LORB_CUDA_TRY(cudaStreamCreateWithFlags(&c->ba_stream2, cudaStreamNonBlocking));
          for (auto& e : c->ba_ev) LORB_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        }
        LORB_CUDA_TRY(cudaEventRecord(c->ba_ev[0], c->stream));
        LORB_CUDA_TRY(cudaStreamWaitEvent(c->ba_stream2, c->ba_ev[0], 0));
        (robust ? ba_cam_rows_kernel<true> : ba_cam_rows_kernel<false>)
            <<<dim3((pb->max_cam_items + 7) / 8, nw), 256, 0, c->ba_stream2>>>(dp, 1, force);
        c->launches++;
        LORB_CUDA_TRY(cudaGetLastError());
        LORB_CUDA_TRY(cudaEventRecord(c->ba_ev[1], c->ba_stream2));
      } else if (pb->max_cam_items > 0) {
        LORB_LAUNCH(c, (robust ? ba_cam_rows_kernel<true> : ba_cam_rows_kernel<false>),
                    dim3((pb->max_cam_items + 7) / 8, nw), 256, 0, dp,
                    full ? 1 : 0, force);
      }
      if (full && pb->max_pair_items > 0)
        LORB_LAUNCH(c, (robust ? ba_schur_pairs_kernel<true> : ba_schur_pairs_kernel<false>),
                    dim3((pb->max_pair_items + 7) / 8, nw), 256, 0, dp);
      if (side) LORB_CUDA_TRY(cudaStreamWaitEvent(c->stream, c->ba_ev[1], 0));
    }
#undef LORB_BUILD
    return LORB_OK;
  };
  // ---- initial evaluation (iteration 0)
  LORB_CUDA_TRY(cudaMemsetAsync(pb->d_states, 0, sizeof(LMState) * (size_t)nw, s));
  LORB_CUDA_TRY(cudaMemsetAsync(pb->lin_base, 0, pb->lin_bytes_total, s));
  LORB_LAUNCH(c, fill_ones_kernel, 128, 256, 0, d0.scale_c, pb->cam_doubles);
  LORB_LAUNCH(c, fill_ones_kernel, 512, 256, 0, d0.scale_p, pb->pt_doubles);
  LORB_LAUNCH(c, ba_camrot_kernel, grid_cam, 128, 0, dp, 0, 1);
  LORB_TRY(launch_build(false, 1));
  if (sharded) {  // one collective: sums and, through the per-rank slots, the gradient maximum
    LORB_LAUNCH(c, ba_gslot_kernel, 1, 1, 0, dp);
    LORB_TRY(dist_allreduce_sum(c, d0.Hcc, (size_t)HCC * d0.C + 12 * (size_t)d0.C + 24));
  }
  LORB_LAUNCH(c, ba_init_finish_kernel, dim3(1, nw), 1024, 0, dp, opt);
  // ---- LM attempts; the device decides, the host polls a counter every few attempts
  const int poll_every = 4;
  const int fuse_control = sharded ? 0 : 1;
  for (int it = 0; it < opt.max_num_iterations; it++) {
    LORB_CUDA_TRY(cudaMemsetAsync(pb->lin_base, 0, pb->lin_bytes_total, s));
    LORB_CUDA_TRY(cudaMemsetAsync(d_active, 0, 4, s));
    prof_begin(c, 0);
    LORB_TRY(launch_build(true, 0));
    prof_end(c, 0);
    if (sharded) {  // ONE all-reduce per build pass: packed S, H_cc, g_c, Schur rhs, scalars, gradient slots
      prof_begin(c, 4);
      LORB_LAUNCH(c, ba_gslot_kernel, 1, 1, 0, dp);
      LORB_TRY(dist_allreduce_sum(c, d0.lin, pb->lin_doubles_max));
      prof_end(c, 4);
    }
    prof_begin(c, 2);
    if (small) {
      LORB_LAUNCH(c, ba_solve_small_kernel, dim3(1, nw), 256, smem_solve, dp, opt);
    } else {
      LORB_LAUNCH(c, ba_gradcheck_kernel, dim3(1, nw), 256, 0, dp, opt, 0);
      LORB_LAUNCH(c, ba_finish_kernel, grid_fin, 256, 0, dp, opt);
      LORB_TRY(run_cholesky(pb));
      LORB_LAUNCH(c, ba_candcam_kernel, dim3(1, nw), 128, 0, dp);
    }
    prof_end(c, 2);
    prof_begin(c, 1);
    if (backsub_cs)
      LORB_LAUNCH(c, LORB_BA_K(ba_backsub_kernel, true), grid_backsub, BA_THREADS, backsub_smem, dp, opt, fuse_control,
                  d_active);
    else
      LORB_LAUNCH(c, LORB_BA_K(ba_backsub_kernel, false), grid_pts, BA_THREADS, 0, dp, opt, fuse_control, d_active);
    prof_end(c, 1);
    if (sharded) {
      prof_begin(c, 4);
      LORB_TRY(dist_allreduce_sum(c, &d0.st->acc_cost2, 4));
      LORB_LAUNCH(c, ba_control_kernel, nw, 1, 0, dp, opt, d_active);
      prof_end(c, 4);
    }
    if ((it + 1) % poll_every == 0 && it + 1 < opt.max_num_iterations) {
      // every rank takes the same decisions (same bits in, see ba_candcam_kernel); the max over
      // the ranks makes leaving the loop a collective decision whatever happens
      if (sharded) LORB_TRY(dist_allreduce_max_i32(c, d_active, 1));
      LORB_CUDA_TRY(cudaMemcpyAsync(h_active, d_active, 4, cudaMemcpyDeviceToHost, s));
      LORB_CUDA_TRY(cudaStreamSynchronize(s));
      if (*h_active == 0) break;
    }
  }
  // gradient at the final point of windows whose last attempt moved it (Ceres tests the
  // gradient tolerance on acceptance); windows without a pending check ignore the pass
  LMState* hs = pb->hstate.as<LMState>();
  LORB_CUDA_TRY(cudaMemcpyAsync(hs, pb->d_states, sizeof(LMState) * (size_t)nw, cudaMemcpyDeviceToHost, s));
  LORB_CUDA_TRY(cudaStreamSynchronize(s));
  bool pending = false;
  for (int w = 0; w < nw; w++) pending |= hs[w].check_gradient != 0;
  if (pending) {
    LORB_CUDA_TRY(cudaMemsetAsync(pb->lin_base, 0, pb->lin_bytes_total, s));
    LORB_LAUNCH(c, ba_camrot_kernel, grid_cam, 128, 0, dp, 0, 2);
    LORB_TRY(launch_build(false, 2));
    if (sharded) {
      LORB_LAUNCH(c, ba_gslot_kernel, 1, 1, 0, dp);
      LORB_TRY(dist_allreduce_sum(c, d0.Hcc, (size_t)HCC * d0.C + 12 * (size_t)d0.C + 24));
    }
    LORB_LAUNCH(c, ba_gradcheck_kernel, dim3(1, nw), 256, 0, dp, opt, 2);
    LORB_CUDA_TRY(cudaMemcpyAsync(hs, pb->d_states, sizeof(LMState) * (size_t)nw, cudaMemcpyDeviceToHost, s));
    LORB_CUDA_TRY(cudaStreamSynchronize(s));
  }
  // make buffer 0 the current one so download / the next solve find the result there
  bool any_cur1 = false;
  for (int w = 0; w < nw; w++) any_cur1 |= hs[w].cur == 1;
  if (any_cur1)
    LORB_LAUNCH(c, ba_make_current_kernel, dim3(std::max(1, std::min(64, (3 * pb->maxP + 255) / 256)), nw), 256, 0, dp);
  for (int w = 0; w < nw; w++) {
    if (sums) {
      lorb_ba_summary& sum = sums[w];
      sum.initial_cost = hs[w].initial_cost;
      sum.final_cost = hs[w].cost;
      sum.final_radius = hs[w].radius;
      sum.final_gradient_max_norm = hs[w].gmax;
      sum.iterations = hs[w].iteration;
      sum.num_successful_steps = hs[w].n_success;
      sum.num_unsuccessful_steps = hs[w].n_fail;
      sum.termination = hs[w].termination;
    }
  }
  LORB_CUDA_TRY(cudaStreamSynchronize(s));
  return LORB_OK;
#undef LORB_BA_K
}

// The host-buffer entry points (lorb_ba_local, lorb_ba_local_batched) reuse one
// problem object per ctx: its device / pinned buffers only ever grow, so a
// steady stream of windows allocates nothing.
static lorb_ba_problem* cached_problem(lorb_ctx* c) {
  if (!c->ba_cache) c->ba_cache = new (std::nothrow) lorb_ba_problem();
  return static_cast<lorb_ba_problem*>(c->ba_cache);
}

static void problem_free(lorb_ba_problem* pb) {
  if (!pb) return;
  if (pb->ctx) {
    cudaSetDevice(pb->ctx->device);
    cudaStreamSynchronize(pb->ctx->stream);
  }
  pb->params.release();
  pb->topo.release();
  pb->work.release();
  pb->descs.release();
  pb->lists.release();
  pb->stage.release();
  pb->list_scratch.release();
  pb->list_scratch2.release();
  pb->hstate.release();
  pb->counter.release();
  delete pb;
}

void ba_cache_free(lorb_ctx* c) {
  if (c && c->ba_cache) {
    problem_free(static_cast<lorb_ba_problem*>(c->ba_cache));
    c->ba_cache = nullptr;
  }
  if (c && c->ba_stream2) {
    cudaStreamDestroy(c->ba_stream2);
    c->ba_stream2 = nullptr;
    for (auto& e : c->ba_ev) {
      if (e) cudaEventDestroy(e);
      e = nullptr;
    }
  }
}

}  // namespace lorb

extern "C" {

int lorb_ba_problem_create(lorb_ctx* c, int C, const double* cams, int P, const double* pts, int O,
                           const int* obs_cam, const int* obs_pt, const float* obs_uv, int F,
                           const int* fix_pt, const float* fix_uv, const float* fix_rt,
                           const float* K, lorb_ba_problem** out) {
  LORB_REQUIRE(c && out && K, "ctx / out / K");
  LORB_REQUIRE(C > 0 && P >= 0 && O >= 0 && F >= 0, "sizes");
  LORB_REQUIRE(cams && (P == 0 || pts), "parameters");
  LORB_REQUIRE(O == 0 || (obs_cam && obs_pt && obs_uv), "observations");
  LORB_REQUIRE(F == 0 || (fix_pt && fix_uv && fix_rt), "fixed observations");
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  lorb_ba_problem* pb = new (std::nothrow) lorb_ba_problem();
  if (!pb) return LORB_ERR_NOMEM;
  std::vector<WindowSpec> ws(1);
  ws[0] = WindowSpec{C, P, O, F, cams, pts, obs_cam, obs_pt, obs_uv, fix_pt, fix_uv, fix_rt};
  int rc = problem_build(pb, c, ws, K);
  if (rc == LORB_OK) rc = problem_reset(pb);
  if (rc != LORB_OK) {
    problem_free(pb);
    return rc;
  }
  *out = pb;
  return LORB_OK;
}

int lorb_shard_range(long long n, int rank, int world, long long* lo, long long* hi) {
  LORB_REQUIRE(n >= 0 && world >= 1 && rank >= 0 && rank < world && lo && hi, "arguments");
  const long long base = n / world, rem = n % world;
  *lo = rank * base + std::min<long long>(rank, rem);
  *hi = *lo + base + (rank < rem ? 1 : 0);
  return LORB_OK;
}

// Which points go to which rank.  Any partition of the points (each with all its observations) is a
// valid shard; this one keeps a rank's points together along the trajectory: points are ordered by
// the lowest window camera that observes them (ties by point index) and that order is cut into
// `world` runs of equal observation count.  A rank then touches a band of cameras -- its camera /
// camera-pair work lists are ~world times shorter than with an arbitrary split, where every rank
// meets every camera pair -- and the ranks carry the same number of observations.
int lorb_ba_shard_points(int P, int O, const int* obs_cam, const int* obs_pt, int rank, int world,
                         int* out_point_ids, int* n_out) {
  LORB_REQUIRE(P >= 0 && O >= 0 && world >= 1 && rank >= 0 && rank < world && n_out, "arguments");
  LORB_REQUIRE(O == 0 || (obs_cam && obs_pt), "observations");
  std::vector<int> key((size_t)P, 0x7fffffff), cnt((size_t)P, 0);
  for (int o = 0; o < O; o++) {
    LORB_REQUIRE(obs_pt[o] >= 0 && obs_pt[o] < P, "observation point index");
    key[obs_pt[o]] = std::min(key[obs_pt[o]], obs_cam[o]);
    cnt[obs_pt[o]]++;
  }
  std::vector<int> order((size_t)P);
  for (int p = 0; p < P; p++) order[p] = p;
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return key[a] < key[b]; });
  // cut k ends at the first position where the running observation count reaches k * O / world
  // (points without observations follow the last observed point into the last rank)
  long long run = 0;
  int n = 0, r = 0;
  for (int i = 0; i < P; i++) {
    const int p = order[i];
    while (r + 1 < world && run >= (long long)O * (r + 1) / world && (run > 0 || O == 0)) r++;
    if (O == 0) r = (int)((long long)i * world / std::max(1, P));
    if (r == rank) {
      if (out_point_ids) out_point_ids[n] = p;
      n++;
    }
    run += cnt[p];
  }
  *n_out = n;
  return LORB_OK;
}

int lorb_ba_problem_create_sharded(lorb_ctx* c, int C, const double* cams, int P, const double* pts,
                                   int O, const int* obs_cam, const int* obs_pt, const float* obs_uv,
                                   int F, const int* fix_pt, const float* fix_uv, const float* fix_rt,
                                   const float* K, int rank, int world, lorb_ba_problem** out,
                                   int* out_point_ids, int* n_points) {
  LORB_REQUIRE(c && out && K && out_point_ids && n_points, "ctx / out / K / point ids");
  LORB_REQUIRE(C > 0 && P >= 0 && O >= 0 && F >= 0, "sizes");
  LORB_REQUIRE(O == 0 || (obs_cam && obs_pt && obs_uv), "observations");
  LORB_REQUIRE(F == 0 || (fix_pt && fix_uv && fix_rt), "fixed observations");
  LORB_REQUIRE(P == 0 || pts, "points");
  int n = 0;
  LORB_TRY(lorb_ba_shard_points(P, O, obs_cam, obs_pt, rank, world, out_point_ids, &n));
  *n_points = n;
  std::vector<int> local((size_t)P, -1);
  for (int i = 0; i < n; i++) local[out_point_ids[i]] = i;
  std::vector<double> spts((size_t)n * 3);
  for (int i = 0; i < n; i++)
    for (int a = 0; a < 3; a++) spts[3 * (size_t)i + a] = pts[3 * (size_t)out_point_ids[i] + a];
  // observations of the shard, grouped by local point (counting sort keeps their input order)
  std::vector<int> start((size_t)n + 1, 0);
  for (int o = 0; o < O; o++)
    if (local[obs_pt[o]] >= 0) start[local[obs_pt[o]] + 1]++;
  for (int i = 0; i < n; i++) start[i + 1] += start[i];
  const int no = start[n];
  std::vector<int> oc((size_t)no), op((size_t)no), fill(start.begin(), start.end() - 1), fp;
  std::vector<float> ouv((size_t)no * 2), fuv, frt;
  for (int o = 0; o < O; o++) {
    const int l = local[obs_pt[o]];
    if (l < 0) continue;
    const int d = fill[l]++;
    oc[d] = obs_cam[o];
    op[d] = l;
    ouv[2 * (size_t)d] = obs_uv[2 * (size_t)o];
    ouv[2 * (size_t)d + 1] = obs_uv[2 * (size_t)o + 1];
  }
  for (int f = 0; f < F; f++) {
    LORB_REQUIRE(fix_pt[f] >= 0 && fix_pt[f] < P, "fixed observation point index");
    if (local[fix_pt[f]] < 0) continue;
    fp.push_back(local[fix_pt[f]]);
    fuv.insert(fuv.end(), fix_uv + 2 * (size_t)f, fix_uv + 2 * (size_t)f + 2);
    frt.insert(frt.end(), fix_rt + 6 * (size_t)f, fix_rt + 6 * (size_t)f + 6);
  }
  return lorb_ba_problem_create(c, C, cams, n, spts.data(), no, oc.data(), op.data(), ouv.data(), (int)fp.size(),
                                fp.data(), fuv.data(), frt.data(), K, out);
}

int lorb_ba_problem_reset(lorb_ba_problem* pb) {
  LORB_REQUIRE(pb, "problem");
  LORB_CUDA_TRY(cudaSetDevice(pb->ctx->device));
  return problem_reset(pb);
}

int lorb_ba_problem_solve(lorb_ba_problem* pb, const lorb_ba_options* opt, int sharded,
                          lorb_ba_summary* summary) {
  LORB_REQUIRE(pb && opt, "problem / options");
  LORB_CUDA_TRY(cudaSetDevice(pb->ctx->device));
  return problem_solve(pb, opt, sharded, summary);
}

int lorb_ba_problem_download(lorb_ba_problem* pb, double* cams, double* pts) {
  LORB_REQUIRE(pb, "problem");
  lorb_ctx* c = pb->ctx;
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  const BADev& d0 = pb->h_dev[0];
  const size_t cb = pb->cam_doubles * 8, pbytes = (pts ? pb->pt_doubles : 0) * 8;
  if (cb + pbytes >= ((size_t)4 << 20) && pb->h_cams_stage) {
    // a large result goes through the pinned staging block (a device-to-pageable copy runs at a
    // fraction of the link) and is handed to the caller's arrays by the host threads
    if (cams) LORB_CUDA_TRY(cudaMemcpyAsync(pb->h_cams_stage, d0.cams[0], cb, cudaMemcpyDeviceToHost, c->stream));
    if (pbytes) LORB_CUDA_TRY(cudaMemcpyAsync(pb->h_pts_stage, d0.pts[0], pbytes, cudaMemcpyDeviceToHost, c->stream));
    LORB_CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (cams) memcpy(cams, pb->h_cams_stage, cb);
    if (pbytes) {
      const int nchunk = 64;
#pragma omp parallel for schedule(static)
      for (int ch = 0; ch < nchunk; ch++) {
        const size_t i0 = pbytes / 8 * ch / nchunk, i1 = pbytes / 8 * (ch + 1) / nchunk;
        memcpy(pts + i0, pb->h_pts_stage + i0, (i1 - i0) * 8);
      }
    }
    return LORB_OK;
  }
  if (cams)
    LORB_CUDA_TRY(cudaMemcpyAsync(cams, d0.cams[0], pb->cam_doubles * 8, cudaMemcpyDeviceToHost, c->stream));
  if (pts && pb->pt_doubles)
    LORB_CUDA_TRY(cudaMemcpyAsync(pts, d0.pts[0], pb->pt_doubles * 8, cudaMemcpyDeviceToHost, c->stream));
  LORB_CUDA_TRY(cudaStreamSynchronize(c->stream));
  return LORB_OK;
}

int lorb_ba_problem_destroy(lorb_ba_problem* pb) {
  problem_free(pb);
  return LORB_OK;
}

int lorb_ba_local(lorb_ctx* c, int C, double* cams, int P, double* pts, int O, const int* obs_cam,
                  const int* obs_pt, const float* obs_uv, int F, const int* fix_pt,
                  const float* fix_uv, const float* fix_rt, const float* K,
                  const lorb_ba_options* opt, lorb_ba_summary* summary) {
  LORB_REQUIRE(c && opt && K, "ctx / options / K");
  LORB_REQUIRE(C > 0 && P >= 0 && O >= 0 && F >= 0, "sizes");
  LORB_REQUIRE(cams && (P == 0 || pts), "parameters");
  LORB_REQUIRE(O == 0 || (obs_cam && obs_pt && obs_uv), "observations");
  LORB_REQUIRE(F == 0 || (fix_pt && fix_uv && fix_rt), "fixed observations");
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  lorb_ba_problem* pb = cached_problem(c);
  if (!pb) return LORB_ERR_NOMEM;
  std::vector<WindowSpec> ws(1);
  ws[0] = WindowSpec{C, P, O, F, cams, pts, obs_cam, obs_pt, obs_uv, fix_pt, fix_uv, fix_rt};
  LORB_TRY(problem_build(pb, c, ws, K));
  LORB_TRY(problem_reset(pb));
  LORB_TRY(problem_solve(pb, opt, 0, summary));
  return lorb_ba_problem_download(pb, cams, pts);
}

// Host-buffer form of the sharded solve: the arrays are THIS RANK'S shard (points with all their
// observations, every camera), e.g. as cut by lorb_shard_range; collective over the ctx communicator.
int lorb_ba_local_shard(lorb_ctx* c, int C, double* cams, int P, double* pts, int O, const int* obs_cam,
                        const int* obs_pt, const float* obs_uv, int F, const int* fix_pt,
                        const float* fix_uv, const float* fix_rt, const float* K,
                        const lorb_ba_options* opt, lorb_ba_summary* summary) {
  LORB_REQUIRE(c && opt && K, "ctx / options / K");
  LORB_REQUIRE(dist_ready(c), "lorb_dist_init was not called");
  LORB_REQUIRE(C > 0 && P >= 0 && O >= 0 && F >= 0, "sizes");
  LORB_REQUIRE(cams && (P == 0 || pts), "parameters");
  LORB_REQUIRE(O == 0 || (obs_cam && obs_pt && obs_uv), "observations");
  LORB_REQUIRE(F == 0 || (fix_pt && fix_uv && fix_rt), "fixed observations");
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  lorb_ba_problem* pb = cached_problem(c);
  if (!pb) return LORB_ERR_NOMEM;
  std::vector<WindowSpec> ws(1);
  ws[0] = WindowSpec{C, P, O, F, cams, pts, obs_cam, obs_pt, obs_uv, fix_pt, fix_uv, fix_rt};
  LORB_TRY(problem_build(pb, c, ws, K));
  LORB_TRY(problem_reset(pb));
  LORB_TRY(problem_solve(pb, opt, 1, summary));
  return lorb_ba_problem_download(pb, cams, pts);
}

static int batched_specs(std::vector<WindowSpec>& ws, int n_windows, const int* cam_off,
                         const double* cams, const int* pt_off, const double* pts,
                         const int* obs_off, const int* obs_cam, const int* obs_pt,
                         const float* obs_uv, const int* fix_off, const int* fix_pt,
                         const float* fix_uv, const float* fix_rt) {
  LORB_REQUIRE(n_windows > 0 && cam_off && pt_off && obs_off && cams, "window offsets");
  ws.resize((size_t)n_windows);
  for (int w = 0; w < n_windows; w++) {
    WindowSpec& W = ws[w];
    W.C = cam_off[w + 1] - cam_off[w];
    W.P = pt_off[w + 1] - pt_off[w];
    W.O = obs_off[w + 1] - obs_off[w];
    W.F = fix_off ? fix_off[w + 1] - fix_off[w] : 0;
    W.cams = cams + 6 * (size_t)cam_off[w];
    W.pts = pts ? pts + 3 * (size_t)pt_off[w] : nullptr;
    W.obs_cam = obs_cam + obs_off[w];
    W.obs_pt = obs_pt + obs_off[w];
    W.obs_uv = obs_uv + 2 * (size_t)obs_off[w];
    W.fix_pt = fix_off ? fix_pt + fix_off[w] : nullptr;
    W.fix_uv = fix_off ? fix_uv + 2 * (size_t)fix_off[w] : nullptr;
    W.fix_rt = fix_off ? fix_rt + 6 * (size_t)fix_off[w] : nullptr;
  }
  return LORB_OK;
}

int lorb_ba_problem_create_batched(lorb_ctx* c, int n_windows, const int* cam_off,
                                   const double* cams, const int* pt_off, const double* pts,
                                   const int* obs_off, const int* obs_cam, const int* obs_pt,
                                   const float* obs_uv, const int* fix_off, const int* fix_pt,
                                   const float* fix_uv, const float* fix_rt, const float* K,
                                   lorb_ba_problem** out) {
  LORB_REQUIRE(c && out && K, "ctx / out / K");
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  std::vector<WindowSpec> ws;
  LORB_TRY(batched_specs(ws, n_windows, cam_off, cams, pt_off, pts, obs_off, obs_cam, obs_pt, obs_uv,
                         fix_off, fix_pt, fix_uv, fix_rt));
  lorb_ba_problem* pb = new (std::nothrow) lorb_ba_problem();
  if (!pb) return LORB_ERR_NOMEM;
  int rc = problem_build(pb, c, ws, K);
  if (rc == LORB_OK) rc = problem_reset(pb);
  if (rc != LORB_OK) {
    problem_free(pb);
    return rc;
  }
  *out = pb;
  return LORB_OK;
}

int lorb_ba_local_batched(lorb_ctx* c, int n_windows, const int* cam_off, double* cams,
                          const int* pt_off, double* pts, const int* obs_off, const int* obs_cam,
                          const int* obs_pt, const float* obs_uv, const int* fix_off,
                          const int* fix_pt, const float* fix_uv, const float* fix_rt,
                          const float* K, const lorb_ba_options* opt, lorb_ba_summary* summaries) {
  LORB_REQUIRE(c && opt && K, "ctx / options / K");
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  std::vector<WindowSpec> ws;
  LORB_TRY(batched_specs(ws, n_windows, cam_off, cams, pt_off, pts, obs_off, obs_cam, obs_pt, obs_uv,
                         fix_off, fix_pt, fix_uv, fix_rt));
  lorb_ba_problem* pb = cached_problem(c);
  if (!pb) return LORB_ERR_NOMEM;
  LORB_TRY(problem_build(pb, c, ws, K));
  LORB_TRY(problem_reset(pb));
  LORB_TRY(problem_solve(pb, opt, 0, summaries));
  return lorb_ba_problem_download(pb, cams, pts);
}

/* Team size of the host-side staging loops (OpenMP) of the calling thread.  A launcher such as
 * torchrun exports OMP_NUM_THREADS=1 to every rank; a host that knows how many ranks share the
 * box gives each its share of the cores here. */
int lorb_set_host_threads(int n) {
  LORB_REQUIRE(n >= 1, "n");
  omp_set_num_threads(n);
  return LORB_OK;
}

}  // extern "C"
