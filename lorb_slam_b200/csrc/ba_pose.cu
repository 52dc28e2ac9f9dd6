// ba_pose.cu — pose-only bundle adjustment on sm_100a.
//
// Replaces the Ceres solve inside BA::ProjectPoseOptimization (reference
// src/bundle_adjust.cpp:158-202): one residual per matched keypoint with the
// PoseCost functor (:22-64) — which uses fx for the v coordinate (:51), kept
// as is — two parameter blocks R[3], T[3], Ceres defaults + DENSE_SCHUR.
// With six unknowns the whole trust-region loop fits one CTA: observations are
// streamed from HBM/L2, the 6x6 normal equations are reduced with warp
// shuffles, thread 0 runs the LM bookkeeping and the 6x6 Cholesky.  One launch
// per call, no host round trips inside the solve.
#include "ba_math.cuh"

namespace lorb {

constexpr int POSE_THREADS = 256;
constexpr int NRED = 28;  // 21 (H upper) + 6 (g) + 1 (cost)

struct PoseShared {
  LMState st;
  double rot[2][CAMROT];
  double x[2][6];
  double scale[6];
  double H[21], g[6];
  double red[POSE_THREADS / 32][NRED];
};

// sum r^2 (and optionally H, g) over all observations at pose `b`.  ROBUST: sum rho(|r|^2) and the
// H, g of the residuals and Jacobians corrected by the loss (kind, a) (robust_correct).
template <bool LIN, bool ROBUST>
__device__ __forceinline__ void pose_pass(PoseShared& sm, int b, int n, const float* __restrict__ xw,
                                          const float* __restrict__ uv, const Intr& K, int kind, double a,
                                          double* out) {
  double acc[NRED];
#pragma unroll
  for (int i = 0; i < NRED; i++) acc[i] = 0.0;
  const double t[3] = {sm.x[b][3], sm.x[b][4], sm.x[b][5]};
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double X[3] = {(double)xw[3 * i], (double)xw[3 * i + 1], (double)xw[3 * i + 2]};
    const double u = (double)uv[2 * i], v = (double)uv[2 * i + 1];
    if (LIN) {
      double r[2], Jc[12];
      obs_eval<true, false>(sm.rot[b], t, X, K, u, v, r, Jc, nullptr);
      double rho = 0.0;
      if (ROBUST) rho = robust_correct(kind, a, r, Jc, nullptr);
      int k = 0;
#pragma unroll
      for (int a = 0; a < 6; a++) {
#pragma unroll
        for (int c = a; c < 6; c++) acc[k++] += Jc[a] * Jc[c] + Jc[6 + a] * Jc[6 + c];
        acc[21 + a] += Jc[a] * r[0] + Jc[6 + a] * r[1];
      }
      acc[27] += ROBUST ? rho : r[0] * r[0] + r[1] * r[1];
    } else {
      const double s = obs_cost(sm.rot[b], t, X, K, u, v);
      if (ROBUST) {
        double rho, rho1;
        loss_eval(kind, a, s, rho, rho1);
        acc[27] += rho;
      } else {
        acc[27] += s;
      }
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = LIN ? 0 : 27; i < NRED; i++) {
    double v = acc[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) sm.red[warp][i] = v;
  }
  __syncthreads();
  if (threadIdx.x < NRED && (LIN || threadIdx.x == 27)) {
    double v = 0;
    for (int w = 0; w < POSE_THREADS / 32; w++) v += sm.red[w][threadIdx.x];
    out[threadIdx.x] = v;
  }
  __syncthreads();
}

__device__ __forceinline__ int uidx(int a, int b) { return a * 6 - (a * (a - 1)) / 2 + (b - a); }

// ROBUST = false: plain least squares (the reference); true: the loss (kind, a), LORB_LOSS_*
template <bool ROBUST>
__global__ void __launch_bounds__(POSE_THREADS)
    pose_only_kernel(int n, const float* __restrict__ xw, const float* __restrict__ uv, Intr K,
                     double* __restrict__ rt, lorb_ba_options opt, lorb_ba_summary* __restrict__ sum, int kind,
                     double a) {
  __shared__ PoseShared sm;
  __shared__ double lin[NRED];
  const int tid = threadIdx.x;
  LMState& st = sm.st;
  if (tid < 6) sm.x[0][tid] = rt[tid];
  if (tid == 0) {
    memset(&st, 0, sizeof(st));
    st.solve_ok = 1;
  }
  __syncthreads();
  if (tid == 0) cam_rotation(sm.x[0], sm.rot[0], true);
  __syncthreads();
  pose_pass<true, ROBUST>(sm, 0, n, xw, uv, K, kind, a, lin);
  if (tid == 0) {
    double gm = 0, xn = 0;
    for (int a = 0; a < 21; a++) sm.H[a] = lin[a];
    for (int a = 0; a < 6; a++) {
      sm.g[a] = lin[21 + a];
      gm = fmax(gm, fabs(sm.g[a]));
      xn += sm.x[0][a] * sm.x[0][a];
      sm.scale[a] = opt.jacobi_scaling ? 1.0 / (1.0 + sqrt(sm.H[uidx(a, a)])) : 1.0;
    }
    st.cost = st.initial_cost = 0.5 * lin[27];
    st.gmax = gm;
    st.x_norm = sqrt(xn);
    st.radius = opt.initial_trust_region_radius;
    st.decrease_factor = 2.0;
    st.termination = LORB_BA_NO_CONVERGENCE;
    if (gm <= opt.gradient_tolerance) {
      st.termination = LORB_BA_CONV_GRADIENT;
      st.done = 1;
    }
    if (opt.max_num_iterations <= 0) st.done = 1;
  }
  __syncthreads();
  while (!st.done) {
    const int cur = st.cur;
    if (tid == 0) {
      // scaled normal equations + clamped LM diagonal, 6x6 Cholesky
      double A[6][6], y[6];
      for (int a = 0; a < 6; a++)
        for (int b = 0; b < 6; b++)
          A[a][b] = sm.H[a <= b ? uidx(a, b) : uidx(b, a)] * sm.scale[a] * sm.scale[b];
      double Hs[6][6];
      for (int a = 0; a < 6; a++)
        for (int b = 0; b < 6; b++) Hs[a][b] = A[a][b];
      for (int a = 0; a < 6; a++) {
        A[a][a] += clamp_diag(Hs[a][a], opt.min_lm_diagonal, opt.max_lm_diagonal) / st.radius;
        y[a] = sm.g[a] * sm.scale[a];
      }
      bool ok = true;
      for (int j = 0; j < 6; j++) {
        double d = A[j][j];
        for (int k = 0; k < j; k++) d -= A[j][k] * A[j][k];
        if (!(d > 0.0)) {
          ok = false;
          d = 1.0;
        }
        d = sqrt(d);
        A[j][j] = d;
        for (int i = j + 1; i < 6; i++) {
          double s = A[i][j];
          for (int k = 0; k < j; k++) s -= A[i][k] * A[j][k];
          A[i][j] = s / d;
        }
      }
      for (int i = 0; i < 6; i++) {
        double s = y[i];
        for (int k = 0; k < i; k++) s -= A[i][k] * y[k];
        y[i] = s / A[i][i];
      }
      for (int i = 5; i >= 0; i--) {
        double s = y[i];
        for (int k = i + 1; k < 6; k++) s -= A[k][i] * y[k];
        y[i] = s / A[i][i];
      }
      // step = -y.  sum m.(r + m/2) with m = J step  ==  step.g_s + step^T H_s step / 2
      double sg = 0, shs = 0, step2 = 0, xc2 = 0;
      for (int a = 0; a < 6; a++) {
        sg += -y[a] * sm.g[a] * sm.scale[a];
        double hv = 0;
        for (int b = 0; b < 6; b++) hv += Hs[a][b] * (-y[b]);
        shs += -y[a] * hv;
        const double d = -y[a] * sm.scale[a];
        sm.x[cur ^ 1][a] = sm.x[cur][a] + d;
        step2 += d * d;
        xc2 += sm.x[cur ^ 1][a] * sm.x[cur ^ 1][a];
        if (!isfinite(y[a])) ok = false;
      }
      st.acc_model = sg + 0.5 * shs;
      st.acc_step2 = step2;
      st.acc_xcand2 = xc2;
      st.solve_ok = ok ? 1 : 0;
      cam_rotation(sm.x[cur ^ 1], sm.rot[cur ^ 1], true);
    }
    __syncthreads();
    pose_pass<false, ROBUST>(sm, cur ^ 1, n, xw, uv, K, kind, a, lin);
    int accepted = 0;
    if (tid == 0) {
      st.acc_cost2 = lin[27];
      accepted = lm_decide(&st, opt);
      if (accepted) st.cur ^= 1;
      st.pad = accepted;
    }
    __syncthreads();
    if (st.pad) {  // HandleSuccessfulStep: relinearise, gradient tolerance
      pose_pass<true, ROBUST>(sm, st.cur, n, xw, uv, K, kind, a, lin);
      if (tid == 0) {
        double gm = 0;
        for (int a = 0; a < 21; a++) sm.H[a] = lin[a];
        for (int a = 0; a < 6; a++) {
          sm.g[a] = lin[21 + a];
          gm = fmax(gm, fabs(sm.g[a]));
        }
        st.gmax = gm;
        st.check_gradient = 0;
        if (gm <= opt.gradient_tolerance) {
          st.termination = LORB_BA_CONV_GRADIENT;
          st.done = 1;
        }
      }
      __syncthreads();
    }
  }
  if (tid < 6) rt[tid] = sm.x[st.cur][tid];
  if (tid == 0) {
    sum->initial_cost = st.initial_cost;
    sum->final_cost = st.cost;
    sum->final_radius = st.radius;
    sum->final_gradient_max_norm = st.gmax;
    sum->iterations = st.iteration;
    sum->num_successful_steps = st.n_success;
    sum->num_unsuccessful_steps = st.n_fail;
    sum->termination = st.termination;
  }
}

}  // namespace lorb

using namespace lorb;

extern "C" int lorb_ba_pose_only(lorb_ctx* c, int n, const float* xw, const float* uv,
                                 const float* K, double* rt, const lorb_ba_options* opt,
                                 lorb_ba_summary* summary) {
  LORB_REQUIRE(c && K && rt && opt, "ctx / K / rt / options");
  LORB_REQUIRE(n >= 0 && (n == 0 || (xw && uv)), "observations");
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  const size_t b_xw = ((size_t)n * 12 + 255) & ~(size_t)255, b_uv = ((size_t)n * 8 + 255) & ~(size_t)255;
  const size_t up = b_xw + b_uv + 64, down = 64 + sizeof(lorb_ba_summary);
  LORB_TRY(pin_reserve(c, 0, up));
  LORB_TRY(pin_reserve(c, 1, down));
  LORB_TRY(dev_reserve(c, 0, up));
  LORB_TRY(dev_reserve(c, 2, down));
  uint8_t* h = c->h[0].as<uint8_t>();
  if (n) {
    memcpy(h, xw, (size_t)n * 12);
    memcpy(h + b_xw, uv, (size_t)n * 8);
  }
  memcpy(h + b_xw + b_uv, rt, 48);
  uint8_t* d = c->d[0].as<uint8_t>();
  uint8_t* dout = c->d[2].as<uint8_t>();
  LORB_CUDA_TRY(cudaMemcpyAsync(d, h, up, cudaMemcpyHostToDevice, c->stream));
  LORB_CUDA_TRY(cudaMemcpyAsync(dout, d + b_xw + b_uv, 48, cudaMemcpyDeviceToDevice, c->stream));
  Intr Kd;
  Kd.fu = (double)K[0];
  Kd.fv = (double)K[0];  // PoseCost projects v with fx (reference src/bundle_adjust.cpp:51)
  Kd.cx = (double)K[2];
  Kd.cy = (double)K[3];
  const lorb_ba_loss loss = c->ba_loss;
  LORB_LAUNCH(c, (loss.kind != LORB_LOSS_TRIVIAL ? pose_only_kernel<true> : pose_only_kernel<false>), 1,
              POSE_THREADS, 0, n, (const float*)d, (const float*)(d + b_xw), Kd, (double*)dout, *opt,
              (lorb_ba_summary*)(dout + 64), loss.kind, loss.scale);
  LORB_CUDA_TRY(cudaMemcpyAsync(c->h[1].p, dout, down, cudaMemcpyDeviceToHost, c->stream));
  LORB_CUDA_TRY(cudaStreamSynchronize(c->stream));
  memcpy(rt, c->h[1].p, 48);
  if (summary) memcpy(summary, c->h[1].as<uint8_t>() + 64, sizeof(lorb_ba_summary));
  return LORB_OK;
}
