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
#include <cmath>

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
// WEIGHTED: the residual of observation i is sqrt(w[i]) r (so s = w[i] |r|^2 enters the loss).
// MASKED: observations with mask[i] == 0 are left out.  mask is written by the classification pass of
// the same launch, so it is read through the coherent path (no __restrict__ / ld.global.nc).
template <bool LIN, bool ROBUST, bool WEIGHTED = false, bool MASKED = false>
__device__ __forceinline__ void pose_pass(PoseShared& sm, int b, int n, const float* __restrict__ xw,
                                          const float* __restrict__ uv, const float* __restrict__ w,
                                          const uint8_t* mask, const Intr& K, int kind, double a,
                                          double* out) {
  double acc[NRED];
#pragma unroll
  for (int i = 0; i < NRED; i++) acc[i] = 0.0;
  const double t[3] = {sm.x[b][3], sm.x[b][4], sm.x[b][5]};
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    if (MASKED && !mask[i]) continue;
    const double X[3] = {(double)xw[3 * i], (double)xw[3 * i + 1], (double)xw[3 * i + 2]};
    const double u = (double)uv[2 * i], v = (double)uv[2 * i + 1];
    if (LIN) {
      double r[2], Jc[12];
      obs_eval<true, false>(sm.rot[b], t, X, K, u, v, r, Jc, nullptr);
      if (WEIGHTED) {
        const double sw = sqrt((double)w[i]);
        r[0] *= sw;
        r[1] *= sw;
#pragma unroll
        for (int k = 0; k < 12; k++) Jc[k] *= sw;
      }
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
      double s = obs_cost(sm.rot[b], t, X, K, u, v);
      if (WEIGHTED) s *= (double)w[i];
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

// One Ceres solve (TrustRegionMinimizer + LevenbergMarquardtStrategy, fresh trust region and Jacobi
// scaling) of the pose from x0[6], run by the whole CTA.  On return the result is sm.x[sm.st.cur], its
// rotation is sm.rot[sm.st.cur] and sm.st holds the summary fields; the caller synchronises before it
// writes shared memory again.
// ROBUST = false: plain least squares (the reference); true: the loss (kind, a), LORB_LOSS_*.
// WEIGHTED / MASKED: see pose_pass.
template <bool ROBUST, bool WEIGHTED, bool MASKED>
__device__ __forceinline__ void pose_lm(PoseShared& sm, double* lin, int n, const float* __restrict__ xw,
                                        const float* __restrict__ uv, const float* __restrict__ w,
                                        const uint8_t* mask, const Intr& K, const double* __restrict__ x0,
                                        const lorb_ba_options& opt, int kind, double a) {
  const int tid = threadIdx.x;
  LMState& st = sm.st;
  if (tid < 6) sm.x[0][tid] = x0[tid];
  if (tid == 0) {
    memset(&st, 0, sizeof(st));
    st.solve_ok = 1;
  }
  __syncthreads();
  if (tid == 0) cam_rotation(sm.x[0], sm.rot[0], true);
  __syncthreads();
  pose_pass<true, ROBUST, WEIGHTED, MASKED>(sm, 0, n, xw, uv, w, mask, K, kind, a, lin);
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
    pose_pass<false, ROBUST, WEIGHTED, MASKED>(sm, cur ^ 1, n, xw, uv, w, mask, K, kind, a, lin);
    int accepted = 0;
    if (tid == 0) {
      st.acc_cost2 = lin[27];
      accepted = lm_decide(&st, opt);
      if (accepted) st.cur ^= 1;
      st.pad = accepted;
    }
    __syncthreads();
    if (st.pad) {  // HandleSuccessfulStep: relinearise, gradient tolerance
      pose_pass<true, ROBUST, WEIGHTED, MASKED>(sm, st.cur, n, xw, uv, w, mask, K, kind, a, lin);
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
}

__device__ __forceinline__ void store_summary(const LMState& st, lorb_ba_summary* sum) {
  sum->initial_cost = st.initial_cost;
  sum->final_cost = st.cost;
  sum->final_radius = st.radius;
  sum->final_gradient_max_norm = st.gmax;
  sum->iterations = st.iteration;
  sum->num_successful_steps = st.n_success;
  sum->num_unsuccessful_steps = st.n_fail;
  sum->termination = st.termination;
}

// ROBUST = false: plain least squares (the reference); true: the loss (kind, a), LORB_LOSS_*
template <bool ROBUST>
__global__ void __launch_bounds__(POSE_THREADS)
    pose_only_kernel(int n, const float* __restrict__ xw, const float* __restrict__ uv, Intr K,
                     double* __restrict__ rt, lorb_ba_options opt, lorb_ba_summary* __restrict__ sum, int kind,
                     double a) {
  __shared__ PoseShared sm;
  __shared__ double lin[NRED];
  pose_lm<ROBUST, false, false>(sm, lin, n, xw, uv, nullptr, nullptr, K, rt, opt, kind, a);
  if (threadIdx.x < 6) rt[threadIdx.x] = sm.x[sm.st.cur][threadIdx.x];
  if (threadIdx.x == 0) store_summary(sm.st, sum);
}

// chi^2 = w |r|^2 of every observation at pose sm.x[b] (rotation sm.rot[b]): inl[i] = chi^2 <= chi2,
// chi2_out[i] = chi^2; *n_in = number of inliers.
template <bool WEIGHTED>
__device__ __forceinline__ void pose_classify(PoseShared& sm, int b, int n, const float* __restrict__ xw,
                                              const float* __restrict__ uv, const float* __restrict__ w,
                                              const Intr& K, double chi2, uint8_t* inl,
                                              double* __restrict__ chi2_out, int* n_in) {
  if (threadIdx.x == 0) *n_in = 0;
  __syncthreads();
  const double t[3] = {sm.x[b][3], sm.x[b][4], sm.x[b][5]};
  int cnt = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double X[3] = {(double)xw[3 * i], (double)xw[3 * i + 1], (double)xw[3 * i + 2]};
    double s = obs_cost(sm.rot[b], t, X, K, (double)uv[2 * i], (double)uv[2 * i + 1]);
    if (WEIGHTED) s *= (double)w[i];
    const bool in = s <= chi2;
    inl[i] = in ? 1 : 0;
    chi2_out[i] = s;
    cnt += in;
  }
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(n_in, cnt);
  __syncthreads();
}

// ORB-SLAM2's PoseOptimization rounds (lorb_ba_pose_rounds_batched), one CTA per frame (blockIdx.x):
// every round is a full pose_lm solve from the input pose over the observations flagged inlier, then
// every observation of the frame is reclassified at the round's pose.  The flags live in inl (the
// output array).  Rounds [0, robust_rounds) use the loss (kind, a) unless it is trivial, later rounds
// plain least squares.  A frame's result does not depend on the other frames of the batch.
template <bool WEIGHTED>
__global__ void __launch_bounds__(POSE_THREADS)
    pose_rounds_kernel(const int* __restrict__ obs_off, const float* __restrict__ xw,
                       const float* __restrict__ uv, const float* __restrict__ w, Intr K,
                       const double* __restrict__ rt_in, double* __restrict__ rt_out, lorb_ba_options opt,
                       int n_rounds, int robust_rounds, double chi2, int kind, double a, uint8_t* inl,
                       double* __restrict__ chi2_out, int* __restrict__ n_inl, int* __restrict__ rounds_run,
                       lorb_ba_summary* __restrict__ sums) {
  __shared__ PoseShared sm;
  __shared__ double lin[NRED];
  __shared__ int n_in;
  const int f = blockIdx.x, tid = threadIdx.x;
  const int o0 = obs_off[f], n = obs_off[f + 1] - o0;
  xw += 3 * (size_t)o0;
  uv += 2 * (size_t)o0;
  if (WEIGHTED) w += o0;
  inl += o0;
  chi2_out += o0;
  const double* x0 = rt_in + 6 * (size_t)f;
  lorb_ba_summary* sum = sums + (size_t)f * n_rounds;
  for (int i = tid; i < n; i += blockDim.x) inl[i] = 1;
  if (tid == 0) n_in = n;
  __syncthreads();
  int ran = 0;
  for (; ran < n_rounds && n_in >= 3; ran++) {
    if (ran < robust_rounds && kind != LORB_LOSS_TRIVIAL)
      pose_lm<true, WEIGHTED, true>(sm, lin, n, xw, uv, w, inl, K, x0, opt, kind, a);
    else
      pose_lm<false, WEIGHTED, true>(sm, lin, n, xw, uv, w, inl, K, x0, opt, kind, a);
    if (tid == 0) store_summary(sm.st, sum + ran);
    pose_classify<WEIGHTED>(sm, sm.st.cur, n, xw, uv, w, K, chi2, inl, chi2_out, &n_in);
  }
  if (ran == 0) {  // fewer than 3 observations: the input pose and its classification
    if (tid < 6) sm.x[0][tid] = x0[tid];
    if (tid == 0) sm.st.cur = 0;
    __syncthreads();
    if (tid == 0) cam_rotation(sm.x[0], sm.rot[0], false);
    __syncthreads();
    pose_classify<WEIGHTED>(sm, 0, n, xw, uv, w, K, chi2, inl, chi2_out, &n_in);
  }
  if (tid < 6) rt_out[6 * (size_t)f + tid] = sm.x[sm.st.cur][tid];
  if (tid == 0) {
    n_inl[f] = n_in;
    rounds_run[f] = ran;
    for (int r = ran; r < n_rounds; r++) memset(sum + r, 0, sizeof(lorb_ba_summary));
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

extern "C" void lorb_ba_default_pose_rounds(lorb_ba_pose_rounds* r) {
  r->n_rounds = 4;
  r->robust_rounds = 3;
  r->chi2 = 5.991;
}

extern "C" int lorb_ba_pose_rounds_batched(lorb_ctx* c, int n_frames, const int* obs_off, const float* xw,
                                           const float* uv, const float* info, const float* K, double* rt,
                                           const lorb_ba_pose_rounds* rounds, const lorb_ba_options* opt,
                                           uint8_t* out_inlier, double* out_chi2, int* n_inliers,
                                           int* rounds_run, lorb_ba_summary* summaries) {
  LORB_REQUIRE(c && K && rounds && opt, "ctx / K / rounds / options");
  LORB_REQUIRE(rounds->n_rounds >= 1 && rounds->n_rounds <= 16, "rounds->n_rounds (1..16)");
  LORB_REQUIRE(rounds->robust_rounds >= 0 && rounds->robust_rounds <= rounds->n_rounds,
               "rounds->robust_rounds (0..n_rounds)");
  LORB_REQUIRE(std::isfinite(rounds->chi2) && rounds->chi2 > 0.0, "rounds->chi2 (finite, > 0)");
  LORB_REQUIRE(n_frames >= 0, "n_frames");
  if (n_frames == 0) return LORB_OK;
  LORB_REQUIRE(obs_off && rt && n_inliers, "obs_off / rt / n_inliers");
  LORB_REQUIRE(obs_off[0] == 0, "obs_off[0] != 0");
  for (int f = 0; f < n_frames; f++) LORB_REQUIRE(obs_off[f + 1] >= obs_off[f], "obs_off not non-decreasing");
  const int O = obs_off[n_frames];
  LORB_REQUIRE(O == 0 || (xw && uv && out_inlier), "xw / uv / out_inlier");
  if (info)
    for (int i = 0; i < O; i++) LORB_REQUIRE(std::isfinite(info[i]) && info[i] > 0.0f, "info (finite, > 0)");
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  const int F = n_frames, R = rounds->n_rounds;
  auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
  // upload: obs_off | xw | uv | info | rt ;  download: rt | n_inl | rounds_run | summaries | inlier | chi2
  const size_t u_off = 0, u_xw = u_off + al((size_t)(F + 1) * 4), u_uv = u_xw + al((size_t)O * 12),
               u_w = u_uv + al((size_t)O * 8), u_rt = u_w + (info ? al((size_t)O * 4) : 0), up = u_rt + (size_t)F * 48;
  const size_t d_rt = 0, d_n = al((size_t)F * 48), d_run = d_n + al((size_t)F * 4), d_sum = d_run + al((size_t)F * 4),
               d_inl = d_sum + al((size_t)F * R * sizeof(lorb_ba_summary)), d_chi = d_inl + al((size_t)O),
               down = d_chi + (size_t)O * 8;
  LORB_TRY(pin_reserve(c, 0, up));
  LORB_TRY(pin_reserve(c, 1, down));
  LORB_TRY(dev_reserve(c, 0, up));
  LORB_TRY(dev_reserve(c, 2, down));
  uint8_t* h = c->h[0].as<uint8_t>();
  memcpy(h + u_off, obs_off, (size_t)(F + 1) * 4);
  if (O) {
    memcpy(h + u_xw, xw, (size_t)O * 12);
    memcpy(h + u_uv, uv, (size_t)O * 8);
    if (info) memcpy(h + u_w, info, (size_t)O * 4);
  }
  memcpy(h + u_rt, rt, (size_t)F * 48);
  uint8_t* d = c->d[0].as<uint8_t>();
  uint8_t* dout = c->d[2].as<uint8_t>();
  LORB_CUDA_TRY(cudaMemcpyAsync(d, h, up, cudaMemcpyHostToDevice, c->stream));
  Intr Kd;
  Kd.fu = (double)K[0];
  Kd.fv = (double)K[0];  // PoseCost projects v with fx (reference src/bundle_adjust.cpp:51)
  Kd.cx = (double)K[2];
  Kd.cy = (double)K[3];
  const lorb_ba_loss loss = c->ba_loss;
  LORB_LAUNCH(c, (info ? pose_rounds_kernel<true> : pose_rounds_kernel<false>), F, POSE_THREADS, 0,
              (const int*)(d + u_off), (const float*)(d + u_xw), (const float*)(d + u_uv),
              (const float*)(info ? d + u_w : nullptr), Kd, (const double*)(d + u_rt), (double*)(dout + d_rt),
              *opt, R, rounds->robust_rounds, rounds->chi2, loss.kind, loss.scale, dout + d_inl,
              (double*)(dout + d_chi), (int*)(dout + d_n), (int*)(dout + d_run),
              (lorb_ba_summary*)(dout + d_sum));
  LORB_CUDA_TRY(cudaMemcpyAsync(c->h[1].p, dout, out_chi2 ? down : d_chi, cudaMemcpyDeviceToHost, c->stream));
  LORB_CUDA_TRY(cudaStreamSynchronize(c->stream));
  const uint8_t* ho = c->h[1].as<uint8_t>();
  memcpy(rt, ho + d_rt, (size_t)F * 48);
  memcpy(n_inliers, ho + d_n, (size_t)F * 4);
  if (rounds_run) memcpy(rounds_run, ho + d_run, (size_t)F * 4);
  if (summaries) memcpy(summaries, ho + d_sum, (size_t)F * R * sizeof(lorb_ba_summary));
  if (O) memcpy(out_inlier, ho + d_inl, (size_t)O);
  if (out_chi2 && O) memcpy(out_chi2, ho + d_chi, (size_t)O * 8);
  return LORB_OK;
}
