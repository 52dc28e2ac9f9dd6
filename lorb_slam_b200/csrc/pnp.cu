// pnp.cu — batched P3P RANSAC on sm_100a (lorb_pnp_ransac_batched; beyond the reference: the pose half of
// VisualOdometry::EstimatePosePnP and of ORB-SLAM2's relocalisation step).
//
// Two launches per call:
//   pnp_score_kernel     grid (hypothesis chunks x problems).  One lane draws and solves one hypothesis
//                        (pnp_math.cuh), keeps its pose in registers and counts its inliers over the problem's
//                        correspondences, which the CTA stages through shared memory in tiles.  The problem's
//                        argmax is one 64-bit atomicMax per warp on ((count + 1) << 32) | (0xFFFFFFFF - h):
//                        most inliers, then lowest h, whatever the schedule.
//   pnp_finalize_kernel  one CTA per problem: decodes h, recomputes that hypothesis with the same device
//                        function, converts R to angle-axis and classifies every correspondence.
#include <cmath>

#include "common.cuh"
#include "pnp_math.cuh"

namespace lorb {
namespace pnp {

constexpr int SCORE_THREADS = 128;  // hypotheses per CTA
constexpr int TILE = 256;           // correspondences per shared-memory tile
constexpr int FIN_THREADS = 256;

// chi^2 = w |r|^2 of one correspondence at P; inlier iff in front of the camera and chi^2 <= chi2.
// Behind the camera (z <= 0) chi^2 is reported as +inf.
__device__ __forceinline__ bool classify(const Pose& P, const F X[3], F u, F v, F w, const Cam& K, double chi2,
                                         double& c2) {
  F e;
  const bool front = reproj2(P, X, u, v, K, e);
  const F s = w * e;
  c2 = front ? s.v : __longlong_as_double(0x7FF0000000000000ll);
  return front && s.v <= chi2;
}

__global__ void __launch_bounds__(SCORE_THREADS)
    pnp_score_kernel(const int* __restrict__ corr_off, const uint64_t* __restrict__ seeds,
                     const float* __restrict__ xw, const float* __restrict__ uv, const float* __restrict__ w,
                     Cam K, int H, int chunks, double chi2, unsigned long long* __restrict__ keys) {
  __shared__ double sx[TILE], sy[TILE], sz[TILE], su[TILE], sv[TILE], sw[TILE];
  const int b = blockIdx.x / chunks, chunk = blockIdx.x - b * chunks;
  const int o0 = corr_off[b], n = corr_off[b + 1] - o0;
  if (n < 4) return;
  const int h = chunk * SCORE_THREADS + threadIdx.x;
  Pose P;
  const bool valid = h < H && hypothesis(seeds[b], (uint32_t)h, n, xw + 3 * (size_t)o0, uv + 2 * (size_t)o0, K, P);
  if (!__syncthreads_or(valid)) return;
  int cnt = 0;
  for (int base = 0; base < n; base += TILE) {
    const int m = min(TILE, n - base);
    for (int i = threadIdx.x; i < m; i += SCORE_THREADS) {
      const size_t j = (size_t)o0 + base + i;
      sx[i] = xw[3 * j];
      sy[i] = xw[3 * j + 1];
      sz[i] = xw[3 * j + 2];
      su[i] = uv[2 * j];
      sv[i] = uv[2 * j + 1];
      sw[i] = w ? (double)w[j] : 1.0;
    }
    __syncthreads();
    if (valid) {
#pragma unroll 4
      for (int i = 0; i < m; i++) {
        const F X[3] = {F{sx[i]}, F{sy[i]}, F{sz[i]}};
        F e;
        const bool front = reproj2(P, X, F{su[i]}, F{sv[i]}, K, e);
        cnt += (front && (F{sw[i]} * e).v <= chi2) ? 1 : 0;
      }
    }
    __syncthreads();
  }
  unsigned long long key =
      valid ? ((unsigned long long)(cnt + 1) << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)h) : 0ull;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
    key = other > key ? other : key;
  }
  if ((threadIdx.x & 31) == 0 && key) atomicMax(keys + b, key);
}

// Angle-axis of a rotation matrix: quaternion by Shepperd's method (the largest of trace and diagonal),
// then Ceres' QuaternionToAngleAxis, which is accurate at theta near 0 and near pi.
__device__ __forceinline__ void rotation_to_angle_axis(const double R[9], double aa[3]) {
  const double tr = R[0] + R[4] + R[8];
  double q[4];
  if (tr >= R[0] && tr >= R[4] && tr >= R[8]) {
    q[0] = 0.5 * sqrt(1.0 + tr);
    const double f = 0.25 / q[0];
    q[1] = (R[7] - R[5]) * f;
    q[2] = (R[2] - R[6]) * f;
    q[3] = (R[3] - R[1]) * f;
  } else if (R[0] >= R[4] && R[0] >= R[8]) {
    q[1] = 0.5 * sqrt(1.0 + R[0] - R[4] - R[8]);
    const double f = 0.25 / q[1];
    q[0] = (R[7] - R[5]) * f;
    q[2] = (R[1] + R[3]) * f;
    q[3] = (R[2] + R[6]) * f;
  } else if (R[4] >= R[8]) {
    q[2] = 0.5 * sqrt(1.0 - R[0] + R[4] - R[8]);
    const double f = 0.25 / q[2];
    q[0] = (R[2] - R[6]) * f;
    q[1] = (R[1] + R[3]) * f;
    q[3] = (R[5] + R[7]) * f;
  } else {
    q[3] = 0.5 * sqrt(1.0 - R[0] - R[4] + R[8]);
    const double f = 0.25 / q[3];
    q[0] = (R[3] - R[1]) * f;
    q[1] = (R[2] + R[6]) * f;
    q[2] = (R[5] + R[7]) * f;
  }
  const double qn = 1.0 / sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  for (int i = 0; i < 4; i++) q[i] *= qn;
  const double s2 = q[1] * q[1] + q[2] * q[2] + q[3] * q[3];
  double k = 2.0;
  if (s2 > 0.0) {
    const double s = sqrt(s2), c = q[0];
    k = 2.0 * (c < 0.0 ? atan2(-s, -c) : atan2(s, c)) / s;
  }
  for (int i = 0; i < 3; i++) aa[i] = q[i + 1] * k;
}

__global__ void __launch_bounds__(FIN_THREADS)
    pnp_finalize_kernel(const int* __restrict__ corr_off, const uint64_t* __restrict__ seeds,
                        const float* __restrict__ xw, const float* __restrict__ uv, const float* __restrict__ w,
                        Cam K, double chi2, const unsigned long long* __restrict__ keys, double* __restrict__ rt,
                        int* __restrict__ best_hyp, int* __restrict__ n_inliers, uint8_t* __restrict__ inl,
                        double* __restrict__ chi2_out) {
  __shared__ Pose sP;
  __shared__ int s_ok, s_cnt;
  const int b = blockIdx.x, tid = threadIdx.x;
  const int o0 = corr_off[b], n = corr_off[b + 1] - o0;
  xw += 3 * (size_t)o0;
  uv += 2 * (size_t)o0;
  if (tid == 0) {
    const unsigned long long key = keys[b];
    const uint32_t h = 0xFFFFFFFFu - (uint32_t)key;
    Pose P;
    // a non-zero key was written by a valid hypothesis, which the same function reproduces
    const bool ok = key != 0ull && hypothesis(seeds[b], h, n, xw, uv, K, P);
    double R[9], aa[3] = {0.0, 0.0, 0.0};
    if (ok) {
      for (int i = 0; i < 9; i++) R[i] = P.R[i].v;
      rotation_to_angle_axis(R, aa);
      sP = P;
    }
    for (int i = 0; i < 3; i++) {
      rt[6 * (size_t)b + i] = aa[i];
      rt[6 * (size_t)b + 3 + i] = ok ? P.t[i].v : 0.0;
    }
    best_hyp[b] = ok ? (int)h : -1;
    s_ok = ok;
    s_cnt = 0;
  }
  __syncthreads();
  const bool ok = s_ok;
  const Pose P = sP;
  int cnt = 0;
  for (int i = tid; i < n; i += FIN_THREADS) {
    double c2 = __longlong_as_double(0x7FF0000000000000ll);
    bool in = false;
    if (ok) {
      const F X[3] = {F{(double)xw[3 * i]}, F{(double)xw[3 * i + 1]}, F{(double)xw[3 * i + 2]}};
      in = classify(P, X, F{(double)uv[2 * i]}, F{(double)uv[2 * i + 1]}, F{w ? (double)w[o0 + i] : 1.0}, K, chi2,
                    c2);
    }
    inl[o0 + i] = in ? 1 : 0;
    if (chi2_out) chi2_out[o0 + i] = c2;
    cnt += in;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if ((tid & 31) == 0) atomicAdd(&s_cnt, cnt);
  __syncthreads();
  if (tid == 0) n_inliers[b] = s_cnt;
}

}  // namespace pnp
}  // namespace lorb

using namespace lorb;

extern "C" void lorb_default_pnp_ransac(lorb_pnp_ransac* p) {
  p->n_hypotheses = 300;
  p->reserved = 0;
  p->chi2 = 5.991;
}

extern "C" int lorb_pnp_ransac_batched(lorb_ctx* c, int n_problems, const int* corr_off, const float* xw,
                                       const float* uv, const float* info, const float* K, const uint64_t* seeds,
                                       const lorb_pnp_ransac* params, double* out_rt, int* best_hyp,
                                       int* n_inliers, uint8_t* out_inlier, double* out_chi2) {
  LORB_REQUIRE(c && K && params, "ctx / K / params");
  LORB_REQUIRE(params->n_hypotheses >= 1 && params->n_hypotheses <= 65536, "params->n_hypotheses (1..65536)");
  LORB_REQUIRE(std::isfinite(params->chi2) && params->chi2 > 0.0, "params->chi2 (finite, > 0)");
  LORB_REQUIRE(std::isfinite(K[0]) && K[0] > 0.0f && std::isfinite(K[1]) && K[1] > 0.0f, "fx / fy (finite, > 0)");
  LORB_REQUIRE(n_problems >= 0, "n_problems");
  if (n_problems == 0) return LORB_OK;
  LORB_REQUIRE(corr_off && out_rt && best_hyp && n_inliers, "corr_off / out_rt / best_hyp / n_inliers");
  LORB_REQUIRE(corr_off[0] == 0, "corr_off[0] != 0");
  for (int b = 0; b < n_problems; b++) LORB_REQUIRE(corr_off[b + 1] >= corr_off[b], "corr_off not non-decreasing");
  const int O = corr_off[n_problems];
  LORB_REQUIRE(O == 0 || (xw && uv && out_inlier), "xw / uv / out_inlier");
  if (info)
    for (int i = 0; i < O; i++) LORB_REQUIRE(std::isfinite(info[i]) && info[i] > 0.0f, "info (finite, > 0)");
  const int H = params->n_hypotheses, chunks = (H + pnp::SCORE_THREADS - 1) / pnp::SCORE_THREADS;
  LORB_REQUIRE((long long)n_problems * chunks <= 0x7FFFFFFFll, "n_problems x hypothesis chunks exceeds the grid");
  LORB_CUDA_TRY(cudaSetDevice(c->device));
  const size_t P = (size_t)n_problems;
  auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
  // upload: keys (zeros) | corr_off | seeds | xw | uv | info ;  download: rt | best_hyp | n_inliers | inlier | chi2
  const size_t u_key = 0, u_off = al(P * 8), u_seed = u_off + al((P + 1) * 4), u_xw = u_seed + al(P * 8),
               u_uv = u_xw + al((size_t)O * 12), u_w = u_uv + al((size_t)O * 8),
               up = u_w + (info ? (size_t)O * 4 : 0);
  const size_t d_rt = 0, d_best = al(P * 48), d_n = d_best + al(P * 4), d_inl = d_n + al(P * 4),
               d_chi = d_inl + al((size_t)O), down = d_chi + (size_t)O * 8;
  LORB_TRY(pin_reserve(c, 0, up));
  LORB_TRY(pin_reserve(c, 1, down));
  LORB_TRY(dev_reserve(c, 0, up));
  LORB_TRY(dev_reserve(c, 2, down));
  uint8_t* h = c->h[0].as<uint8_t>();
  memset(h + u_key, 0, P * 8);
  memcpy(h + u_off, corr_off, (P + 1) * 4);
  uint64_t* hs = reinterpret_cast<uint64_t*>(h + u_seed);
  for (size_t b = 0; b < P; b++) hs[b] = seeds ? seeds[b] : (uint64_t)b;
  if (O) {
    memcpy(h + u_xw, xw, (size_t)O * 12);
    memcpy(h + u_uv, uv, (size_t)O * 8);
    if (info) memcpy(h + u_w, info, (size_t)O * 4);
  }
  uint8_t* d = c->d[0].as<uint8_t>();
  uint8_t* dout = c->d[2].as<uint8_t>();
  LORB_CUDA_TRY(cudaMemcpyAsync(d, h, up, cudaMemcpyHostToDevice, c->stream));
  const pnp::Cam Kd = {(double)K[0], (double)K[1], (double)K[2], (double)K[3]};
  const float* dw = info ? (const float*)(d + u_w) : nullptr;
  LORB_LAUNCH(c, pnp::pnp_score_kernel, (unsigned)(P * chunks), pnp::SCORE_THREADS, 0, (const int*)(d + u_off),
              (const uint64_t*)(d + u_seed), (const float*)(d + u_xw), (const float*)(d + u_uv), dw, Kd, H, chunks,
              params->chi2, (unsigned long long*)(d + u_key));
  LORB_LAUNCH(c, pnp::pnp_finalize_kernel, (unsigned)P, pnp::FIN_THREADS, 0, (const int*)(d + u_off),
              (const uint64_t*)(d + u_seed), (const float*)(d + u_xw), (const float*)(d + u_uv), dw, Kd,
              params->chi2, (const unsigned long long*)(d + u_key), (double*)(dout + d_rt), (int*)(dout + d_best),
              (int*)(dout + d_n), dout + d_inl, out_chi2 ? (double*)(dout + d_chi) : nullptr);
  LORB_CUDA_TRY(cudaMemcpyAsync(c->h[1].p, dout, out_chi2 ? down : d_chi, cudaMemcpyDeviceToHost, c->stream));
  LORB_CUDA_TRY(cudaStreamSynchronize(c->stream));
  const uint8_t* ho = c->h[1].as<uint8_t>();
  memcpy(out_rt, ho + d_rt, P * 48);
  memcpy(best_hyp, ho + d_best, P * 4);
  memcpy(n_inliers, ho + d_n, P * 4);
  if (O) memcpy(out_inlier, ho + d_inl, (size_t)O);
  if (out_chi2 && O) memcpy(out_chi2, ho + d_chi, (size_t)O * 8);
  return LORB_OK;
}
