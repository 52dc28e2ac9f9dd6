/*
 * tests/ba_rounds_ref.cpp -- TEST INFRASTRUCTURE ONLY: the outlier-round form of the pose-only BA
 * oracle (ORB-SLAM2's Optimizer::PoseOptimization on top of the Ceres restatement).
 *
 * A weighted observation is the residual sqrt(w) r, with the robust loss (ba_robust_ref.cpp) applied
 * to s = w |r|^2, as in Ceres with a scaled cost function and a LossFunction.  rounds_ref.py builds
 * the library from the robust oracle of robust_ref.py (oracle/ba_ref.cpp with ba_robust_ref.cpp
 * spliced in, both unchanged): it renames the robust linearize() / eval_cost() to robust_linearize /
 * robust_eval_cost, inserts the first part of this file after them and appends the second part.
 * Without weights the solver is exactly the robust oracle (and, with the trivial loss, the plain one).
 */
// ---- part 1: inside the oracle's anonymous namespace, after robust_linearize / robust_eval_cost

/* per-observation weights of the following solves, indexed like const_xw (NULL = unweighted) */
const float* g_w = nullptr;

/* 1/2 sum rho(w |r|^2) at (cams, pts) */
double eval_cost(const Problem& pb, const double* cams, const double* pts) {
  if (!g_w) return robust_eval_cost(pb, cams, pts);
  double c = 0;
  for (size_t i = 0; i < pb.res.size(); i++) {
    double r[2], rho[3];
    eval_residual(pb, cams, pts, (int)i, r, nullptr, nullptr);
    const double s = (r[0] * r[0] + r[1] * r[1]) * (double)g_w[pb.res[i].pt];
    loss_eval(g_loss, g_loss_a, s, rho);
    c += rho[0];
  }
  return 0.5 * c;
}

/* residuals and Jacobians scaled by sqrt(w), then corrected by the loss (Ceres' Corrector) */
double linearize(const Problem& pb, Lin& L) {
  if (!g_w) return robust_linearize(pb, L);
  plain_linearize(pb, L);
  double c = 0;
  for (size_t i = 0; i < pb.res.size(); i++) {
    double* r = &L.r[2 * i];
    const double sw = std::sqrt((double)g_w[pb.res[i].pt]);
    for (int k = 0; k < 2; k++) r[k] *= sw;
    for (int k = 0; k < 12; k++) L.Jc[12 * i + k] *= sw;
    for (int k = 0; k < 6; k++) L.Jp[6 * i + k] *= sw;
    double rho[3];
    loss_eval(g_loss, g_loss_a, r[0] * r[0] + r[1] * r[1], rho);
    const double w = std::sqrt(rho[1]);
    for (int k = 0; k < 2; k++) r[k] *= w;
    for (int k = 0; k < 12; k++) L.Jc[12 * i + k] *= w;
    for (int k = 0; k < 6; k++) L.Jp[6 * i + k] *= w;
    c += rho[0];
  }
  return 0.5 * c;
}

// ---- part 2: appended after the oracle's C entry points
extern "C" {

/* w |r|^2 of every observation at pose rt -> chi2[n]; inl[i] = chi2[i] <= th; returns the inlier count */
static int orc_classify(int n, const float* xw, const float* uv, const float* info, const float* K,
                        const double* rt, double th, unsigned char* inl, double* chi2) {
  Problem pb;
  pb.C = 1;
  pb.cams.assign(rt, rt + 6);
  pb.const_xw.assign(xw, xw + 3 * (size_t)n);
  pb.fx = K[0];
  pb.fy = K[1];
  pb.cx = K[2];
  pb.cy = K[3];
  pb.res.resize(n);
  int n_in = 0;
  for (int i = 0; i < n; i++) {
    Residual& R = pb.res[i];
    R.kind = RES_POSE_ONLY;
    R.cam = 0;
    R.pt = i;
    R.u = uv[2 * i];
    R.v = uv[2 * i + 1];
    double r[2];
    eval_residual(pb, pb.cams.data(), nullptr, i, r, nullptr, nullptr);
    double s = r[0] * r[0] + r[1] * r[1];
    if (info) s *= (double)info[i];
    chi2[i] = s;
    inl[i] = s <= th ? 1 : 0;
    n_in += inl[i];
  }
  return n_in;
}

/* One frame of lorb_ba_pose_rounds_batched (include/lorb_cuda.h), with the loss of orc_ba_set_loss. */
int orc_ba_pose_rounds(int n, const float* xw, const float* uv, const float* info, const float* K, double* rt,
                       int n_rounds, int robust_rounds, double th, const lorb_ba_options* opt,
                       unsigned char* inl, double* chi2, int* n_inliers, int* rounds_run,
                       lorb_ba_summary* sums) {
  const int loss = g_loss;
  const double x0[6] = {rt[0], rt[1], rt[2], rt[3], rt[4], rt[5]};
  std::vector<float> sxw, suv, sw;
  for (int i = 0; i < n; i++) inl[i] = 1;
  int n_in = n, ran = 0;
  for (; ran < n_rounds && n_in >= 3; ran++) {
    sxw.clear();
    suv.clear();
    sw.clear();
    for (int i = 0; i < n; i++) {
      if (!inl[i]) continue;
      sxw.insert(sxw.end(), xw + 3 * i, xw + 3 * i + 3);
      suv.insert(suv.end(), uv + 2 * i, uv + 2 * i + 2);
      if (info) sw.push_back(info[i]);
    }
    for (int k = 0; k < 6; k++) rt[k] = x0[k];
    g_loss = ran < robust_rounds ? loss : LORB_LOSS_TRIVIAL;
    g_w = info ? sw.data() : nullptr;
    orc_ba_pose_only(n_in, sxw.data(), suv.data(), K, rt, opt, &sums[ran]);
    g_w = nullptr;
    g_loss = loss;
    n_in = orc_classify(n, xw, uv, info, K, rt, th, inl, chi2);
  }
  if (ran == 0) n_in = orc_classify(n, xw, uv, info, K, rt, th, inl, chi2);
  for (int r = ran; r < n_rounds; r++) std::memset(&sums[r], 0, sizeof(lorb_ba_summary));
  *n_inliers = n_in;
  *rounds_run = ran;
  return 0;
}
}
