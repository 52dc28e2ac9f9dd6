/*
 * tests/ba_oracle_ext.cpp -- TEST INFRASTRUCTURE ONLY: the BA oracle (oracle/ba_ref.cpp, unchanged)
 * extended with robust losses, per-residual weights and ORB-SLAM2's outlier rounds, as the reference
 * of lorb_ba_set_loss, lorb_ba_pose_rounds_batched and lorb_ba_local_rounds_batched.
 *
 * Ceres applies a LossFunction through its Corrector, per residual block, at the point of
 * linearisation: for losses with rho'' <= 0 (Huber, soft-L1, Cauchy) the curvature term vanishes and
 * the correction is r~ = sqrt(rho'(s)) r, J~ = sqrt(rho'(s)) J with s = |r|^2, while the cost becomes
 * 1/2 sum rho(s).  A weighted observation is the residual sqrt(w) r, with the loss applied to
 * s = w |r|^2, as in Ceres with a scaled cost function and a LossFunction.  The gradient, the
 * Gauss-Newton matrix, the Jacobi scaling and the model decrease of the trust-region loop all follow
 * from the corrected r~ and J~.  So the extended solver is the oracle's own with exactly two functions
 * replaced: linearize() and eval_cost().  oracle_ext.py builds it: it renames the oracle's two
 * definitions to plain_linearize / plain_eval_cost, inserts the first part of this file after them
 * (inside the oracle's namespace) and appends the second part (the C entry points).  Without weights
 * and with the trivial loss the solver is exactly the oracle.
 */
// ---- part 1: inside the oracle's anonymous namespace, after plain_linearize / plain_eval_cost

/* robust loss of the following solves (orc_ba_set_loss); read-only while a solve runs */
int g_loss = LORB_LOSS_TRIVIAL;
double g_loss_a = 1.0;

/* per-residual weights of the following solves, indexed like Problem::res, whose residual i is
 * observation i in orc_ba_pose_only and in-window / fixed observation i / i - O in orc_ba_local
 * (NULL = unweighted) */
const float* g_w = nullptr;

/* rho(s), rho'(s), rho''(s) with scale a (ceres::HuberLoss, SoftLOneLoss, CauchyLoss; b = a^2,
 * c = 1/b).  rho of soft-L1 / Cauchy avoids the cancellation of 2b (sqrt(1 + sc) - 1) and
 * log(1 + sc) when sc << 1, as the library does. */
void loss_eval(int kind, double a, double s, double rho[3]) {
  const double b = a * a, c = 1.0 / b;
  if (kind == LORB_LOSS_HUBER) {
    if (s > b) {
      const double r = std::sqrt(s);
      rho[0] = 2.0 * a * r - b;
      rho[1] = std::fmax(std::numeric_limits<double>::min(), a / r);
      rho[2] = -rho[1] / (2.0 * s);
    } else {
      rho[0] = s;
      rho[1] = 1.0;
      rho[2] = 0.0;
    }
  } else if (kind == LORB_LOSS_SOFTLONE) {
    const double sum = 1.0 + s * c, tmp = std::sqrt(sum);
    rho[0] = 2.0 * s / (tmp + 1.0); /* = 2b (tmp - 1) */
    rho[1] = std::fmax(std::numeric_limits<double>::min(), 1.0 / tmp);
    rho[2] = -(c * rho[1]) / (2.0 * sum);
  } else if (kind == LORB_LOSS_CAUCHY) {
    const double sum = 1.0 + s * c, inv = 1.0 / sum;
    rho[0] = b * std::log1p(s * c);
    rho[1] = std::fmax(std::numeric_limits<double>::min(), inv);
    rho[2] = -c * (inv * inv);
  } else {
    rho[0] = s;
    rho[1] = 1.0;
    rho[2] = 0.0;
  }
}

/* 1/2 sum rho(w |r|^2) at (cams, pts) */
double eval_cost(const Problem& pb, const double* cams, const double* pts) {
  if (g_loss == LORB_LOSS_TRIVIAL && !g_w) return plain_eval_cost(pb, cams, pts);
  double c = 0;
  for (size_t i = 0; i < pb.res.size(); i++) {
    double r[2], rho[3];
    eval_residual(pb, cams, pts, (int)i, r, nullptr, nullptr);
    double s = r[0] * r[0] + r[1] * r[1];
    if (g_w) s *= (double)g_w[i];
    loss_eval(g_loss, g_loss_a, s, rho);
    c += rho[0];
  }
  return 0.5 * c;
}

/* residuals and Jacobians scaled by sqrt(w), then corrected by the loss (Ceres' Corrector) */
double linearize(const Problem& pb, Lin& L) {
  if (g_loss == LORB_LOSS_TRIVIAL && !g_w) return plain_linearize(pb, L);
  plain_linearize(pb, L);
  double c = 0;
  for (size_t i = 0; i < pb.res.size(); i++) {
    double* r = &L.r[2 * i];
    if (g_w) {
      const double sw = std::sqrt((double)g_w[i]);
      for (int k = 0; k < 2; k++) r[k] *= sw;
      for (int k = 0; k < 12; k++) L.Jc[12 * i + k] *= sw;
      for (int k = 0; k < 6; k++) L.Jp[6 * i + k] *= sw;
    }
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

/* w |r|^2 and the depth of residual i at (cams, pts) */
void chi2_depth(const Problem& pb, const double* cams, const double* pts, int i, double w, double* chi2,
                double* depth) {
  const Residual& R = pb.res[i];
  double r[2];
  eval_residual(pb, cams, pts, i, r, nullptr, nullptr);
  *chi2 = w * (r[0] * r[0] + r[1] * r[1]);
  double rv[3], tv[3], X[3], q[3];
  for (int k = 0; k < 3; k++) {
    rv[k] = R.kind == RES_MP_FIXED ? (double)R.frt[k] : cams[6 * R.cam + k];
    tv[k] = R.kind == RES_MP_FIXED ? (double)R.frt[3 + k] : cams[6 * R.cam + 3 + k];
    X[k] = pts[3 * R.pt + k];
  }
  AngleAxisRotatePoint(rv, X, q);
  *depth = q[2] + tv[2];
}

// ---- part 2: appended after the oracle's C entry points
extern "C" {

/* Robust loss of the following orc_ba_* solves and costs of this library (0 = trivial). */
void orc_ba_set_loss(int kind, double scale) {
  g_loss = kind;
  g_loss_a = scale;
}

/* rho, rho', rho'' of one residual block with squared norm s. */
void orc_ba_loss_eval(int kind, double scale, double s, double* rho) { loss_eval(kind, scale, s, rho); }

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

/* One window of lorb_ba_local_rounds_batched (include/lorb_cuda.h), with the loss of orc_ba_set_loss.
 * Each round hands orc_ba_local the inlier subset (every camera and point stays a parameter) and
 * continues from the previous round's result; after it every observation is classified. */
int orc_ba_local_rounds(int C, double* cams, int P, double* pts, int O, const int* obs_cam, const int* obs_pt,
                        const float* obs_uv, const float* obs_w, int F, const int* fix_pt, const float* fix_uv,
                        const float* fix_rt, const float* fix_w, const float* K, int n_rounds, int robust_rounds,
                        double th, int depth_check, const lorb_ba_options* opt /* [n_rounds] */, unsigned char* obs_in,
                        double* obs_chi2, unsigned char* fix_in, double* fix_chi2, int* n_inliers,
                        lorb_ba_summary* sums) {
  const int loss = g_loss;
  for (int i = 0; i < O; i++) obs_in[i] = 1;
  for (int i = 0; i < F; i++) fix_in[i] = 1;
  int n_in = O + F;
  for (int rd = 0; rd < n_rounds; rd++) {
    std::vector<int> oc, op, fp;
    std::vector<float> ouv, fuv, frt, w;
    for (int i = 0; i < O; i++) {
      if (!obs_in[i]) continue;
      oc.push_back(obs_cam[i]);
      op.push_back(obs_pt[i]);
      ouv.insert(ouv.end(), obs_uv + 2 * i, obs_uv + 2 * i + 2);
      w.push_back(obs_w ? obs_w[i] : 1.0f);
    }
    for (int i = 0; i < F; i++) {
      if (!fix_in[i]) continue;
      fp.push_back(fix_pt[i]);
      fuv.insert(fuv.end(), fix_uv + 2 * i, fix_uv + 2 * i + 2);
      frt.insert(frt.end(), fix_rt + 6 * i, fix_rt + 6 * i + 6);
      w.push_back(fix_w ? fix_w[i] : 1.0f);
    }
    g_loss = rd < robust_rounds ? loss : LORB_LOSS_TRIVIAL;
    g_w = (obs_w || fix_w) ? w.data() : nullptr;
    const int rc = orc_ba_local(C, cams, P, pts, (int)oc.size(), oc.data(), op.data(), ouv.data(), (int)fp.size(),
                                fp.data(), fuv.data(), frt.data(), K, &opt[rd], &sums[rd]);
    g_w = nullptr;
    g_loss = loss;
    if (rc != 0) return rc;
    /* classification of every observation at the round's result */
    Problem pb;
    pb.C = C;
    pb.P = P;
    pb.fx = K[0];
    pb.fy = K[1];
    pb.cx = K[2];
    pb.cy = K[3];
    pb.res.resize((size_t)O + F);
    for (int i = 0; i < O; i++) {
      Residual& R = pb.res[i];
      R.kind = RES_POSE_MP;
      R.cam = obs_cam[i];
      R.pt = obs_pt[i];
      R.u = obs_uv[2 * i];
      R.v = obs_uv[2 * i + 1];
    }
    for (int i = 0; i < F; i++) {
      Residual& R = pb.res[(size_t)O + i];
      R.kind = RES_MP_FIXED;
      R.cam = -1;
      R.pt = fix_pt[i];
      R.u = fix_uv[2 * i];
      R.v = fix_uv[2 * i + 1];
      for (int k = 0; k < 6; k++) R.frt[k] = fix_rt[6 * i + k];
    }
    n_in = 0;
    for (int i = 0; i < O + F; i++) {
      const bool fixed = i >= O;
      const float* wv = fixed ? fix_w : obs_w;
      const int j = fixed ? i - O : i;
      double c2, z;
      chi2_depth(pb, cams, pts, i, wv ? (double)wv[j] : 1.0, &c2, &z);
      const unsigned char in = c2 <= th && (!depth_check || z > 0.0) ? 1 : 0;
      (fixed ? fix_in : obs_in)[j] = in;
      (fixed ? fix_chi2 : obs_chi2)[j] = c2;
      n_in += in;
    }
  }
  *n_inliers = n_in;
  return 0;
}
}
