/*
 * tests/ba_local_rounds_ref.cpp -- TEST INFRASTRUCTURE ONLY: the outlier-round form of the local BA
 * oracle (ORB-SLAM2's Optimizer::LocalBundleAdjustment on top of the Ceres restatement).
 *
 * A weighted observation is the residual sqrt(w) r, with the robust loss (ba_robust_ref.cpp) applied
 * to s = w |r|^2.  local_rounds_ref.py builds the library from the robust oracle of robust_ref.py
 * (oracle/ba_ref.cpp with ba_robust_ref.cpp spliced in, both unchanged): it renames the robust
 * linearize() / eval_cost() to robust_linearize / robust_eval_cost, inserts the first part of this
 * file after them and appends the second part.  Without weights the solver is exactly the robust
 * oracle (and, with the trivial loss, the plain one).
 */
// ---- part 1: inside the oracle's anonymous namespace, after robust_linearize / robust_eval_cost

/* per-residual weights of the following solves, indexed like Problem::res (NULL = unweighted) */
const float* g_w = nullptr;

/* 1/2 sum rho(w |r|^2) at (cams, pts) */
double eval_cost(const Problem& pb, const double* cams, const double* pts) {
  if (!g_w) return robust_eval_cost(pb, cams, pts);
  double c = 0;
  for (size_t i = 0; i < pb.res.size(); i++) {
    double r[2], rho[3];
    eval_residual(pb, cams, pts, (int)i, r, nullptr, nullptr);
    const double s = (r[0] * r[0] + r[1] * r[1]) * (double)g_w[i];
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
    const double sw = std::sqrt((double)g_w[i]);
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
