/*
 * tests/ba_robust_ref.cpp -- TEST INFRASTRUCTURE ONLY: the robust-loss form of the BA oracle.
 *
 * Ceres applies a LossFunction through its Corrector, per residual block, at the point of
 * linearisation: for losses with rho'' <= 0 (Huber, soft-L1, Cauchy) the curvature term vanishes and
 * the correction is r~ = sqrt(rho'(s)) r, J~ = sqrt(rho'(s)) J with s = |r|^2, while the cost becomes
 * 1/2 sum rho(s).  The gradient, the Gauss-Newton matrix, the Jacobi scaling and the model decrease
 * of the trust-region loop all follow from the corrected r~ and J~.  So the robust solver is the
 * oracle's own (oracle/ba_ref.cpp, unchanged) with exactly two functions replaced: linearize() and
 * eval_cost().  robust_ref.py builds it: it renames the oracle's two definitions to plain_linearize /
 * plain_eval_cost, inserts the first part of this file in their place (inside the oracle's namespace)
 * and appends the second part (the C entry points).
 */
// ---- part 1: inside the oracle's anonymous namespace, after plain_linearize / plain_eval_cost

/* robust loss of the following solves (orc_ba_set_loss); read-only while a solve runs */
int g_loss = LORB_LOSS_TRIVIAL;
double g_loss_a = 1.0;

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

double eval_cost(const Problem& pb, const double* cams, const double* pts) {
  if (g_loss == LORB_LOSS_TRIVIAL) return plain_eval_cost(pb, cams, pts);
  double c = 0;
  for (size_t i = 0; i < pb.res.size(); i++) {
    double r[2], rho[3];
    eval_residual(pb, cams, pts, (int)i, r, nullptr, nullptr);
    loss_eval(g_loss, g_loss_a, r[0] * r[0] + r[1] * r[1], rho);
    c += rho[0];
  }
  return 0.5 * c;
}

double linearize(const Problem& pb, Lin& L) {
  const double plain = plain_linearize(pb, L);
  if (g_loss == LORB_LOSS_TRIVIAL) return plain;
  double c = 0;
  for (size_t i = 0; i < pb.res.size(); i++) {
    double* r = &L.r[2 * i];
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

/* Robust loss of the following orc_ba_* solves and costs of this library (0 = trivial). */
void orc_ba_set_loss(int kind, double scale) {
  g_loss = kind;
  g_loss_a = scale;
}

/* rho, rho', rho'' of one residual block with squared norm s. */
void orc_ba_loss_eval(int kind, double scale, double s, double* rho) { loss_eval(kind, scale, s, rho); }
}
