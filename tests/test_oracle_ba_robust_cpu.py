"""CPU: robust losses (Huber, soft-L1, Cauchy) of the BA oracle (tests/oracle_ext.py).  The loss functions are checked
against finite differences, the trivial loss against the default call bit for bit, and the minimum
the oracle finds under each loss against scipy.optimize.least_squares, which implements the same
three losses independently."""
import numpy as np
import pytest

import oracle_ext as rr
import robust_cases as rc
from oracle import ref

TIGHT = dict(max_num_iterations=200, function_tolerance=1e-15, gradient_tolerance=1e-14,
             parameter_tolerance=1e-14)


@pytest.mark.parametrize("name", sorted(rc.LOSSES))
def test_loss_derivatives_match_finite_differences(name):
    kind, a = rc.LOSSES[name], 1.7
    b = a * a
    # both sides of the Huber knee (s = b), far out, and near zero
    for s in [1e-3, 0.5 * b, 0.9 * b, 1.1 * b, 3.0 * b, 400.0]:
        rho, rho1, rho2 = rr.loss_eval(kind, a, s)
        h = 1e-6 * s
        fp, fm = rr.loss_eval(kind, a, s + h), rr.loss_eval(kind, a, s - h)
        assert abs((fp[0] - fm[0]) / (2 * h) - rho1) < 1e-6 * max(1.0, abs(rho1))
        assert abs((fp[1] - fm[1]) / (2 * h) - rho2) < 1e-5 * max(1e-3, abs(rho2))
    # at s = 0 every loss is s to first order with unit slope
    rho, rho1, rho2 = rr.loss_eval(kind, a, 0.0)
    assert rho == 0.0 and rho1 == 1.0
    h = 1e-7
    assert abs(rr.loss_eval(kind, a, h)[0] / h - 1.0) < 1e-6
    assert abs((rr.loss_eval(kind, a, h)[1] - rho1) / h - rho2) < 1e-4 * max(1e-3, abs(rho2))


def test_loss_closed_forms():
    a = 2.0
    assert rr.loss_eval(rr.LOSS_TRIVIAL, a, 9.0) == (9.0, 1.0, 0.0)
    assert rr.loss_eval(rr.LOSS_HUBER, a, 3.0) == (3.0, 1.0, 0.0)  # inside the knee: s
    np.testing.assert_allclose(rr.loss_eval(rr.LOSS_HUBER, a, 9.0), (2 * a * 3 - a * a, a / 3, -a / 3 / 18))
    np.testing.assert_allclose(rr.loss_eval(rr.LOSS_SOFTLONE, a, 9.0)[0], 2 * 4 * (np.sqrt(1 + 9 / 4) - 1))
    np.testing.assert_allclose(rr.loss_eval(rr.LOSS_CAUCHY, a, 9.0)[0], 4 * np.log(1 + 9 / 4))


def test_trivial_loss_is_bit_identical_to_the_oracle():
    """The robust oracle with the trivial loss is the plain oracle, bit for bit, whatever ran before."""
    po = rc.pose_only(5, 300)
    pb = rc.local(6, C=4, P=80, obs_per_point=(3, 4), fixed_frac=0.2)
    rt0, s0 = ref.ba_pose_only(po["xw"], po["uv"], po["K"], po["rt"])
    c0, p0, t0 = ref.ba_local(pb)
    for before in (None, (rr.LOSS_HUBER, 1.0)):
        if before:
            rr.ba_local(pb, loss=before)
        rt1, s1 = rr.ba_pose_only(po["xw"], po["uv"], po["K"], po["rt"], loss=(rr.LOSS_TRIVIAL, 3.0))
        assert np.array_equal(rt0, rt1) and s0 == s1
        c1, p1, t1 = rr.ba_local(pb, loss=(rr.LOSS_TRIVIAL, 1.0))
        assert np.array_equal(c0, c1) and np.array_equal(p0, p1) and t0 == t1
        c2, p2, t2 = rr.ba_local(pb)
        assert np.array_equal(c0, c2) and np.array_equal(p0, p2) and t0 == t2
        assert rr.ba_local_cost(pb) == ref.ba_local_cost(pb)


def _project(rv, tv, X, fu, fv, K):
    """Ceres AngleAxisRotatePoint (Rodrigues) + pinhole, row-wise over rv [n, 3], tv [n, 3], X [n, 3]."""
    th = np.linalg.norm(rv, axis=1, keepdims=True)
    k = rv / th
    c, s = np.cos(th), np.sin(th)
    q = X * c + np.cross(k, X) * s + k * np.sum(k * X, axis=1, keepdims=True) * (1 - c) + tv
    return np.stack([q[:, 0] / q[:, 2] * fu + K[2], q[:, 1] / q[:, 2] * fv + K[3]], 1)


def _pose_residual_norms(po):
    """|r| of every pose-only observation as a function of the pose (PoseCost: fx for v)."""
    xw, uv, K = po["xw"].astype(np.float64), po["uv"].astype(np.float64), po["K"].astype(np.float64)

    def fun(x):
        n = len(xw)
        r = _project(np.broadcast_to(x[:3], (n, 3)), np.broadcast_to(x[3:], (n, 3)), xw, K[0], K[0], K) - uv
        return np.linalg.norm(r, axis=1)
    return fun


def _local_residual_norms(pb):
    """|r| of every observation (in-window PoseMPCost, then fixed-pose MPCost) as a function of
    (cameras, points)."""
    C, P = len(pb["cams"]), len(pb["pts"])
    K = pb["K"].astype(np.float64)
    frt = pb["fix_rt"].astype(np.float64).reshape(-1, 6)
    uv = np.concatenate([pb["obs_uv"], pb["fix_uv"]]).astype(np.float64)

    def fun(x):
        c, p = x[:6 * C].reshape(C, 6), x[6 * C:].reshape(P, 3)
        rv = np.concatenate([c[pb["obs_cam"], :3], frt[:, :3]])
        tv = np.concatenate([c[pb["obs_cam"], 3:], frt[:, 3:]])
        X = np.concatenate([p[pb["obs_pt"]], p[pb["fix_pt"]]])
        return np.linalg.norm(_project(rv, tv, X, K[0], K[1], K) - uv, axis=1)
    return fun


_SCIPY = {rr.LOSS_HUBER: "huber", rr.LOSS_SOFTLONE: "soft_l1", rr.LOSS_CAUCHY: "cauchy"}


def _scipy_min(fun, x0, kind, a):
    """scipy applies its loss per scalar residual: one residual |r| per observation makes its
    huber / soft_l1 / cauchy the per-block losses of Ceres."""
    from scipy.optimize import least_squares
    return least_squares(fun, x0, jac="3-point", loss=_SCIPY[kind], f_scale=a, x_scale="jac", method="trf",
                         xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=400)


@pytest.mark.parametrize("name", sorted(rc.LOSSES))
def test_pose_only_minimum_matches_scipy(name):
    kind, a = rc.LOSSES[name], rc.SCALE
    po = rc.pose_only(21, 300)
    rt, s = rr.ba_pose_only(po["xw"], po["uv"], po["K"], po["rt"], ref.ba_options(**TIGHT), loss=(kind, a))
    sol = _scipy_min(_pose_residual_norms(po), po["rt"].copy(), kind, a)
    assert abs(sol.cost - s["final_cost"]) <= 1e-9 * s["final_cost"]
    np.testing.assert_allclose(rt, sol.x, rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("name", sorted(rc.LOSSES))
def test_local_minimum_matches_scipy(name):
    kind, a = rc.LOSSES[name], rc.SCALE
    # the fixed observers anchor the gauge, so the minimiser is unique
    pb = rc.local(23, C=3, P=40, obs_per_point=(3,), fixed_frac=0.3)
    cams, pts, s = rr.ba_local(pb, ref.ba_options(**TIGHT), loss=(kind, a))
    assert abs(rr.ba_local_cost(pb, cams, pts, loss=(kind, a)) - s["final_cost"]) <= 1e-12 * s["final_cost"]
    x0 = np.concatenate([pb["cams"].ravel(), pb["pts"].ravel()])
    fun = _local_residual_norms(pb)
    np.testing.assert_allclose(0.5 * np.sum(fun(x0) ** 2), ref.ba_local_cost(pb), rtol=1e-12)
    # scipy's trf crawls on this problem under the Cauchy loss (thousands of evaluations from x0), so
    # it starts from the oracle's answer: a point that is not the minimum would be left for a lower one
    sol = _scipy_min(fun, np.concatenate([cams.ravel(), pts.ravel()]), kind, a)
    assert abs(sol.cost - s["final_cost"]) <= 1e-9 * s["final_cost"]
    np.testing.assert_allclose(np.concatenate([cams.ravel(), pts.ravel()]), sol.x, rtol=1e-6, atol=1e-6)


def test_huber_rejects_outliers_in_pose_only():
    po = rc.pose_only(31, 500)
    rt0, _ = ref.ba_pose_only(po["xw"], po["uv"], po["K"], po["rt"])
    rt1, _ = rr.ba_pose_only(po["xw"], po["uv"], po["K"], po["rt"], loss=(rr.LOSS_HUBER, rc.SCALE))
    e0, e1 = np.linalg.norm(rt0 - po["rt_true"]), np.linalg.norm(rt1 - po["rt_true"])
    assert e1 * 10 <= e0
