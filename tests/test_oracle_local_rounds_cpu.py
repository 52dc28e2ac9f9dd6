"""CPU: the outlier-round reference of lorb_ba_local_rounds_batched (tests/oracle_ext.py).  One
round with unit weights and no threshold is the plain and the robust oracle bit for bit; the last round
is the weighted minimum of scipy.optimize.least_squares on its inlier set; the rounds find planted
outliers; the depth check flags a point behind its camera; a window without inliers stops at its
first gradient test."""
import numpy as np
import pytest

import local_rounds_cases as lc
import oracle_ext as lr
import robust_cases as rc
from oracle import ref

TIGHT = dict(max_num_iterations=200, function_tolerance=1e-15, gradient_tolerance=1e-14,
             parameter_tolerance=1e-14)


def test_one_round_without_threshold_is_the_oracle():
    pb = rc.local(5, C=6, P=300, obs_per_point=(3, 4, 5), fixed_frac=0.1)
    O, F = len(pb["obs_cam"]), pb["F"]
    opt = ref.ba_options(max_num_iterations=10)
    for loss in [None] + [(k, rc.SCALE) for k in rc.LOSSES.values()]:
        oc, op, o = lr.ba_local(pb, opt, loss=loss)
        for w, fw in ((None, None), (np.ones(O, np.float32), np.ones(F, np.float32))):
            cams, pts, inl, _, finl, _, n_in, sums = lr.ba_local_rounds(
                pb, w, fw, n_rounds=1, robust_rounds=1, chi2=1e30, opt=opt, loss=loss)
            assert np.array_equal(cams, oc) and np.array_equal(pts, op) and sums[0] == o
            assert inl.all() and finl.all() and n_in == O + F


def _weighted_norms(pb, w, fw):
    """sqrt(w) |r| of every observation (in-window PoseMPCost, then fixed-pose MPCost) as a function of
    (cameras, points)."""
    C, P = len(pb["cams"]), len(pb["pts"])
    K = pb["K"].astype(np.float64)
    frt = pb["fix_rt"].astype(np.float64).reshape(-1, 6)
    uv = np.concatenate([pb["obs_uv"], pb["fix_uv"]]).astype(np.float64)
    sw = np.sqrt(np.concatenate([w, fw]).astype(np.float64))

    def fun(x):
        c, p = x[:6 * C].reshape(C, 6), x[6 * C:].reshape(P, 3)
        rv = np.concatenate([c[pb["obs_cam"], :3], frt[:, :3]])
        tv = np.concatenate([c[pb["obs_cam"], 3:], frt[:, 3:]])
        X = np.concatenate([p[pb["obs_pt"]], p[pb["fix_pt"]]])
        R = lc.synth.rodrigues(rv)
        q = np.einsum("nij,nj->ni", R, X) + tv
        r = np.stack([q[:, 0] / q[:, 2] * K[0] + K[2], q[:, 1] / q[:, 2] * K[1] + K[3]], 1) - uv
        return sw * np.linalg.norm(r, axis=1)
    return fun


def test_last_round_is_the_weighted_minimum_on_its_inlier_set():
    from scipy.optimize import least_squares
    # the fixed observers anchor the gauge, so the minimiser is unique
    pb, w, fw, _, _ = lc.planted(23, 0.1, C=3, P=60, obs_per_point=(3,), fixed_frac=0.3)
    opt = [ref.ba_options(**TIGHT)] * 2
    # the plain second round solves over the classification after the robust first one
    _, _, inl0, _, finl0, _, _, _ = lr.ba_local_rounds(pb, w, fw, n_rounds=1, opt=opt[:1], loss=lc.HUBER)
    cams, pts, _, _, _, _, _, sums = lr.ba_local_rounds(pb, w, fw, opt=opt, loss=lc.HUBER)
    assert not inl0.all() and sums[1]["iterations"] > 0
    sub = dict(pb, obs_cam=pb["obs_cam"][inl0], obs_pt=pb["obs_pt"][inl0], obs_uv=pb["obs_uv"][inl0],
               fix_pt=pb["fix_pt"][finl0], fix_uv=pb["fix_uv"][finl0], fix_rt=pb["fix_rt"][finl0])
    fun = _weighted_norms(sub, w[inl0], fw[finl0])
    x = np.concatenate([cams.ravel(), pts.ravel()])
    np.testing.assert_allclose(0.5 * np.sum(fun(x) ** 2), sums[1]["final_cost"], rtol=1e-10)
    sol = least_squares(fun, x, jac="3-point", x_scale="jac", method="trf", xtol=1e-15, ftol=1e-15, gtol=1e-15,
                        max_nfev=400)
    assert abs(sol.cost - sums[1]["final_cost"]) <= 1e-9 * sums[1]["final_cost"]
    np.testing.assert_allclose(x, sol.x, rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("frac", [0.1, 0.3])
def test_rounds_flag_planted_outliers(frac):
    # 8-10 observations per point: with 30 % moved, a point still has a clean majority
    pb, w, fw, bad, fbad = lc.planted(51, frac, C=10, P=800, obs_per_point=(8, 9, 10), fixed_frac=0.1)
    cams, pts, inl, chi2, finl, fchi2, n_in, sums = lr.ba_local_rounds(pb, w, fw, loss=lc.HUBER)
    assert n_in == inl.sum() + finl.sum()
    flags, c2, moved = np.concatenate([inl, finl]), np.concatenate([chi2, fchi2]), np.concatenate([bad, fbad])
    assert np.array_equal(flags, c2 <= 5.991)  # no point ends up behind a camera here
    assert (~flags[moved]).mean() >= 0.95
    # unit pixel noise and weights <= 1: at most the 5 % chi-square tail of the clean observations
    assert (~flags[~moved]).mean() <= 0.05


def test_depth_check_flags_a_point_behind_its_camera():
    pb0 = rc.local(61, 0.0, C=5, P=100, obs_per_point=(3,), fixed_frac=0.2)
    pb, i = lc.behind_camera(pb0, 7)
    # classification at the input parameters, by depth alone
    kw = dict(n_rounds=1, chi2=1e30, opt=[ref.ba_options(max_num_iterations=0)])
    _, _, _, chi2_0, _, _, _, _ = lr.ba_local_rounds(pb0, **kw)
    for depth_check in (0, 1):
        _, _, inl, chi2, _, _, _, _ = lr.ba_local_rounds(pb, depth_check=depth_check, **kw)
        np.testing.assert_allclose(chi2[i], chi2_0[i], rtol=1e-9)
        assert inl[i] == (depth_check == 0) and inl[pb["obs_pt"] != 7].all()


def test_window_without_inliers_stops_at_the_gradient_test():
    pb = rc.local(71, 0.1, C=4, P=80, obs_per_point=(3,), fixed_frac=0.2)
    c1, p1, _, _, _, _, _, s1 = lr.ba_local_rounds(pb, n_rounds=1, chi2=1e-30, opt=lr.budgets(2, None)[:1])
    cams, pts, inl, _, finl, _, n_in, sums = lr.ba_local_rounds(pb, chi2=1e-30)
    assert n_in == 0 and not inl.any() and not finl.any()
    assert sums[0] == s1[0] and sums[1]["termination"] == lc.CONV_GRADIENT and sums[1]["iterations"] == 0
    assert np.array_equal(cams, c1) and np.array_equal(pts, p1)
