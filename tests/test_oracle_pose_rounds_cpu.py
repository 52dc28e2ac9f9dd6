"""CPU: the outlier-round reference of lorb_ba_pose_rounds_batched (tests/oracle_ext.py).  One round
without a threshold is the plain and the robust oracle bit for bit; the weighted minimum of the last
round matches scipy.optimize.least_squares; the rounds find planted outliers; the skip rule holds."""
import numpy as np
import pytest

import oracle_ext as rd
import robust_cases as rc
from oracle import ref

TIGHT = dict(max_num_iterations=200, function_tolerance=1e-15, gradient_tolerance=1e-14,
             parameter_tolerance=1e-14)
SCALE_FACTOR = 1.2  # ORB pyramid


def octave_weights(n, seed):
    """w = 1 / sigma^2 of a random ORB octave 0..7 (Frame::mvInvLevelSigma2)."""
    oct_ = np.random.default_rng(seed + 3).integers(0, 8, n)
    return (1.0 / (SCALE_FACTOR ** oct_) ** 2).astype(np.float32)


def planted(seed, n, frac, sigma0=0.5):
    """pose_only data with `frac` of the observations moved 20-80 px, keypoint noise sigma0 * 1.2^octave
    (so the octave weights are the true inverse variances), the weights, and the mask of the moved rows."""
    clean = rc.synth.make_pose_only(seed, n, pixel_noise=0.0)
    po = rc.pose_only(seed, n, frac, pixel_noise=0.0)
    w = octave_weights(n, seed)
    noise = np.random.default_rng(seed + 5).normal(0, sigma0, (n, 2)) / np.sqrt(w)[:, None]
    po["uv"] = (po["uv"] + noise).astype(np.float32)
    return po, w, np.any(po["uv"] != (clean["uv"] + noise).astype(np.float32), axis=1)


def pose_err(rt, po):
    return np.linalg.norm(rt - po["rt_true"])


@pytest.mark.parametrize("weights", [False, True])
def test_one_round_without_threshold_is_the_oracle(weights):
    po = rc.pose_only(5, 300)
    w = np.ones(300, np.float32) if weights else None
    rt0, s0 = ref.ba_pose_only(po["xw"], po["uv"], po["K"], po["rt"])
    rt1, inl, _, n_in, run, sums = rd.ba_pose_rounds(po["xw"], po["uv"], po["K"], po["rt"], w, n_rounds=1,
                                                     robust_rounds=1, chi2=1e30)
    assert np.array_equal(rt0, rt1) and sums[0] == s0
    assert inl.all() and n_in == 300 and run == 1
    for kind in rc.LOSSES.values():
        rt0, s0 = rd.ba_pose_only(po["xw"], po["uv"], po["K"], po["rt"], loss=(kind, rc.SCALE))
        rt1, _, _, _, _, sums = rd.ba_pose_rounds(po["xw"], po["uv"], po["K"], po["rt"], w, n_rounds=1,
                                                  robust_rounds=1, chi2=1e30, loss=(kind, rc.SCALE))
        assert np.array_equal(rt0, rt1) and sums[0] == s0


def _weighted_norms(xw, uv, K, w):
    """sqrt(w) |r| of every observation as a function of the pose (PoseCost: fx for v)."""
    xw, uv, K, sw = xw.astype(np.float64), uv.astype(np.float64), K.astype(np.float64), np.sqrt(w.astype(np.float64))

    def fun(x):
        th = np.linalg.norm(x[:3])
        k = x[:3] / th
        c, s = np.cos(th), np.sin(th)
        q = xw * c + np.cross(k, xw) * s + np.outer(xw @ k, k) * (1 - c) + x[3:]
        r = np.stack([q[:, 0] / q[:, 2] * K[0] + K[2], q[:, 1] / q[:, 2] * K[0] + K[3]], 1) - uv
        return sw * np.linalg.norm(r, axis=1)
    return fun


@pytest.mark.parametrize("name", sorted(rc.LOSSES))
def test_last_round_is_the_weighted_minimum_on_its_inlier_set(name):
    from scipy.optimize import least_squares
    po = rc.pose_only(41, 400, 0.2)
    w = octave_weights(400, 41)
    opt, loss = ref.ba_options(**TIGHT), (rc.LOSSES[name], rc.SCALE)
    # the inlier set the fourth (plain) round solves over is the classification after the third
    _, inl3, _, _, run3, _ = rd.ba_pose_rounds(po["xw"], po["uv"], po["K"], po["rt"], w, n_rounds=3, opt=opt, loss=loss)
    rt, _, _, _, run, sums = rd.ba_pose_rounds(po["xw"], po["uv"], po["K"], po["rt"], w, opt=opt, loss=loss)
    assert run3 == 3 and run == 4
    fun = _weighted_norms(po["xw"][inl3], po["uv"][inl3], po["K"], w[inl3])
    sol = least_squares(fun, po["rt"].copy(), jac="3-point", x_scale="jac", method="trf", xtol=1e-15, ftol=1e-15,
                        gtol=1e-15, max_nfev=400)
    assert abs(sol.cost - sums[3]["final_cost"]) <= 1e-9 * sums[3]["final_cost"]
    np.testing.assert_allclose(rt, sol.x, rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("frac", [0.1, 0.3])
@pytest.mark.parametrize("name", sorted(rc.LOSSES))
def test_rounds_flag_planted_outliers(frac, name):
    po, w, bad = planted(51, 2000, frac)
    rt0, _ = ref.ba_pose_only(po["xw"], po["uv"], po["K"], po["rt"])
    rt, inl, chi2, n_in, run, _ = rd.ba_pose_rounds(po["xw"], po["uv"], po["K"], po["rt"], w,
                                                    loss=(rc.LOSSES[name], rc.SCALE))
    assert run == 4 and n_in == inl.sum()
    assert np.array_equal(inl, chi2 <= 5.991)
    assert (~inl[bad]).mean() >= 0.99
    assert (~inl[~bad]).mean() <= 0.02
    assert pose_err(rt, po) * 10 <= pose_err(rt0, po)


def test_fewer_than_three_observations_run_no_round():
    po = rc.pose_only(61, 4, 0.0)
    for n in range(4):
        rt, inl, chi2, n_in, run, sums = rd.ba_pose_rounds(po["xw"][:n], po["uv"][:n], po["K"], po["rt"])
        if n < 3:
            assert np.array_equal(rt, po["rt"]) and run == 0
            assert all(all(v == 0 for v in s.values()) for s in sums)
            assert np.array_equal(inl, chi2 <= 5.991) and n_in == inl.sum()
        else:
            assert run >= 1 and sums[0]["iterations"] > 0


def test_round_that_would_start_with_two_inliers_is_skipped():
    po = rc.pose_only(71, 8, 0.0)
    # chi^2 at the pose of round 0 (which does not depend on the threshold); a threshold between the
    # second and third smallest leaves two inliers for round 1
    rt1, _, c2, _, _, s1 = rd.ba_pose_rounds(po["xw"], po["uv"], po["K"], po["rt"], n_rounds=1, chi2=1e30)
    th = float(np.mean(np.sort(c2)[1:3]))
    rt, inl, chi2, n_in, run, sums = rd.ba_pose_rounds(po["xw"], po["uv"], po["K"], po["rt"], chi2=th)
    assert run == 1 and n_in == 2 and inl.sum() == 2
    assert np.array_equal(rt, rt1) and np.array_equal(chi2, c2) and sums[0] == s1[0]
    assert all(all(v == 0 for v in s.values()) for s in sums[1:])
