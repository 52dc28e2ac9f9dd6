"""CPU: the host restatement of lorb_pnp_ransac_batched (tests/pnp_ref.py).  The sampler draws four distinct,
in-range, roughly uniform indices as a pure function of (seed, h, n); the P3P solution set matches OpenCV's P3P
and recovers a planted pose exactly; RANSAC finds the planted pose and its inliers at 0-60 % outliers (as does
cv2.solvePnPRansac); degenerate inputs select nothing and produce no NaN; the angle-axis conversion round-trips."""
import cv2
import numpy as np
import pytest

import pnp_ref as pr
from lorb_slam_b200 import synth

CHI2 = 5.991


def _rot_err_deg(rv, rv_true):
    R, Rt = synth.rodrigues(rv), synth.rodrigues(rv_true)
    return np.degrees(np.arccos(np.clip((np.trace(R.T @ Rt) - 1) / 2, -1, 1)))


def test_sampler_draws_four_distinct_indices_as_a_pure_function():
    for n in (4, 5, 7, 300, 100000):
        for h in range(200):
            idx = pr.draw4(12345, h, n)
            assert idx is not None and len(set(idx.tolist())) == 4 and idx.min() >= 0 and idx.max() < n
            assert np.array_equal(idx, pr.draw4(12345, h, n))
    assert not np.array_equal(pr.draw4(1, 0, 300), pr.draw4(2, 0, 300))
    assert not np.array_equal(pr.draw4(1, 0, 300), pr.draw4(1, 1, 300))
    assert pr.draw4(0, 0, 3) is None  # three indices cannot give four distinct ones


def test_sampler_is_roughly_uniform():
    n = 50
    draws = np.concatenate([pr.draw4(99, h, n) for h in range(25000)])  # 10^5 indices
    counts = np.bincount(draws, minlength=n)
    e = len(draws) / n
    chi2 = ((counts - e) ** 2 / e).sum()
    assert chi2 < 120  # 49 degrees of freedom: p ~ 1e-7 at 120


def _project(rt, X, K):
    q = X @ synth.rodrigues(rt[:3]).T + rt[3:]
    return np.stack([K[0] * q[:, 0] / q[:, 2] + K[2], K[1] * q[:, 1] / q[:, 2] + K[3]], 1), q[:, 2]


def _reproj_ok(R, t, X, uv, K, tol=1e-6):
    q = X @ R.T + t
    p = np.stack([K[0] * q[:, 0] / q[:, 2] + K[2], K[1] * q[:, 1] / q[:, 2] + K[3]], 1)
    return np.abs(p - uv).max() <= tol


def test_p3p_solution_set_matches_opencv():
    rng = np.random.default_rng(3)
    K = np.array([458.0, 452.0, 320.0, 240.0], np.float32)
    Km = np.array([[K[0], 0, K[2]], [0, K[1], K[3]], [0, 0, 1]], np.float64)
    compared = 0
    for _ in range(1000):
        rt = np.concatenate([rng.normal(0, 0.5, 3), rng.normal(0, 1.0, 3)])
        Xc = np.stack([rng.uniform(-4, 4, 3), rng.uniform(-3, 3, 3), rng.uniform(3, 20, 3)], 1)
        X = ((Xc - rt[3:]) @ synth.rodrigues(rt[:3])).astype(np.float32)
        uv = _project(rt, X.astype(np.float64), K.astype(np.float64))[0].astype(np.float32)
        Xd, uvd = X.astype(np.float64), uv.astype(np.float64)
        R, t = pr.p3p(X, uv, K)
        ours = [(Ri, ti) for Ri, ti in zip(R, t) if _reproj_ok(Ri, ti, Xd, uvd, K)]
        _, rv, tv = cv2.solveP3P(Xd, uvd, Km, None, flags=cv2.SOLVEPNP_P3P)
        theirs = [(cv2.Rodrigues(r)[0], tt.reshape(3)) for r, tt in zip(rv, tv)]
        theirs = [(Ri, ti) for Ri, ti in theirs if _reproj_ok(Ri, ti, Xd, uvd, K)]
        same = lambda a, b: np.abs(a[0] - b[0]).max() <= 1e-6 and np.abs(a[1] - b[1]).max() <= 1e-6
        assert all(any(same(a, b) for b in theirs) for a in ours)
        assert all(any(same(a, b) for a in ours) for b in theirs)
        compared += len(ours)
    assert compared >= 1000


def test_p3p_recovers_an_exactly_representable_planted_pose():
    # dyadic camera points, signed-permutation rotations and dyadic translations: xw and uv are exact floats,
    # so the noise-free solution must equal the planted pose to rounding
    rng = np.random.default_rng(4)
    K = np.array([512.0, 256.0, 320.0, 256.0], np.float32)
    for _ in range(200):
        P = np.eye(3)[rng.permutation(3)] * rng.choice([-1.0, 1.0], 3)[:, None]
        if np.linalg.det(P) < 0:
            P[0] *= -1
        t = rng.integers(-64, 64, 3) / 16.0
        z = 2.0 ** rng.integers(2, 5, 3)
        xc = np.stack([rng.integers(-128, 128, 3) / 64.0 * z / 4, rng.integers(-128, 128, 3) / 64.0 * z / 4, z], 1)
        X = (xc - t) @ P  # P^T (xc - t), exact
        uv = np.stack([K[0] * xc[:, 0] / xc[:, 2] + K[2], K[1] * xc[:, 1] / xc[:, 2] + K[3]], 1)
        assert np.array_equal(X.astype(np.float32), X) and np.array_equal(uv.astype(np.float32), uv)
        R, tt = pr.p3p(X, uv, K)
        err = [max(np.abs(Ri - P).max(), np.abs(ti - t).max()) for Ri, ti in zip(R, tt)]
        if np.linalg.matrix_rank(np.stack([X[0] - X[1], X[0] - X[2]])) == 2 and len(set(map(tuple, uv))) == 3:
            assert min(err) <= 1e-9, err


@pytest.mark.parametrize("frac", [0.0, 0.3, 0.6])
def test_ransac_finds_planted_pose_and_inliers(frac):
    for seed in range(3):
        d = synth.make_pnp_problems(20 + seed, n=300, outlier_frac=frac, noise="uniform")
        rt, best, n_in, inl, c2 = pr.ransac(d["corr_off"], d["xw"], d["uv"], d["K"], d["info"])
        truth = d["rt_true"][0]
        depth = np.median(_project(truth, d["xw"].astype(np.float64), d["K"])[1])
        assert best[0] >= 0 and n_in[0] == inl.sum()
        assert np.array_equal(inl, c2 <= CHI2)
        assert _rot_err_deg(rt[0, :3], truth[:3]) < 1.0
        assert np.linalg.norm(rt[0, 3:] - truth[3:]) < 0.02 * depth
        ti = ~d["outlier"]  # every planted inlier is within the threshold at the planted pose (|noise| <= 1 px)
        assert (inl & ti).sum() >= 0.95 * ti.sum()
        # OpenCV on the same data
        Km = np.array([[d["K"][0], 0, d["K"][2]], [0, d["K"][1], d["K"][3]], [0, 0, 1]], np.float64)
        ok, rv, tv, _ = cv2.solvePnPRansac(d["xw"].astype(np.float64), d["uv"].astype(np.float64), Km, None,
                                           flags=cv2.SOLVEPNP_P3P, iterationsCount=300,
                                           reprojectionError=float(np.sqrt(CHI2)))
        assert ok and _rot_err_deg(rv.reshape(3), truth[:3]) < 1.0
        assert np.linalg.norm(tv.reshape(3) - truth[3:]) < 0.02 * depth


def test_degenerate_inputs_select_nothing():
    d = synth.make_pnp_problems(5, n=200, outlier_frac=0.0, collinear=True)
    rt, best, n_in, inl, c2 = pr.ransac(d["corr_off"], d["xw"], d["uv"], d["K"], d["info"])
    assert best[0] == -1 and n_in[0] == 0 and not inl.any()
    assert np.array_equal(rt, np.zeros((1, 6))) and np.all(c2 == np.inf)
    for n in range(4):
        d = synth.make_pnp_problems(6, n=n, outlier_frac=0.0)
        rt, best, n_in, inl, c2 = pr.ransac(d["corr_off"], d["xw"], d["uv"], d["K"])
        assert best[0] == -1 and n_in[0] == 0 and not inl.any() and np.all(c2 == np.inf)
        assert np.array_equal(rt, np.zeros((1, 6)))


def test_angle_axis_round_trip():
    rng = np.random.default_rng(8)
    axes = rng.normal(0, 1, (300, 3))
    axes /= np.linalg.norm(axes, axis=1)[:, None]
    thetas = np.concatenate([rng.uniform(0, np.pi, 100), 10.0 ** rng.uniform(-14, -8, 100),
                             np.pi - 10.0 ** rng.uniform(-10, -6, 100)])
    for k, th in zip(axes, thetas):
        w = k * th
        assert np.abs(pr.rotation_to_angle_axis(synth.rodrigues(w)) - w).max() <= 1e-12, th
    assert np.array_equal(pr.rotation_to_angle_axis(np.eye(3)), np.zeros(3))
