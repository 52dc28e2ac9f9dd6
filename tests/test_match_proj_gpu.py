"""GPU parity: projection-guided searches through the C ABI vs the line-by-line
oracle (oracle/match_ref.c).  Bar: bit-exact assignments, including the
reference's sequential claim order and tie-breaks."""
import numpy as np
import pytest

from lorb_slam_b200 import synth
from oracle import ref

pytestmark = pytest.mark.gpu


def _cmp_points(ctx, fr, pts, th):
    r, o = ctx.search_proj_points(fr, pts, th), ref.search_proj_points(fr, pts, th)
    assert r["n_candidates"] == o["n_candidates"]
    assert np.array_equal(r["kp_for_point"], o["kp_for_point"])
    assert np.array_equal(r["point_for_kp"], o["point_for_kp"])
    assert r["n_matches"] == o["n_matches"]
    return o


@pytest.mark.parametrize("th", [1.0, 3.0, 15.0])
@pytest.mark.parametrize("nobs", [1, 0, (0, 1, 2)])
@pytest.mark.parametrize("stereo", [False, True])
def test_points_cfg2(ctx, th, nobs, stereo):
    """BASELINE config 2: 5k map points into a 2000-keypoint 640x480 frame."""
    fr = synth.make_frame(2000, seed=3, stereo=stereo, claimed_frac=0.1)
    pts = synth.make_proj_points(fr, 5000, seed=3, nobs=nobs, inactive_frac=0.05)
    o = _cmp_points(ctx, fr, pts, th)
    assert o["n_matches"] > 100


def test_points_dense_conflicts(ctx):
    """Many points fighting for few keypoints: long claim-dependency chains."""
    fr = synth.make_frame(60, seed=9)
    fr["kp_x"] = (300 + 20 * np.random.default_rng(1).random(60)).astype(np.float32)
    fr["kp_y"] = (200 + 20 * np.random.default_rng(2).random(60)).astype(np.float32)
    fr["kp_octave"][:] = 1
    rng = np.random.default_rng(3)
    n = 3000
    pts = synth.make_proj_points(fr, n, seed=4, true_frac=1.0, sigma_px=4.0, p_flip=0.15,
                                 nobs=(0, 0, 1))
    pts["level"][:] = rng.integers(1, 3, n)
    _cmp_points(ctx, fr, pts, 1.0)
    _cmp_points(ctx, fr, pts, 4.0)


def test_points_edge_cases(ctx):
    fr = synth.make_frame(500, seed=5)
    # keypoints on the right/bottom border round to cell 64/48 and vanish from the grid
    fr["kp_x"][:50] = np.linspace(634.0, 639.99, 50).astype(np.float32)
    fr["kp_y"][50:100] = np.linspace(474.0, 479.99, 50).astype(np.float32)
    pts = synth.make_proj_points(fr, 800, seed=6, true_frac=0.9)
    pts["proj_x"][:20] = -50.0  # windows fully outside
    pts["proj_x"][20:40] = 700.0
    pts["proj_y"][40:60] = 479.9
    pts["level"][60:80] = 0      # minLevel = -1 -> bCheckLevels still true (maxLevel >= 0)
    _cmp_points(ctx, fr, pts, 1.0)
    # nothing active / no points / no keypoints
    pts2 = dict(pts)
    pts2["active"] = np.zeros(800, np.uint8)
    r = ctx.search_proj_points(fr, pts2, 1.0)
    assert r["n_matches"] == 0 and (r["kp_for_point"] == -1).all()
    empty = synth.make_proj_points(fr, 0, seed=1)
    r = ctx.search_proj_points(fr, empty, 1.0)
    assert r["n_matches"] == 0 and (r["point_for_kp"] == -1).all()
    fr0 = synth.make_frame(0, seed=1)
    pts0 = synth.make_proj_points(synth.make_frame(10, seed=1), 50, seed=2)
    r = ctx.search_proj_points(fr0, pts0, 1.0)
    assert r["n_matches"] == 0
    # a very large frame: 15 000 keypoints
    big = synth.make_frame(15000, seed=15000, stereo=True, claimed_frac=0.2)
    _cmp_points(ctx, big, synth.make_proj_points(big, 3000, seed=15000, nobs=(0, 1, 2), inactive_frac=0.1), 1.0)


@pytest.mark.parametrize("motion", ["forward", "backward", "still"])
@pytest.mark.parametrize("th", [15.0, 30.0])
@pytest.mark.parametrize("stereo", [False, True])
def test_frame_search(ctx, motion, th, stereo):
    """Matcher::SearchByProjection(Cur, Last, th) with th = 15 then 30
    (reference src/visual_odometry.cpp:124,129)."""
    for seed in (0, 1):
        cur, last = synth.make_frame_pair(2000, seed=seed, motion=motion, stereo=stereo)
        cur["kp_claim_obs"] = np.where(np.random.default_rng(seed).random(2000) < 0.05, 2, -1).astype(np.int32)
        r, o = ctx.search_proj_frame(cur, last, th), ref.search_proj_frame(cur, last, th)
        assert r["n_candidates"] == o["n_candidates"]
        assert np.array_equal(r["kp_for_item"], o["kp_for_item"])
        assert np.array_equal(r["state_for_kp"], o["state_for_kp"])
        assert r["n_matches"] == o["n_matches"]
        assert o["n_matches"] > 200 and (o["state_for_kp"] == -2).sum() > 0


def test_frame_search_unprotected_overwrites(ctx):
    """mnObs == 0 everywhere: claims never protect, keypoints get overwritten and
    pushed into the rotation histogram more than once (reference :176-188)."""
    cur, last = synth.make_frame_pair(1500, seed=7, motion="still", nobs=(0,))
    r, o = ctx.search_proj_frame(cur, last, 30.0), ref.search_proj_frame(cur, last, 30.0)
    assert np.array_equal(r["kp_for_item"], o["kp_for_item"])
    assert np.array_equal(r["state_for_kp"], o["state_for_kp"])
    assert r["n_matches"] == o["n_matches"]
    taken = o["kp_for_item"][o["kp_for_item"] >= 0]
    assert len(taken) > len(np.unique(taken))  # some keypoint was taken twice


@pytest.mark.parametrize("stereo", [False, True])
def test_candidate_arena_overflow_retry(ctx, stereo):
    """More candidates than the first-attempt arena holds (max(128 per point, 2^18)): the search is
    repeated with the exact size and the claim resolution of the overflowed attempt must not run on
    segments that point past the arena (found by the soak: th = 30 on a 3000-keypoint frame hung)."""
    fr = synth.make_frame(3000, seed=21, stereo=stereo, claimed_frac=0.2)
    pts = synth.make_proj_points(fr, 2500, seed=21, nobs=(0, 1, 2), inactive_frac=0.1)
    o = _cmp_points(ctx, fr, pts, 30.0)
    assert o["n_candidates"] > max(2500 * 128, 1 << 18)
    _cmp_points(ctx, fr, pts, 1.0)  # and the context is fine afterwards
    cur, last = synth.make_frame_pair(3000, seed=5, motion="forward", stereo=stereo)
    r, o = ctx.search_proj_frame(cur, last, 120.0), ref.search_proj_frame(cur, last, 120.0)
    assert o["n_candidates"] > max(3000 * 128, 1 << 18)
    assert r["n_candidates"] == o["n_candidates"] and r["n_matches"] == o["n_matches"]
    assert np.array_equal(r["kp_for_item"], o["kp_for_item"])
    assert np.array_equal(r["state_for_kp"], o["state_for_kp"])


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_frustum_project(ctx, seed):
    """SURVEY 8(f) rank 1: Frame::IsInFrustum + PredictScale, bit-exact vs the oracle."""
    fp = synth.make_frustum_points(20000, seed)
    g, o = ctx.frustum_project(fp), ref.frustum_project(fp)
    assert 2000 < o["in_view"].sum() < 19000
    for k in ("in_view", "proj_x", "proj_y", "proj_xr", "level", "view_cos"):
        assert np.array_equal(g[k], o[k]), k
    # its outputs feed the local-map search unchanged
    fr = synth.make_frame(2000, seed=seed)
    m = int(min(5000, fp["n"]))
    pts = synth.make_proj_points(fr, m, seed=seed)
    pts["proj_x"], pts["proj_y"], pts["proj_xr"] = g["proj_x"][:m], g["proj_y"][:m], g["proj_xr"][:m]
    pts["level"] = np.clip(g["level"][:m], 0, 7).astype(np.int32)
    pts["view_cos"], pts["active"] = g["view_cos"][:m], g["in_view"][:m]
    r, q = ctx.search_proj_points(fr, pts, 1.0), ref.search_proj_points(fr, pts, 1.0)
    assert np.array_equal(r["kp_for_point"], q["kp_for_point"]) and r["n_matches"] == q["n_matches"]
