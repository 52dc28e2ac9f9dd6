"""GPU: pose-only BA with outlier rounds (lorb_ba_pose_rounds_batched) against the outlier-round
reference (tests/oracle_ext.py): pose within 1e-6, identical flags, inlier counts, rounds run and LM
trajectories; the single-round limit against lorb_ba_pose_only bit for bit; a mixed batch against the
single-frame calls bit for bit; refusal of invalid arguments; and the drop-in tracking loop
(lorb_host::PoseOptimization, then Matcher::SearchByProjection reading its mvbOutlier flags)."""
import ctypes as C

import numpy as np
import pytest

import oracle_ext as rd
import robust_cases as rc
from lorb_slam_b200 import capi, synth
from oracle import ref
from test_oracle_pose_rounds_cpu import octave_weights, planted

pytestmark = pytest.mark.gpu
NAMES = ["trivial"] + sorted(rc.LOSSES)
CHI2 = 5.991


@pytest.fixture
def lctx(ctx):
    """The session ctx, put back to the trivial loss afterwards."""
    yield ctx
    ctx.ba_set_loss(capi.LOSS_TRIVIAL)


def _loss(name):
    return None if name == "trivial" else (rc.LOSSES[name], rc.SCALE)


def _set(ctx, name):
    ctx.ba_set_loss(*(_loss(name) or (capi.LOSS_TRIVIAL, 1.0)))


def _same_summary(s, o):
    for k in ("iterations", "num_successful_steps", "num_unsuccessful_steps", "termination"):
        assert s[k] == o[k], (k, s, o)
    np.testing.assert_allclose(s["initial_cost"], o["initial_cost"], rtol=1e-10)
    # a frame of 3 observations (6 residuals, 6 unknowns) is fitted exactly: its final cost is rounding noise
    # (~1e-20), and so is the step quality of the last steps, which sets the radius growth (x1 .. x3)
    floor = 1e-15 * o["initial_cost"]
    if o["final_cost"] <= floor:
        assert s["final_cost"] <= floor, (s, o)
        return
    np.testing.assert_allclose(s["final_cost"], o["final_cost"], rtol=1e-8)
    np.testing.assert_allclose(s["final_radius"], o["final_radius"], rtol=1e-5)


def _same_as_reference(g, o, chi2=CHI2):
    """g, o: (rt, inlier, chi2, n_inliers, rounds_run, summaries) of one frame."""
    # a flag may only differ where the reference's chi^2 is within 1e-6 of the threshold: no case may lie there
    assert not np.any(np.abs(o[2] - chi2) <= 1e-6 * chi2), "a chi^2 lies in the band of the threshold"
    np.testing.assert_allclose(g[0], o[0], rtol=1e-6, atol=1e-8)
    assert np.array_equal(g[1], o[1])
    assert g[3] == o[3] and g[4] == o[4]
    np.testing.assert_allclose(g[2], o[2], rtol=1e-6, atol=1e-9)
    for r, (s, t) in enumerate(zip(g[5], o[5])):
        if r < o[4]:
            _same_summary(s, t)
        else:
            assert all(v == 0 for v in s.values()) and all(v == 0 for v in t.values())


@pytest.mark.parametrize("weights", [False, True])
@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("n", [50, 300, 2000])
def test_matches_reference(lctx, n, name, weights):
    po, w, _ = planted(100 + n, n, 0.2)
    w = w if weights else None
    _set(lctx, name)
    g = lctx.ba_pose_rounds(po["xw"], po["uv"], po["K"], po["rt"], info=w)
    o = rd.ba_pose_rounds(po["xw"], po["uv"], po["K"], po["rt"], w, loss=_loss(name))
    assert o[4] == (1 if (n, name, weights) == (50, "trivial", False) else 4)  # plain LS can leave < 3 inliers
    _same_as_reference(g, o)


@pytest.mark.parametrize("name", NAMES)
def test_one_round_without_threshold_is_pose_only(lctx, name):
    po = rc.pose_only(9, 700)
    _set(lctx, name)
    rt0, s0 = lctx.ba_pose_only(po["xw"], po["uv"], po["K"], po["rt"])
    rt1, inl, _, n_in, run, sums = lctx.ba_pose_rounds(
        po["xw"], po["uv"], po["K"], po["rt"], rounds=capi.pose_rounds_options(n_rounds=1, robust_rounds=1, chi2=1e30))
    assert np.array_equal(rt0, rt1) and sums[0] == s0
    assert inl.all() and n_in == 700 and run == 1


def _mixed_batch(seed, n_frames=300):
    rng = np.random.default_rng(seed)
    sizes = rng.choice([0, 1, 2, 3, 17, 1000, 5000], n_frames, p=[.05, .05, .05, .05, .3, .4, .1])
    frames = []
    for f, n in enumerate(sizes):
        frac = 0.0 if rng.random() < 0.5 else rng.uniform(0.05, 0.4)
        if n >= 3:
            po, w, _ = planted(1000 + f, int(n), frac)
        else:
            po = rc.pose_only(1000 + f, max(int(n), 1), 0.0)
            po = dict(po, xw=po["xw"][:n], uv=po["uv"][:n])
            w = octave_weights(int(n), f)
        frames.append((po, w))
    off = np.cumsum([0] + [len(p["xw"]) for p, _ in frames]).astype(np.int32)
    cat = lambda k, d: np.concatenate([p[k].reshape(-1, d) for p, _ in frames])
    return (frames, off, cat("xw", 3), cat("uv", 2), np.stack([p["rt"] for p, _ in frames]),
            np.concatenate([w for _, w in frames]))


@pytest.mark.parametrize("name", ["trivial", "huber"])
def test_batch_equals_single_frames_and_reference(lctx, name):
    frames, off, xw, uv, rt, w = _mixed_batch(3)
    K = frames[0][0]["K"]
    _set(lctx, name)
    B = lctx.ba_pose_rounds_batched(off, xw, uv, K, rt, info=w)
    assert set(np.diff(off)) == {0, 1, 2, 3, 17, 1000, 5000}
    for f, (po, wf) in enumerate(frames):
        a, b = off[f], off[f + 1]
        g = lctx.ba_pose_rounds(po["xw"], po["uv"], K, po["rt"], info=wf)
        assert np.array_equal(B[0][f], g[0]) and np.array_equal(B[1][a:b], g[1]) and np.array_equal(B[2][a:b], g[2])
        assert B[3][f] == g[3] and B[4][f] == g[4] and B[5][f] == g[5]
        if b - a in (0, 1, 2, 3, 17, 1000) or f % 4 == 0:  # the reference is slow at 5000 x 4 rounds
            _same_as_reference(g, rd.ba_pose_rounds(po["xw"], po["uv"], K, po["rt"], wf, loss=_loss(name)))
    assert B[4][np.diff(off) < 3].max() == 0


def test_invalid_arguments_are_refused_and_outputs_untouched(lctx):
    lib = capi.load_library()
    po, w, _ = planted(5, 40, 0.1)
    n = 40
    off = np.array([0, 20, n], np.int32)
    xw, uv, K = po["xw"], po["uv"], po["K"]
    rt = np.tile(po["rt"], (2, 1))
    opt = capi.ba_options()
    P = lambda a: a.ctypes.data_as(C.c_void_p)

    def call(off=off, w=w, rounds=None, nf=2):
        rt1, inl = rt.copy(), np.full(n, 7, np.uint8)
        chi2, n_in, run = np.full(n, -1.0), np.full(2, -1, np.int32), np.full(2, -1, np.int32)
        sums = (capi.BASummary * 32)()
        for s in sums:
            s.iterations = -9
        rounds = rounds or capi.pose_rounds_options()
        rc_ = lib.lorb_ba_pose_rounds_batched(lctx._h, nf, P(off), P(xw), P(uv), P(w) if w is not None else None,
                                              P(K), P(rt1), C.byref(rounds), C.byref(opt), P(inl), P(chi2),
                                              P(n_in), P(run), sums)
        untouched = (np.array_equal(rt1, rt) and (inl == 7).all() and (chi2 == -1).all() and (n_in == -1).all()
                     and (run == -1).all() and all(s.iterations == -9 for s in sums))
        return rc_, untouched

    assert call()[0] == 0
    bad = [dict(off=np.array([1, 20, n], np.int32)), dict(off=np.array([0, 30, 20], np.int32)),
           dict(nf=-1),
           dict(w=np.where(np.arange(n) == 3, 0.0, w).astype(np.float32)),
           dict(w=np.where(np.arange(n) == 3, -1.0, w).astype(np.float32)),
           dict(w=np.where(np.arange(n) == 3, np.nan, w).astype(np.float32)),
           dict(w=np.where(np.arange(n) == 3, np.inf, w).astype(np.float32)),
           dict(rounds=capi.pose_rounds_options(n_rounds=0)), dict(rounds=capi.pose_rounds_options(n_rounds=17)),
           dict(rounds=capi.pose_rounds_options(robust_rounds=-1)),
           dict(rounds=capi.pose_rounds_options(robust_rounds=5)),
           dict(rounds=capi.pose_rounds_options(chi2=0.0)), dict(rounds=capi.pose_rounds_options(chi2=float("inf"))),
           dict(rounds=capi.pose_rounds_options(chi2=float("nan")))]
    for kw in bad:
        rc_, untouched = call(**kw)
        assert rc_ == -1, kw
        assert untouched, kw
    # n_frames = 0 is a no-op
    rc_, untouched = call(nf=0)
    assert rc_ == 0 and untouched


def test_dropin_pose_optimization_closes_the_tracking_loop(lctx):
    from lorb_slam_b200.host import build_host
    H = C.CDLL(build_host.build())
    P = lambda a: a.ctypes.data_as(C.c_void_p)
    cur, last = synth.make_frame_pair(2000, seed=4, motion="forward")
    cur["kp_claim_obs"][:] = -1
    Kd = last["K"]
    K6 = np.array([Kd["fx"], Kd["fy"], Kd["cx"], Kd["cy"], Kd["mbf"], Kd["mb"]], np.float32)
    n_last = last["n_last"]
    # Last's keypoints: its map points seen from Last (at the identity) with octave noise, 15 % moved 20-80 px
    rng = np.random.default_rng(44)
    sf = cur["scale_factors"].astype(np.float32)
    xw = last["xw"].astype(np.float64)
    luv = np.stack([xw[:, 0] / xw[:, 2] * K6[0] + K6[2], xw[:, 1] / xw[:, 2] * K6[0] + K6[3]], 1)
    luv += rng.normal(0, 0.5, luv.shape) * sf[last["octave"]][:, None]
    moved = rng.random(n_last) < 0.15
    ang = rng.uniform(0, 2 * np.pi, n_last)
    mag = rng.uniform(20, 80, n_last)
    luv[moved] += np.stack([mag * np.cos(ang), mag * np.sin(ang)], 1)[moved]
    luv = np.ascontiguousarray(luv, np.float32)
    rt = np.array([0.004, -0.003, 0.002, 0.03, -0.02, 0.05], np.float32)
    rt_in = rt.copy()
    outl, tcw_last = np.zeros(n_last, np.uint8), np.zeros(16, np.float32)
    state, n_m = np.zeros(cur["n_kp"], np.int32), C.c_int()
    n_in = H.harness_pose_rounds_search(
        cur["n_kp"], P(cur["kp_x"]), P(cur["kp_y"]), P(cur["kp_octave"]), P(cur["kp_angle"]), P(cur["kp_uright"]),
        P(cur["desc"]), C.c_float(cur["min_x"]), C.c_float(cur["max_x"]), C.c_float(cur["min_y"]),
        C.c_float(cur["max_y"]), cur["n_levels"], P(sf), P(last["tcw_cur"]), P(K6), n_last, P(last["valid"]),
        P(last["xw"]), P(last["octave"]), P(last["angle"]), P(luv), P(last["mp_desc"]), P(last["mp_nobs"]),
        P(rt), C.c_float(15.0), P(outl), P(tcw_last), P(state), C.byref(n_m))
    # the same solve through Python: octave weights, Huber sqrt(5.991) in rounds 0-2, 10 iterations a round
    v = last["valid"].astype(bool)
    w = (np.float32(1) / (sf[last["octave"][v]] * sf[last["octave"][v]])).astype(np.float32)
    lctx.ba_set_loss(capi.LOSS_HUBER, float(np.sqrt(CHI2)))
    g = lctx.ba_pose_rounds(last["xw"][v], luv[v], K6[:4], rt_in.astype(np.float64), info=w,
                            opt=capi.ba_options(max_num_iterations=10))
    assert np.array_equal(rt, g[0].astype(np.float32))
    assert n_in == g[3] and np.array_equal(outl[v].astype(bool), ~g[1]) and not outl[~v].any()
    assert (~g[1][moved[v]]).mean() >= 0.99 and (~g[1][~moved[v]]).mean() <= 0.02
    # SearchByProjection with that frame as Last: the flagged points take no part
    lv = dict(last, valid=(v & ~outl.astype(bool)).astype(np.uint8), tcw_last=tcw_last)
    o = ref.search_proj_frame(cur, lv, 15.0)
    assert n_m.value == o["n_matches"] > 200
    exp = o["state_for_kp"].copy()
    exp[exp == -1] = -2
    assert np.array_equal(state, exp)
    assert not np.isin(state[state >= 0], np.flatnonzero(outl)).any()
