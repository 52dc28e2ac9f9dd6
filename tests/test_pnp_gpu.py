"""GPU: batched P3P RANSAC (lorb_pnp_ransac_batched) against its host restatement (tests/pnp_ref.py): identical
selections, counts and flags, poses within 1e-12 and chi^2 within 1e-9 relative over mixed batches; the device
P3P on exactly representable planted poses; a problem alone equals it in a batch bit for bit; refusals; the
RANSAC -> pose-rounds chain against the reference chain; and the drop-in lorb_host::PoseFromMatches."""
import ctypes as C

import numpy as np
import pytest

import oracle_ext as rd
import pnp_ref as pr
from lorb_slam_b200 import capi, synth

pytestmark = pytest.mark.gpu
CHI2 = 5.991


@pytest.fixture
def lctx(ctx):
    """The session ctx, put back to the trivial loss afterwards."""
    yield ctx
    ctx.ba_set_loss(capi.LOSS_TRIVIAL)


def _same(g, o):
    assert np.array_equal(g[1], o[1])
    assert np.array_equal(g[2], o[2])
    assert np.array_equal(g[3], o[3])
    np.testing.assert_allclose(g[0], o[0], rtol=0, atol=1e-12)
    fin = np.isfinite(o[4])
    assert np.array_equal(np.isfinite(g[4]), fin) and np.all(g[4][~fin] == o[4][~fin])
    np.testing.assert_allclose(g[4][fin], o[4][fin], rtol=1e-9, atol=0)


def _mixed(seed, sizes, fracs):
    """One batch: problem b has sizes[b] correspondences and outlier fraction fracs[b]."""
    parts = [synth.make_pnp_problems(seed * 1000 + b, n=int(n), outlier_frac=float(f))
             for b, (n, f) in enumerate(zip(sizes, fracs))]
    cat = lambda k: np.concatenate([p[k] for p in parts])
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    return dict(corr_off=off, xw=cat("xw"), uv=cat("uv"), info=cat("info"), K=parts[0]["K"],
                rt_true=np.concatenate([p["rt_true"] for p in parts]))


@pytest.mark.parametrize("weights", [False, True])
@pytest.mark.parametrize("H", [1, 31, 32, 300, 4096])
def test_matches_reference(ctx, H, weights):
    rng = np.random.default_rng(H)
    sizes = [3, 4, 5, 50, 300, 700, 3000, 0, 300] if H < 4096 else [4, 5, 50, 300, 700]
    fracs = rng.uniform(0.0, 0.7, len(sizes))
    d = _mixed(H, sizes, fracs)
    info = d["info"] if weights else None
    seeds = rng.integers(0, 2 ** 63, len(sizes), dtype=np.uint64)
    prm = capi.pnp_ransac_params(n_hypotheses=H)
    g = ctx.pnp_ransac_batched(d["corr_off"], d["xw"], d["uv"], d["K"], info=info, seeds=seeds, params=prm)
    o = pr.ransac(d["corr_off"], d["xw"], d["uv"], d["K"], info, seeds, n_hypotheses=H)
    _same(g, o)
    assert (g[1][np.diff(d["corr_off"]) < 4] == -1).all()
    if H >= 300:
        assert (g[1][np.diff(d["corr_off"]) >= 50] >= 0).all()
    # without seeds, problem b uses seed b
    g = ctx.pnp_ransac_batched(d["corr_off"], d["xw"], d["uv"], d["K"], info=info, params=prm)
    _same(g, pr.ransac(d["corr_off"], d["xw"], d["uv"], d["K"], info, None, n_hypotheses=H))


def test_device_p3p_recovers_exact_planted_poses(ctx):
    # four correspondences, one hypothesis: the sample is the four points, so this is the device P3P itself.
    # Dyadic camera points, signed-permutation rotations and dyadic translations make xw and uv exact floats.
    # Samples with a thin triangle or keypoints closer than 32 px are left out: there the closed-form rotation
    # Y X^-1 loses digits to cancellation (up to 1.7e-8 on this generator), which is conditioning, not a fault.
    rng = np.random.default_rng(11)
    K = np.array([512.0, 256.0, 320.0, 256.0], np.float32)
    xw, uv, Ps, ts = [], [], [], []
    while len(Ps) < 2000:
        P = np.eye(3)[rng.permutation(3)] * rng.choice([-1.0, 1.0], 3)[:, None]
        if np.linalg.det(P) < 0:
            P[0] *= -1
        t = rng.integers(-64, 64, 3) / 16.0
        z = 2.0 ** rng.integers(2, 5, 4)
        xc = np.stack([rng.integers(-128, 128, 4) / 64.0 * z / 4, rng.integers(-128, 128, 4) / 64.0 * z / 4, z], 1)
        X = (xc - t) @ P
        if min(np.linalg.norm(np.cross(X[a] - X[b], X[a] - X[c])) for a, b, c in
               ((0, 1, 2), (0, 1, 3), (0, 2, 3), (1, 2, 3))) < 0.5:
            continue
        p = np.stack([K[0] * xc[:, 0] / xc[:, 2] + K[2], K[1] * xc[:, 1] / xc[:, 2] + K[3]], 1)
        if min(np.linalg.norm(p[a] - p[b]) for a in range(4) for b in range(a)) < 32.0:
            continue
        xw.append(X)
        uv.append(p)
        Ps.append(P)
        ts.append(t)
    off = np.arange(0, 4 * 2001, 4, dtype=np.int32)
    rt, best, n_in, inl, _ = ctx.pnp_ransac_batched(off, np.concatenate(xw), np.concatenate(uv), K,
                                                    params=capi.pnp_ransac_params(n_hypotheses=1))
    assert (best == 0).all() and (n_in == 4).all() and inl.all()
    R = synth.rodrigues(rt[:, :3])
    assert np.abs(R - np.array(Ps)).max() <= 1e-9
    assert np.abs(rt[:, 3:] - np.array(ts)).max() <= 1e-9


def test_batch_equals_single_problems(ctx):
    rng = np.random.default_rng(5)
    sizes = rng.choice([0, 3, 4, 20, 300, 1000], 60)
    d = _mixed(7, sizes, rng.uniform(0, 0.6, len(sizes)))
    seeds = rng.integers(0, 2 ** 63, len(sizes), dtype=np.uint64)
    B = ctx.pnp_ransac_batched(d["corr_off"], d["xw"], d["uv"], d["K"], info=d["info"], seeds=seeds)
    off = d["corr_off"]
    for b in range(len(sizes)):
        a, e = off[b], off[b + 1]
        g = ctx.pnp_ransac_batched([0, e - a], d["xw"][a:e], d["uv"][a:e], d["K"], info=d["info"][a:e],
                                   seeds=seeds[b:b + 1])
        assert np.array_equal(B[0][b], g[0][0]) and B[1][b] == g[1][0] and B[2][b] == g[2][0]
        assert np.array_equal(B[3][a:e], g[3]) and np.array_equal(B[4][a:e], g[4])


def test_invalid_arguments_are_refused_and_outputs_untouched(ctx):
    lib = capi.load_library()
    d = synth.make_pnp_problems(3, n=[20, 20])
    n = 40
    P = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
    launches = ctx.launch_count

    def call(off=d["corr_off"], w=d["info"], K=d["K"], params=None, nb=2, inl_null=False, rt_null=False):
        rt, best, n_in = np.full((2, 6), -3.0), np.full(2, -7, np.int32), np.full(2, -7, np.int32)
        inl, c2 = np.full(n, 7, np.uint8), np.full(n, -1.0)
        params = params or capi.pnp_ransac_params()
        rc_ = lib.lorb_pnp_ransac_batched(ctx._h, nb, P(off), P(d["xw"]), P(d["uv"]), P(w), P(K), None,
                                          C.byref(params), None if rt_null else P(rt), P(best), P(n_in),
                                          None if inl_null else P(inl), P(c2))
        untouched = ((rt == -3).all() and (best == -7).all() and (n_in == -7).all() and (inl == 7).all()
                     and (c2 == -1).all())
        return rc_, untouched

    assert call()[0] == 0
    launches_ok = ctx.launch_count
    assert launches_ok - launches == 2
    w = d["info"]
    bad = [dict(off=np.array([1, 20, n], np.int32)), dict(off=np.array([0, 30, 20], np.int32)), dict(nb=-1),
           dict(w=np.where(np.arange(n) == 3, 0.0, w).astype(np.float32)),
           dict(w=np.where(np.arange(n) == 3, -1.0, w).astype(np.float32)),
           dict(w=np.where(np.arange(n) == 3, np.nan, w).astype(np.float32)),
           dict(w=np.where(np.arange(n) == 3, np.inf, w).astype(np.float32)),
           dict(K=np.array([0, 458, 320, 240], np.float32)), dict(K=np.array([458, -1, 320, 240], np.float32)),
           dict(K=np.array([np.nan, 458, 320, 240], np.float32)), dict(K=np.array([458, np.inf, 320, 240], np.float32)),
           dict(params=capi.pnp_ransac_params(n_hypotheses=0)),
           dict(params=capi.pnp_ransac_params(n_hypotheses=65537)),
           dict(params=capi.pnp_ransac_params(chi2=0.0)), dict(params=capi.pnp_ransac_params(chi2=-1.0)),
           dict(params=capi.pnp_ransac_params(chi2=float("inf"))),
           dict(params=capi.pnp_ransac_params(chi2=float("nan"))),
           dict(off=None), dict(inl_null=True), dict(rt_null=True)]
    for kw in bad:
        rc_, untouched = call(**kw)
        assert rc_ == -1, kw
        assert untouched, kw
    rc_, untouched = call(nb=0)  # n_problems = 0 is a no-op
    assert rc_ == 0 and untouched
    assert ctx.launch_count == launches_ok


def _chain_inputs():
    d = synth.make_pnp_problems(31, n=600, outlier_frac=0.4)
    assert d["K"][0] == d["K"][1]  # PoseCost projects v with fx
    return d


def test_ransac_then_pose_rounds_recovers_planted_pose(lctx):
    d = _chain_inputs()
    rt, best, n_in, inl, _ = lctx.pnp_ransac_batched(d["corr_off"], d["xw"], d["uv"], d["K"], info=d["info"])
    ort, obest, on_in, oinl, _ = pr.ransac(d["corr_off"], d["xw"], d["uv"], d["K"], d["info"])
    assert best[0] == obest[0] >= 0 and np.array_equal(inl, oinl)
    xw, uv, w = d["xw"][inl], d["uv"][inl], d["info"][inl]
    g = lctx.ba_pose_rounds(xw, uv, d["K"], rt[0], info=w)
    o = rd.ba_pose_rounds(xw, uv, d["K"], ort[0], w)
    np.testing.assert_allclose(g[0], o[0], rtol=1e-6, atol=1e-6)
    assert g[3] == o[3]
    truth = d["rt_true"][0]
    R, Rt = synth.rodrigues(g[0][:3]), synth.rodrigues(truth[:3])
    # 1 px x 1.2^octave noise on ~350 inliers 3-20 m away: hundredths of a degree and a few centimetres
    assert np.degrees(np.arccos(np.clip((np.trace(R.T @ Rt) - 1) / 2, -1, 1))) < 0.05
    assert np.linalg.norm(g[0][3:] - truth[3:]) < 0.05
    R0 = synth.rodrigues(rt[0][:3])
    assert np.linalg.norm(g[0][3:] - truth[3:]) <= np.linalg.norm(rt[0][3:] - truth[3:])
    assert np.trace(R.T @ Rt) >= np.trace(R0.T @ Rt) - 1e-12


@pytest.mark.parametrize("min_inliers", [10, 100000])
def test_dropin_pose_from_matches(lctx, min_inliers):
    from lorb_slam_b200.host import build_host
    H = C.CDLL(build_host.build())
    P = lambda a: a.ctypes.data_as(C.c_void_p)
    d = _chain_inputs()
    n = len(d["xw"])
    rng = np.random.default_rng(9)
    sf = synth.scale_factors(8).astype(np.float32)
    # the octaves the generator drew: its weights are 1 / (1.2^octave)^2
    oct_ = np.rint(np.log(1.0 / d["info"].astype(np.float64)) / (2 * np.log(1.2))).astype(np.int32)
    has = (rng.random(n) < 0.9).astype(np.uint8)
    rt = np.array([0.1, -0.2, 0.3, 1.0, 2.0, 3.0], np.float32)
    rt_in = rt.copy()
    out_has, out_outl = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
    K = d["K"].astype(np.float32)
    r = H.harness_pose_from_matches(n, P(d["xw"]), P(d["uv"]), P(oct_), P(has), 8, P(sf), P(K), min_inliers, P(rt),
                                    P(out_has), P(out_outl))
    # the same chain through Python: RANSAC over the matched slots with octave weights, then PoseOptimization's
    # rounds (Huber sqrt(5.991) in rounds 0-2, 10 iterations a round) from the float RANSAC pose
    v = has.astype(bool)
    w = (np.float32(1) / (sf[oct_[v]] * sf[oct_[v]])).astype(np.float32)
    grt, gbest, gn, ginl, _ = lctx.pnp_ransac_batched([0, v.sum()], d["xw"][v], d["uv"][v], K, info=w)
    if gn[0] < min_inliers:
        assert r == gn[0]
        assert np.array_equal(rt, rt_in) and np.array_equal(out_has, has) and not out_outl.any()
        return
    lctx.ba_set_loss(capi.LOSS_HUBER, float(np.sqrt(CHI2)))
    g = lctx.ba_pose_rounds(d["xw"][v][ginl], d["uv"][v][ginl], K, grt[0].astype(np.float32).astype(np.float64),
                            info=w[ginl], opt=capi.ba_options(max_num_iterations=10))
    assert r == g[3]
    assert np.array_equal(rt, g[0].astype(np.float32))
    kept = np.flatnonzero(v)[ginl]
    exp_has = np.zeros(n, np.uint8)
    exp_has[kept] = 1
    assert np.array_equal(out_has, exp_has)
    exp_out = np.zeros(n, np.uint8)
    exp_out[kept] = ~g[1]
    assert np.array_equal(out_outl, exp_out)
    truth = d["rt_true"][0]
    assert np.linalg.norm(rt[3:] - truth[3:]) < 0.05
