"""GPU: local BA with outlier rounds (lorb_ba_local_rounds_batched) against the round reference of
tests/oracle_ext.py on every build path, under all four losses, with and without weights and with
fixed observers: cameras and points within 1e-6, the same LM bookkeeping in every round, the same flags
and counts, chi^2 within 1e-6.  Also: mixed batches, parameters without inliers, the single-round limit,
a later lorb_ba_local on the same ctx, and refusals."""
import ctypes as C

import numpy as np
import pytest

import local_rounds_cases as lc
import oracle_ext as lr
import robust_cases as rc
from lorb_slam_b200 import capi, synth
from oracle import ref

pytestmark = pytest.mark.gpu
RTOL, ATOL = 1e-6, 1e-8
LOSSES = {"trivial": None, **{k: (v, rc.SCALE) for k, v in rc.LOSSES.items()}}


@pytest.fixture
def lctx(ctx):
    """The session ctx, put back to the trivial loss afterwards."""
    yield ctx
    ctx.ba_set_loss(capi.LOSS_TRIVIAL)


def _set_loss(ctx, loss):
    if loss is None:
        ctx.ba_set_loss(capi.LOSS_TRIVIAL)
    else:
        ctx.ba_set_loss(*loss)


def _same_summary(s, o):
    for k in ("iterations", "num_successful_steps", "num_unsuccessful_steps", "termination"):
        assert s[k] == o[k], (k, s, o)
    np.testing.assert_allclose(s["initial_cost"], o["initial_cost"], rtol=1e-10, atol=1e-300)
    np.testing.assert_allclose(s["final_cost"], o["final_cost"], rtol=1e-8, atol=1e-300)
    np.testing.assert_allclose(s["final_radius"], o["final_radius"], rtol=1e-5)


def _same_rounds(got, want, chi2, what=""):
    """got / want: (cams, pts, inl, chi2, finl, fchi2, n_in, sums) of one window."""
    np.testing.assert_allclose(got[0], want[0], rtol=RTOL, atol=ATOL, err_msg="cameras " + what)
    np.testing.assert_allclose(got[1], want[1], rtol=RTOL, atol=ATOL, err_msg="points " + what)
    for g, o in zip(got[7], want[7]):
        _same_summary(g, o)
    for k in (3, 5):  # a flag cannot flip on rounding: no reference chi^2 sits at the threshold
        assert not np.any(np.abs(want[k] - chi2) <= 1e-6 * chi2), "chi2 at the threshold " + what
        np.testing.assert_allclose(got[k], want[k], rtol=1e-6, atol=1e-9, err_msg="chi2 " + what)
    assert np.array_equal(got[2], want[2]) and np.array_equal(got[4], want[4]), "flags " + what
    assert int(got[6]) == want[6], "count " + what


def _weights(pb, weighted, seed):
    if not weighted:
        return None, None
    return lc.octave_weights(len(pb["obs_cam"]), seed), lc.octave_weights(pb["F"], seed + 1)


def _with_duplicate(pb):
    """pb with one (point, camera) pair observed twice (the second pixel 0.7 px off)."""
    pb = dict(pb)
    i = 0
    pb["obs_cam"] = np.insert(pb["obs_cam"], i + 1, pb["obs_cam"][i])
    pb["obs_pt"] = np.insert(pb["obs_pt"], i + 1, pb["obs_pt"][i])
    pb["obs_uv"] = np.insert(pb["obs_uv"], i + 1, pb["obs_uv"][i] + np.float32(0.7), axis=0)
    return pb


CASES = {
    "dense": lambda: rc.local(2, C=8, P=600, obs_per_point=(5, 6, 7), fixed_frac=0.15),
    "privatised_duplicate": lambda: _with_duplicate(rc.local(4, C=8, P=500, obs_per_point=(5, 6, 7),
                                                             fixed_frac=0.15)),
    "privatised": lambda: rc.local(12, C=14, P=700, obs_per_point=(3, 4, 5), traj_len=5.0, fixed_frac=0.1),
    "work_lists": lambda: rc.local(13, C=24, P=1500, obs_per_point=(4, 5, 6), traj_len=6.0, fixed_frac=0.1),
}


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("name", sorted(LOSSES))
@pytest.mark.parametrize("case", sorted(CASES))
def test_parity_with_the_reference(lctx, case, name, weighted):
    pb = CASES[case]()
    w, fw = _weights(pb, weighted, 17)
    loss = LOSSES[name]
    _set_loss(lctx, loss)
    got = lctx.ba_local_rounds(pb, w, fw)
    want = lr.ba_local_rounds(pb, w, fw, loss=loss)
    _same_rounds(got, want, 5.991, case)
    assert 0 < got[6] < len(pb["obs_cam"]) + pb["F"]


@pytest.mark.parametrize("name", sorted(LOSSES))
def test_mixed_batch_equals_the_reference_window_by_window(lctx, name):
    # One window with 17 cameras puts the whole batch on the work-list path.  Under plain least squares the
    # windows carry no planted mismatches: a first round without a robust loss, dragged by 10 % gross
    # outliers, leaves points of these small windows with at most one inlier, whose 3x3 blocks are singular
    # up to the LM damping, and such a solve is not reproducible to 1e-6 by any second implementation.
    frac = 0.1 if LOSSES[name] else 0.0
    pbs = [rc.local(300 + 7 * i + C, frac, C=C, P=200 + 30 * i, obs_per_point=(4, 5, min(C, 6)),
                    traj_len=float(max(3.0, 0.4 * C)), fixed_frac=0.15) for i, C in enumerate((10, 17, 5, 14))]
    bt = synth.batch_windows(pbs)
    ws = [_weights(pb, True, 40 + i) for i, pb in enumerate(pbs)]
    w, fw = np.concatenate([x[0] for x in ws]), np.concatenate([x[1] for x in ws])
    loss = LOSSES[name]
    _set_loss(lctx, loss)
    cams, pts, inl, chi2, finl, fchi2, n_in, sums = lctx.ba_local_rounds_batched(bt, w, fw)
    for i, pb in enumerate(pbs):
        c0, c1 = bt["cam_off"][i:i + 2]
        p0, p1 = bt["pt_off"][i:i + 2]
        o0, o1 = bt["obs_off"][i:i + 2]
        f0, f1 = bt["fix_off"][i:i + 2]
        got = (cams[c0:c1], pts[p0:p1], inl[o0:o1], chi2[o0:o1], finl[f0:f1], fchi2[f0:f1], n_in[i], sums[i])
        _same_rounds(got, lr.ba_local_rounds(pb, ws[i][0], ws[i][1], loss=loss), 5.991, f"window {i}")


@pytest.mark.slow
def test_parity_at_config5_size(lctx):
    """A config-5-sized window (200 cameras, 20000 points) on the work-list path, Huber and octave weights."""
    pb = rc.local(5, C=200, P=20000, obs_per_point=(6,), traj_len=40.0, fixed_frac=0.1)
    w, fw = _weights(pb, True, 23)
    lctx.ba_set_loss(*lc.HUBER)
    got = lctx.ba_local_rounds(pb, w, fw)
    want = lr.ba_local_rounds(pb, w, fw, loss=lc.HUBER)
    _same_rounds(got, want, 5.991, "config 5")


def test_parameters_without_inliers_keep_their_bits(lctx):
    pb = rc.local(21, 0.0, C=6, P=300, obs_per_point=(4, 5), fixed_frac=0.1)
    p0 = 11
    # every observation of p0 a gross mismatch, moved 300 px one way or the other: no position of the point
    # fits any of them
    uv, fuv = pb["obs_uv"].copy(), pb["fix_uv"].copy()
    io, jf = np.flatnonzero(pb["obs_pt"] == p0), np.flatnonzero(pb["fix_pt"] == p0)
    sign = np.where(np.arange(len(io) + len(jf)) % 2 == 0, 1.0, -1.0).astype(np.float32)[:, None]
    uv[io] += np.float32(300.0) * sign[:len(io)]
    fuv[jf] += np.float32(300.0) * sign[len(io):]
    pb = dict(pb, obs_uv=uv, fix_uv=fuv)
    lctx.ba_set_loss(*lc.HUBER)
    # round 0 takes no step, so its classification is that of the input: p0 enters round 1 without inliers
    # and with its input bits (two calls are not compared: fp64 atomic sums differ in the last bits)
    opt = [capi.ba_options(max_num_iterations=0), capi.ba_options(max_num_iterations=10)]
    cams, pts, inl, _, finl, _, _, sums = lctx.ba_local_rounds(pb, rounds=capi.local_rounds_options(chi2=1e4),
                                                               opt=opt)
    assert not inl[pb["obs_pt"] == p0].any() and not finl[pb["fix_pt"] == p0].any()
    assert sums[0]["iterations"] == 0 and sums[1]["num_successful_steps"] > 0
    assert np.array_equal(pts[p0], pb["pts"][p0])
    others = np.arange(len(pts)) != p0
    assert not np.any(np.all(pts[others] == pb["pts"][others], axis=1)) and not np.any(cams == pb["cams"])


@pytest.mark.parametrize("name", sorted(LOSSES))
def test_one_round_with_unit_weights_is_lorb_ba_local(lctx, name):
    pb = CASES["dense"]()
    _set_loss(lctx, LOSSES[name])
    opt = capi.ba_options(max_num_iterations=10)
    cams, pts, s = lctx.ba_local(pb, opt)
    O, F = len(pb["obs_cam"]), pb["F"]
    got = lctx.ba_local_rounds(pb, np.ones(O, np.float32), np.ones(F, np.float32),
                               rounds=capi.local_rounds_options(n_rounds=1, chi2=1e30), opt=[opt])
    np.testing.assert_allclose(got[0], cams, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(got[1], pts, rtol=RTOL, atol=ATOL)
    _same_summary(got[7][0], s)
    assert got[2].all() and got[4].all() and got[6] == O + F


def test_a_later_lorb_ba_local_sees_no_round_state(lctx):
    """lorb_ba_local after rounds calls on the same ctx gives what a fresh ctx gives."""
    pb = CASES["work_lists"]()
    pb_small = CASES["dense"]()
    lctx.ba_set_loss(*lc.HUBER)
    w, fw = _weights(pb_small, True, 5)
    lctx.ba_local_rounds(pb_small, w, fw)
    lctx.ba_local_rounds(pb, *_weights(pb, True, 6))
    after = [lctx.ba_local(p, capi.ba_options(max_num_iterations=8)) for p in (pb, pb_small)]
    fresh = capi.Context(0)
    try:
        fresh.ba_set_loss(*lc.HUBER)
        clean = [fresh.ba_local(p, capi.ba_options(max_num_iterations=8)) for p in (pb, pb_small)]
    finally:
        fresh.close()
    for a, b in zip(after, clean):  # fp64 atomic sums: equal to the parity bar, not to the last bit
        np.testing.assert_allclose(a[0], b[0], rtol=RTOL, atol=ATOL)
        np.testing.assert_allclose(a[1], b[1], rtol=RTOL, atol=ATOL)
        _same_summary(a[2], b[2])


def test_invalid_arguments_are_refused_with_outputs_untouched(lctx):
    lib = capi.load_library()
    pb = rc.local(8, C=4, P=60, obs_per_point=(3,), fixed_frac=0.2)
    O, F = len(pb["obs_cam"]), pb["F"]
    K = np.ascontiguousarray(pb["K"], np.float32)
    oc, op = np.ascontiguousarray(pb["obs_cam"], np.int32), np.ascontiguousarray(pb["obs_pt"], np.int32)
    ouv, fp = np.ascontiguousarray(pb["obs_uv"], np.float32), np.ascontiguousarray(pb["fix_pt"], np.int32)
    fuv, frt = np.ascontiguousarray(pb["fix_uv"], np.float32), np.ascontiguousarray(pb["fix_rt"], np.float32)
    good_w = np.ones(O, np.float32)

    def call(rounds=None, opt="default", w=good_w, obs_cam=oc, inl_null=False):
        cams, pts = pb["cams"].copy(), pb["pts"].copy()
        inl, chi2 = np.full(O, 7, np.uint8), np.full(O, -1.0)
        finl, n_in = np.full(F, 7, np.uint8), np.full(1, -5, np.int32)
        rounds = rounds or capi.local_rounds_options()
        opts = capi._round_opts(rounds, None) if opt == "default" else None
        rc_ = lib.lorb_ba_local_rounds_single(
            lctx._h, len(cams), capi._ptr(cams), len(pts), capi._ptr(pts), O, capi._ptr(obs_cam), capi._ptr(op),
            capi._ptr(ouv), capi._ptr(w), F, capi._ptr(fp), capi._ptr(fuv), capi._ptr(frt), None, capi._ptr(K),
            C.byref(rounds), opts, None if inl_null else capi._ptr(inl), capi._ptr(chi2), capi._ptr(finl), None,
            capi._ptr(n_in), None)
        untouched = (np.array_equal(cams, pb["cams"]) and np.array_equal(pts, pb["pts"]) and (inl == 7).all()
                     and (chi2 == -1.0).all() and (finl == 7).all() and n_in[0] == -5)
        return rc_, untouched

    assert call() == (capi.OK, False)  # the valid call writes its outputs
    bad_cam = oc.copy()
    bad_cam[3] = 4
    for kw in (dict(rounds=capi.local_rounds_options(n_rounds=0)), dict(rounds=capi.local_rounds_options(n_rounds=17)),
               dict(rounds=capi.local_rounds_options(robust_rounds=3)),
               dict(rounds=capi.local_rounds_options(robust_rounds=-1)),
               dict(rounds=capi.local_rounds_options(chi2=0.0)), dict(rounds=capi.local_rounds_options(chi2=np.nan)),
               dict(rounds=capi.local_rounds_options(chi2=np.inf)),
               dict(rounds=capi.local_rounds_options(depth_check=2)), dict(opt=None),
               dict(w=np.where(np.arange(O) == 5, 0.0, 1.0).astype(np.float32)),
               dict(w=np.where(np.arange(O) == 5, np.nan, 1.0).astype(np.float32)),
               dict(w=np.where(np.arange(O) == 5, -1.0, 1.0).astype(np.float32)),
               dict(inl_null=True), dict(obs_cam=bad_cam)):
        assert call(**kw) == (-1, True), kw
    # no windows: a no-op
    r0 = capi.local_rounds_options()
    assert lib.lorb_ba_local_rounds_batched(lctx._h, 0, *([None] * 14), capi._ptr(K), C.byref(r0),
                                            capi._round_opts(r0, None), *([None] * 7)) == capi.OK
