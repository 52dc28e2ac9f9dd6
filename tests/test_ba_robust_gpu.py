"""GPU parity of the robust losses (Huber, soft-L1, Cauchy; lorb_ba_set_loss) on every BA solver
path against the fp64 oracle, with the bar of the plain solves: cameras, points and poses within
1e-6 relative and the same LM trajectory (iterations, steps, termination, costs)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_ext as rr
import robust_cases as rc
from lorb_slam_b200 import capi, synth
from oracle import ref

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RTOL, ATOL = 1e-6, 1e-8
NAMES = sorted(rc.LOSSES)


@pytest.fixture
def lctx(ctx):
    """The session ctx, put back to the trivial loss afterwards."""
    yield ctx
    ctx.ba_set_loss(capi.LOSS_TRIVIAL)


def _close(a, b, what):
    np.testing.assert_allclose(a, b, rtol=RTOL, atol=ATOL, err_msg=what)


def _same_summary(s, o):
    for k in ("iterations", "num_successful_steps", "num_unsuccessful_steps", "termination"):
        assert s[k] == o[k], (k, s, o)
    np.testing.assert_allclose(s["initial_cost"], o["initial_cost"], rtol=1e-10)
    np.testing.assert_allclose(s["final_cost"], o["final_cost"], rtol=1e-8)
    np.testing.assert_allclose(s["final_radius"], o["final_radius"], rtol=1e-5)


def _loss(name):
    return rc.LOSSES[name], rc.SCALE


def _run_pose(ctx, po, name, **kw):
    ctx.ba_set_loss(*_loss(name))
    rt, s = ctx.ba_pose_only(po["xw"], po["uv"], po["K"], po["rt"], capi.ba_options(**kw))
    ort, o = rr.ba_pose_only(po["xw"], po["uv"], po["K"], po["rt"], ref.ba_options(**kw), loss=_loss(name))
    _close(rt, ort, "pose")
    _same_summary(s, o)
    return rt, s


def _run_local(ctx, pb, name, **kw):
    ctx.ba_set_loss(*_loss(name))
    cams, pts, s = ctx.ba_local(pb, capi.ba_options(**kw))
    oc, op, o = rr.ba_local(pb, ref.ba_options(**kw), loss=_loss(name))
    _close(cams, oc, "cameras")
    _close(pts, op, "points")
    _same_summary(s, o)
    return s


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("n", [6, 500, 2000])
def test_pose_only(lctx, name, n):
    for seed in range(2):
        _, s = _run_pose(lctx, rc.pose_only(seed, n), name)
        assert s["final_cost"] < s["initial_cost"]


@pytest.mark.parametrize("name", NAMES)
def test_pose_only_hard_start(lctx, name):
    _run_pose(lctx, rc.pose_only(5, 300, pose_noise=(0.4, 1.5)), name, max_num_iterations=30)


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("case", ["cfg3_dense", "ragged", "fixed_observers", "privatised", "blocked_cholesky",
                                  "large"])
def test_local(lctx, name, case):
    # Fixed observers in every window but config 3: with 10 % outliers down-weighted, a window with a free
    # gauge and points seen twice is so ill-conditioned that the oracle itself moves by more than the
    # 1e-6 bar when its input moves by 1e-15.
    if case == "cfg3_dense":  # BASELINE config 3: the DMMA dense build
        pb = rc.local(0, C=10, P=5000)
        s = _run_local(lctx, pb, name, max_num_iterations=10)
        assert s["final_cost"] < s["initial_cost"]
    elif case == "ragged":    # 3..20 observations per point, 24 cameras
        _run_local(lctx, rc.local(3, C=24, P=900, obs_per_point=tuple(range(3, 21)), traj_len=3.0, fixed_frac=0.1),
                   name, max_num_iterations=10)
    elif case == "fixed_observers":
        pb = rc.local(2, C=8, P=600, obs_per_point=(5, 6, 7), fixed_frac=0.15)
        assert pb["F"] > 100
        _run_local(lctx, pb, name, max_num_iterations=12)
    elif case == "privatised":  # 11..16 cameras: the shared-memory copy of the system
        _run_local(lctx, rc.local(12, C=14, P=700, obs_per_point=(3, 4, 5), traj_len=5.0, fixed_frac=0.1), name,
                   max_num_iterations=8)
    elif case == "blocked_cholesky":  # 240 x 240 reduced system
        _run_local(lctx, rc.local(7, C=40, P=3000, obs_per_point=(6, 7, 8), traj_len=12.0, fixed_frac=0.1), name,
                   max_num_iterations=8)
    else:                     # n = 6C > 96: work lists, camera rows and Schur pairs kernels
        _run_local(lctx, rc.local(13, C=20, P=1500, obs_per_point=(4, 5, 6), traj_len=6.0, fixed_frac=0.1),
                   name, max_num_iterations=8)


@pytest.mark.parametrize("name", NAMES)
def test_batched_windows_of_mixed_solver_paths(lctx, name):
    pbs = [rc.local(300 + 7 * i + C, C=C, P=120 + 30 * i, obs_per_point=(3, 4, min(C, 6)),
                    traj_len=float(max(3.0, 0.4 * C)), fixed_frac=0.1) for i, C in enumerate((10, 17, 5, 14))]
    bt = synth.batch_windows(pbs)
    lctx.ba_set_loss(*_loss(name))
    cams, pts, sums = lctx.ba_local_batched(bt, capi.ba_options(max_num_iterations=8))
    for i, pb in enumerate(pbs):
        oc, op, o = rr.ba_local(pb, ref.ba_options(max_num_iterations=8), loss=_loss(name))
        _close(cams[bt["cam_off"][i]:bt["cam_off"][i + 1]], oc, f"cameras of window {i}")
        _close(pts[bt["pt_off"][i]:bt["pt_off"][i + 1]], op, f"points of window {i}")
        _same_summary(sums[i], o)


def test_batched_dense_windows_against_batched_oracle(lctx):
    bt = rc.batched([400 + i for i in range(6)], C=10, P=2000)
    lctx.ba_set_loss(capi.LOSS_HUBER, rc.SCALE)
    cams, pts, sums = lctx.ba_local_batched(bt, capi.ba_options(max_num_iterations=6))
    oc, op, os_ = rr.ba_local_batched(bt["cam_off"], bt["cams"], bt["pt_off"], bt["pts"], bt["obs_off"],
                                       bt["obs_cam"], bt["obs_pt"], bt["obs_uv"], bt["K"],
                                       ref.ba_options(max_num_iterations=6), loss=(rr.LOSS_HUBER, rc.SCALE))
    _close(cams, oc, "cameras")
    _close(pts, op, "points")
    for a, b in zip(sums, os_):
        _same_summary(a, b)


def test_resident_problem_reads_the_loss_at_solve_time(lctx):
    pb = rc.local(8, C=6, P=500, fixed_frac=0.1)
    opt = capi.ba_options(max_num_iterations=6)
    prob = lctx.ba_problem(pb)  # created under the trivial loss
    try:
        for name in NAMES + ["huber"]:
            lctx.ba_set_loss(*_loss(name))
            prob.reset()
            s = prob.solve(opt)
            c, p = prob.download()
            oc, op, o = rr.ba_local(pb, ref.ba_options(max_num_iterations=6), loss=_loss(name))
            _close(c, oc, f"cameras ({name})")
            _close(p, op, f"points ({name})")
            _same_summary(s, o)
        lctx.ba_set_loss(capi.LOSS_TRIVIAL)
        prob.reset()
        s = prob.solve(opt)
        c, p = prob.download()
    finally:
        prob.close()
    oc, op, o = ref.ba_local(pb, ref.ba_options(max_num_iterations=6))
    _close(c, oc, "cameras (trivial again)")
    _same_summary(s, o)


def test_trivial_after_robust_reproduces_the_default(lctx):
    """default -> Huber -> trivial on one ctx.  The pose-only solve is one CTA in a fixed order: bit for
    bit.  The local solves accumulate with fp64 atomics, whose order varies from run to run even
    between two default solves, so they are held to the re-solve bar of test_ba_gpu (1e-9) and to the
    same LM trajectory."""
    po = rc.pose_only(9, 700)
    pb = rc.local(10, C=10, P=1500)
    pl = rc.local(11, C=20, P=800, obs_per_point=(4, 5), traj_len=6.0)

    def run():
        rt, s = lctx.ba_pose_only(po["xw"], po["uv"], po["K"], po["rt"])
        c, p, s2 = lctx.ba_local(pb, capi.ba_options(max_num_iterations=6))
        c3, p3, s3 = lctx.ba_local(pl, capi.ba_options(max_num_iterations=4))
        return [rt, c, p, c3, p3], [s, s2, s3]

    assert lctx.ba_get_loss() == (capi.LOSS_TRIVIAL, 1.0)
    a0, s0 = run()
    lctx.ba_set_loss(capi.LOSS_HUBER, 1.5)
    assert lctx.ba_get_loss() == (capi.LOSS_HUBER, 1.5)
    a1, _ = run()
    assert not np.array_equal(a0[0], a1[0])
    lctx.ba_set_loss(capi.LOSS_TRIVIAL)
    a2, s2 = run()
    assert np.array_equal(a0[0], a2[0]) and s0[0] == s2[0]
    for x, y in zip(a0[1:], a2[1:]):
        np.testing.assert_allclose(y, x, rtol=1e-9, atol=1e-12)
    for x, y in zip(s0[1:], s2[1:]):
        for k in ("iterations", "num_successful_steps", "num_unsuccessful_steps", "termination"):
            assert x[k] == y[k]


def test_invalid_loss_is_refused_and_leaves_the_ctx_unchanged(lctx):
    lctx.ba_set_loss(capi.LOSS_CAUCHY, 3.0)
    for kind, scale in ((4, 1.0), (-1, 1.0), (capi.LOSS_HUBER, 0.0), (capi.LOSS_HUBER, -2.0),
                        (capi.LOSS_SOFTLONE, float("nan")), (capi.LOSS_CAUCHY, float("inf"))):
        with pytest.raises(capi.LorbError):
            lctx.ba_set_loss(kind, scale)
        assert lctx.ba_get_loss() == (capi.LOSS_CAUCHY, 3.0)
    lctx.ba_set_loss(capi.LOSS_TRIVIAL, 0.0)  # the trivial loss has no scale to check
    assert lctx.ba_get_loss() == (capi.LOSS_TRIVIAL, 1.0)


@pytest.mark.parametrize("name", NAMES)
def test_huge_scale_matches_trivial(lctx, name):
    """a = 1e6 px, far above every residual (no outliers here): rho' differs from 1 by at most
    |r|^2 / a^2 ~ 1e-11, so the solution is the trivial one.  Pose-only to 1e-12; the local solve to
    the 1e-9 run-to-run spread of its atomic accumulation."""
    po = synth.make_pose_only(12, 500)
    pb = synth.make_ba_problem(13, C=8, P=900, fixed_frac=0.1)
    rt0, s0 = lctx.ba_pose_only(po["xw"], po["uv"], po["K"], po["rt"])
    c0, p0, t0 = lctx.ba_local(pb, capi.ba_options(max_num_iterations=6))
    lctx.ba_set_loss(rc.LOSSES[name], 1e6)
    rt1, s1 = lctx.ba_pose_only(po["xw"], po["uv"], po["K"], po["rt"])
    c1, p1, t1 = lctx.ba_local(pb, capi.ba_options(max_num_iterations=6))
    np.testing.assert_allclose(rt1, rt0, rtol=1e-12, atol=1e-12)
    # the robust cost itself is a different function: rho(s) = s (1 + O(s / a^2))
    np.testing.assert_allclose(s1["final_cost"], s0["final_cost"], rtol=1e-10)
    np.testing.assert_allclose(c1, c0, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(p1, p0, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(t1["final_cost"], t0["final_cost"], rtol=1e-9)
    assert t1["iterations"] == t0["iterations"] and t1["termination"] == t0["termination"]


def test_sharded_large_ba_huber():
    """The Huber large BA sharded over min(2, devices) ranks against the oracle."""
    import torch
    n = min(2, torch.cuda.device_count())
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n),
           "--master-addr", "127.0.0.1", "--master-port", "29617",
           os.path.join(ROOT, "tests", "multi_gpu", "sharded_ba_robust.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "SHARDED_BA_ROBUST_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
