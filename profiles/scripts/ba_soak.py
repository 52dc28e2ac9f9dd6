"""Soak: lorb_ba_local on random windows of every solver path (dense <= 10 cameras, privatised
11..16, work lists > 16) against the fp64 oracle (rtol 1e-6), with fixed observers and varied
observation counts per point.

LORB_SOAK_LOSS=huber|softlone|cauchy (opt-in; default: plain least squares) runs every solve under
that robust loss (scale LORB_SOAK_LOSS_SCALE, default 2 px) on inputs with 10 % gross outliers."""
import os
import sys

import numpy as np

sys.path.insert(0, ".")
from lorb_slam_b200 import capi, synth  # noqa: E402
from oracle import ref  # noqa: E402

LOSS_NAME = os.environ.get("LORB_SOAK_LOSS", "")
LOSS = None
if LOSS_NAME:
    sys.path.insert(0, "tests")
    import robust_cases  # noqa: E402
    import robust_ref  # noqa: E402
    LOSS = (robust_cases.LOSSES[LOSS_NAME], float(os.environ.get("LORB_SOAK_LOSS_SCALE", 2.0)))
    _orng = np.random.default_rng(5)  # outliers from a stream of their own: the problem draws stay as they are


def oracle_local(pb, opt):
    return ref.ba_local(pb, opt) if LOSS is None else robust_ref.ba_local(pb, opt, loss=LOSS)


def oracle_pose(po, opt):
    args = (po["xw"], po["uv"], po["K"], po["rt"], opt)
    return ref.ba_pose_only(*args) if LOSS is None else robust_ref.ba_pose_only(*args, loss=LOSS)


def outliers(d, key):
    """With a robust loss: move 10 % of d[key] (pixels) by 20-80 px."""
    if LOSS is not None and len(d[key]):
        d[key] = robust_cases._move(d[key], _orng, 0.1)
    return d

n = int(sys.argv[1]) if len(sys.argv) > 1 else 40
rng = np.random.default_rng(int(os.environ.get("LORB_SOAK_SEED", 77)))
bad = soft = 0
with capi.Context(0) as ctx:
    if LOSS is not None:
        ctx.ba_set_loss(*LOSS)
        print("robust loss", LOSS_NAME, LOSS[1])
    for s in range(n):
        C = int(rng.choice([2, 3, 5, 8, 10, 11, 14, 16, 17, 24, 40]))
        P = int(rng.integers(30, 600))
        k = tuple(int(v) for v in rng.choice(np.arange(2, min(C, 12) + 1), size=3))
        ff = float(rng.choice([0.0, 0.0, 0.1, 0.3]))
        pb = synth.make_ba_problem(900 + s, C=C, P=P, obs_per_point=k, fixed_frac=ff, traj_len=float(max(3.0, C * 0.4)))
        outliers(outliers(pb, "obs_uv"), "fix_uv")
        it = int(rng.choice([3, 6, 50]))
        kw = dict(max_num_iterations=it)
        try:
            cams, pts, sm = ctx.ba_local(pb, capi.ba_options(**kw))
            oc, op, so = oracle_local(pb, ref.ba_options(**kw))
            np.testing.assert_allclose(cams, oc, rtol=1e-6, atol=1e-8)
            np.testing.assert_allclose(pts, op, rtol=1e-6, atol=1e-8)
            assert sm["iterations"] == so["iterations"] and sm["termination"] == so["termination"]
        except Exception as e:  # noqa: BLE001
            # an under-determined window (two cameras, two observations per point, no fixed observer)
            # is ill-conditioned: measure the oracle against itself on an input moved by 1e-15 relative
            pb2 = dict(pb, pts=pb["pts"] * (1.0 + 1e-15))
            oc2, op2, _ = oracle_local(pb2, ref.ba_options(**kw))
            sens = max(np.abs(oc2 - oc).max(), np.abs(op2 - op).max())
            diff = max(np.abs(cams - oc).max(), np.abs(pts - op).max())
            if diff <= 10.0 * sens and sm["termination"] == so["termination"]:
                soft += 1
                print("ill-conditioned", s, C, P, k, ff, it, "gpu-oracle %.3g, oracle self-sensitivity %.3g" % (diff, sens))
            else:
                bad += 1
                print("MISMATCH", s, C, P, k, ff, it, str(e)[:200].replace("\n", " "))
    # pose-only BA (BA::ProjectPoseOptimization): observation counts from the minimum up, good and bad starts
    bad_p = noise_p = 0
    for s in range(n):
        m = int(rng.choice([3, 4, 6, 10, 50, 300, 2000, 5000]))
        po = synth.make_pose_only(4000 + s, m, pixel_noise=float(rng.choice([0.0, 1.0, 3.0])),
                                  pose_noise=(float(rng.choice([0.0, 0.02, 0.3])), float(rng.choice([0.0, 0.1, 1.0]))))
        outliers(po, "uv")
        it = int(rng.choice([1, 5, 50]))
        rt, sm = ctx.ba_pose_only(po["xw"], po["uv"], po["K"], po["rt"], capi.ba_options(max_num_iterations=it))
        ort, so = oracle_pose(po, ref.ba_options(max_num_iterations=it))
        same_x = np.allclose(rt, ort, rtol=1e-6, atol=1e-8)
        if same_x and so["final_cost"] < 1e-18 and sm["iterations"] != so["iterations"]:
            # exactly determined (3 observations, no noise): the cost reaches rounding noise and the
            # tolerance tests of the last iterations fire on it -- same pose, iteration counts may differ
            noise_p += 1
        elif not (same_x and sm["iterations"] == so["iterations"] and sm["termination"] == so["termination"]):
            bad_p += 1
            print("POSE MISMATCH", s, m, it, np.abs(rt - ort).max(), sm["iterations"], so["iterations"])
    print("%d pose-only solves, %d differ (%d more: same pose, zero-cost problem stopping one iteration apart)" % (n, bad_p, noise_p))
    # heterogeneous batches: windows of different solver paths (dense / privatised / work lists) in
    # one lorb_ba_local_batched call, every window against the oracle's single-window solve
    nb = bad_b = 0
    for s in range(n // 4):
        nwin = int(rng.integers(2, 9))
        pbs = []
        for w in range(nwin):
            C = int(rng.choice([3, 5, 8, 10, 10, 11, 14, 16, 17, 24]))
            k = tuple(int(v) for v in rng.choice(np.arange(3, min(C, 10) + 1), size=3))
            pbs.append(synth.make_ba_problem(5000 + 16 * s + w, C=C, P=int(rng.integers(30, 400)), obs_per_point=k,
                                             fixed_frac=float(rng.choice([0.0, 0.0, 0.15])), traj_len=float(max(3.0, C * 0.4))))
            outliers(outliers(pbs[-1], "obs_uv"), "fix_uv")
        it = int(rng.choice([3, 6, 20]))
        kw = dict(max_num_iterations=it)
        bt = synth.batch_windows(pbs)
        cams, pts, sums = ctx.ba_local_batched(bt, capi.ba_options(**kw))
        for w, pb in enumerate(pbs):
            nb += 1
            oc, op, so = oracle_local(pb, ref.ba_options(**kw))
            gc = cams[bt["cam_off"][w]:bt["cam_off"][w + 1]]
            gp = pts[bt["pt_off"][w]:bt["pt_off"][w + 1]]
            ok = (np.allclose(gc, oc, rtol=1e-6, atol=1e-8) and np.allclose(gp, op, rtol=1e-6, atol=1e-8)
                  and sums[w]["iterations"] == so["iterations"] and sums[w]["termination"] == so["termination"])
            if not ok and LOSS is not None:
                # as for single windows: a window whose oracle moves as much under a 1e-15 input change
                pb2 = dict(pb, pts=pb["pts"] * (1.0 + 1e-15))
                oc2, op2, _ = oracle_local(pb2, ref.ba_options(**kw))
                sens = max(np.abs(oc2 - oc).max(), np.abs(op2 - op).max())
                diff = max(np.abs(gc - oc).max(), np.abs(gp - op).max())
                if diff <= 10.0 * sens and sums[w]["termination"] == so["termination"]:
                    soft += 1
                    print("ill-conditioned batch window", s, w, "gpu-oracle %.3g, oracle self-sensitivity %.3g" % (diff, sens))
                    continue
            if not ok:
                bad_b += 1
                print("BATCH MISMATCH", s, w, [q["C"] for q in pbs], it, np.abs(gc - oc).max(), np.abs(gp - op).max(),
                      sums[w]["iterations"], so["iterations"])
    print("%d batched windows in %d heterogeneous batches, %d differ" % (nb, n // 4, bad_b))
print("%d windows, %d differ, %d more within 10x the oracle's own sensitivity to a 1e-15 input change" % (n, bad, soft))
