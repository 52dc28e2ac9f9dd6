"""Inputs of the robust-loss BA tests: problems of lorb_slam_b200.synth with a share of gross
outliers (observations moved 20-80 px), as SearchByProjection mismatches put into a real solve."""
import numpy as np

from lorb_slam_b200 import synth
import oracle_ext as rr

LOSSES = {"huber": rr.LOSS_HUBER, "softlone": rr.LOSS_SOFTLONE, "cauchy": rr.LOSS_CAUCHY}
SCALE = 2.0  # pixels: the kernel's knee sits at twice the 1 px observation noise


def _move(uv, rng, frac):
    """Move `frac` of the rows of uv [n, 2] by 20-80 px in a random direction."""
    uv = np.array(uv, np.float32, copy=True)
    idx = rng.choice(len(uv), size=max(1, int(round(frac * len(uv)))), replace=False)
    ang = rng.uniform(0, 2 * np.pi, len(idx))
    mag = rng.uniform(20.0, 80.0, len(idx))
    uv[idx] += np.stack([mag * np.cos(ang), mag * np.sin(ang)], 1).astype(np.float32)
    return uv


def pose_only(seed, n, frac=0.1, **kw):
    po = synth.make_pose_only(seed, n, **kw)
    po["uv"] = _move(po["uv"], np.random.default_rng(seed + 7), frac)
    return po


def local(seed, frac=0.1, **kw):
    pb = synth.make_ba_problem(seed, **kw)
    rng = np.random.default_rng(seed + 11)
    pb["obs_uv"] = _move(pb["obs_uv"], rng, frac)
    if pb["F"]:
        pb["fix_uv"] = _move(pb["fix_uv"], rng, frac)
    return pb


def batched(seeds, frac=0.1, **kw):
    return synth.batch_windows([local(s, frac, **kw) for s in seeds])
