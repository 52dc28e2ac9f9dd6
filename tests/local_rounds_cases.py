"""Inputs of the local-BA outlier-round tests: windows of lorb_slam_b200.synth with octave weights and a
share of gross outliers (robust_cases._move), and the mask of the moved observations."""
import numpy as np

import oracle_ext as rr
import robust_cases as rc
from lorb_slam_b200 import synth

SCALE_FACTOR = 1.2  # ORB pyramid
HUBER = (rr.LOSS_HUBER, float(np.sqrt(5.991)))  # ORB-SLAM2's kernel: Huber at sqrt(chi2)
CONV_GRADIENT = 2


def octave_weights(n, seed):
    """w = 1 / sigma^2 of a random ORB octave 0..7 (KeyFrame::mvInvLevelSigma2)."""
    oct_ = np.random.default_rng(seed).integers(0, 8, n)
    return (1.0 / (SCALE_FACTOR ** oct_) ** 2).astype(np.float32)


def planted(seed, frac, **kw):
    """rc.local(seed, frac, **kw), its octave weights (in-window, fixed) and the masks of the moved
    observations (in-window, fixed)."""
    clean = synth.make_ba_problem(seed, **kw)
    pb = rc.local(seed, frac, **kw)
    bad = np.any(pb["obs_uv"] != clean["obs_uv"], axis=1)
    fbad = np.any(pb["fix_uv"] != clean["fix_uv"], axis=1) if pb["F"] else np.zeros(0, bool)
    return pb, octave_weights(len(pb["obs_cam"]), seed + 3), octave_weights(pb["F"], seed + 4), bad, fbad


def behind_camera(pb, p0):
    """pb with point p0 mirrored through the centre of its first in-window observer: its depth there turns
    negative while its projection, hence its residual, stays the same.  -> (pb, index of that observation)."""
    pb = dict(pb)
    i = int(np.flatnonzero(pb["obs_pt"] == p0)[0])
    c = pb["cams"][pb["obs_cam"][i]]
    R = synth.rodrigues(c[None, :3])[0]
    centre = -R.T @ c[3:]
    pts = pb["pts"].copy()
    pts[p0] = 2 * centre - pts[p0]
    pb["pts"] = pts
    return pb, i
