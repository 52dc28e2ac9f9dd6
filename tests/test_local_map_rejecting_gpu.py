"""GPU: LocalMapIndex::OptimizeRejectingOutliers (ORB-SLAM2's LocalBundleAdjustment in the mapper's loop)
on a keyframe sequence with planted SearchByProjection-style mismatches: the planted observations are
erased (mvpMapPoints NULLed, mnObs decremented, gone from the next Assemble), and the poses end closer to
the truth than with LocalMapIndex::Optimize."""
import ctypes as C

import numpy as np
import pytest

import robust_cases as rc
from lorb_slam_b200 import synth
from lorb_slam_b200.host import build_host

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def H():
    return C.CDLL(build_host.build())


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _sequence(seed, n_kf=8, P=800, n_cov=3, frac=0.1):
    pb = synth.make_ba_problem(seed, C=n_kf, P=P, obs_per_point=(4, 5, 6))
    rng = np.random.default_rng(seed)
    clean = pb["obs_uv"]
    moved = rc._move(clean, rng, frac)
    bad = np.any(moved != clean, axis=1)
    octave = rng.integers(0, 8, len(clean)).astype(np.int32)
    slots = [[] for _ in range(n_kf)]
    for c, p, uv, o, b in zip(pb["obs_cam"], pb["obs_pt"], moved, octave, bad):
        slots[c].append((int(p), uv, int(o), bool(b)))
    for k in range(n_kf):  # a few keypoints without a map point, shuffled slot order
        slots[k] += [(-1, np.zeros(2, np.float32), 0, False)] * 5
        rng.shuffle(slots[k])
    flat = [s for x in slots for s in x]
    cov = [[j for j in range(k - 1, max(-1, k - 1 - n_cov), -1)] for k in range(n_kf)]
    return dict(
        pb=pb, n_kf=n_kf, P=P,
        kf_off=np.cumsum([0] + [len(x) for x in slots]).astype(np.int32),
        slot_pt=np.array([s[0] for s in flat], np.int32),
        slot_uv=np.array([s[1] for s in flat], np.float32),
        slot_oct=np.array([s[2] for s in flat], np.int32),
        planted=np.array([s[3] for s in flat], bool),
        cov_off=np.cumsum([0] + [len(x) for x in cov]).astype(np.int32),
        cov_idx=np.array([j for x in cov for j in x] + [0], np.int32))


def _run(H, sq, reject, first_ba=2):
    n_kf, P, S = sq["n_kf"], sq["P"], len(sq["slot_pt"])
    kf_rt = sq["pb"]["cams"].astype(np.float32)
    pts = sq["pb"]["pts"].astype(np.float32)
    cams, opts = np.zeros((n_kf, 6), np.float32), np.zeros((P, 3), np.float32)
    null, assembled, mnobs = np.zeros(S, np.uint8), np.zeros(S, np.uint8), np.zeros(P, np.int32)
    n = H.harness_local_mapping_rejecting(n_kf, _p(kf_rt), _p(sq["kf_off"]), _p(sq["slot_pt"]), _p(sq["slot_uv"]),
                                          _p(sq["slot_oct"]), _p(sq["cov_off"]), _p(sq["cov_idx"]), P, _p(pts),
                                          _p(sq["pb"]["K"]), first_ba, int(reject), _p(cams), _p(opts), _p(null),
                                          _p(assembled), _p(mnobs))
    return n, cams, opts, null.astype(bool), assembled.astype(bool), mnobs


@pytest.mark.parametrize("seed", [3, 4])
def test_rejecting_outliers_erases_planted_mismatches(H, seed):
    sq = _sequence(seed)
    n, cams, _, null, assembled, mnobs = _run(H, sq, True)
    n0, cams0, _, null0, _, mnobs0 = _run(H, sq, False)
    has = sq["slot_pt"] >= 0
    planted = sq["planted"]
    assert n0 == 0 and not null0.any()
    assert n == null.sum() > 0
    # the planted mismatches are erased.  A clean observation is judged by every local BA whose window
    # reaches it (up to four here), the first ones before the noisy initial keyframes have converged, so
    # the clean share erased is the chi-square tail compounded over those judgements
    assert null[planted].mean() >= 0.95
    assert null[has & ~planted].mean() <= 0.15
    # erased observations are gone from the map point's count and from the next Assemble
    assert not np.any(assembled & null)
    kept = np.bincount(sq["slot_pt"][has & ~null], minlength=sq["P"])
    assert np.array_equal(mnobs, kept) and np.array_equal(mnobs0, np.bincount(sq["slot_pt"][has], minlength=sq["P"]))
    # and the poses are closer to the truth than with the plain solve
    truth = sq["pb"]["cams_true"]
    err, err0 = np.linalg.norm(cams - truth), np.linalg.norm(cams0 - truth)
    assert err < err0, (err, err0)
