"""CPU side of the ORBextractor stages (SURVEY 8(f) rank 5): the restated oracle against the
compiled reference's outputs, and the pins of the arithmetic the device restates (libm sinf/cosf,
cv::fastAtan2, the umax table)."""
import ctypes as C

import numpy as np
import pytest

import orb_checks as OC
import ref_cases as RC
from lorb_slam_b200 import capi
from oracle import ref


@pytest.mark.parametrize("c", RC.ORB_DESCRIBE, ids=[c[0] for c in RC.ORB_DESCRIBE])
def test_oracle_orb_describe(c):
    OC.check_orb_describe(lambda oi, pat: ref.orb_describe(oi, pat, OC.golden()["orb/umax"]), c)


def test_fast_atan2_restatement_matches_cv2():
    g = OC.golden()
    got = np.array([ref.fast_atan2(float(y), float(x)) for y, x in zip(g["atan2/y"], g["atan2/x"])], np.float32)
    assert np.array_equal(got.view(np.uint32), g["atan2/deg"].view(np.uint32))


def test_sincosf_restatement_matches_libm():
    """Host instantiation of lorb_slam_b200/csrc/libm_sincosf.cuh == this process's libm, on every
    7th float of [0, 7] and its negative (155 M arguments; the full range was run once: 0 differ).
    The descriptor stage only uses [0, 2*pi]."""
    hi = int(np.float32(7.0).view(np.uint32))
    assert ref.sincosf_mismatches(0, hi, 7) == 0
    x = np.linspace(0, 119.9, 200001).astype(np.float32)  # the rest of the fast-reduction range
    a, b = ref.libm_sincosf(x), ref.libm_sincosf(x, restated=True)
    assert np.array_equal(a[0].view(np.uint32), b[0].view(np.uint32))
    assert np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))


def test_libm_is_not_correctly_rounded():
    """Why the restatement exists: rounding the double result is NOT what the reference gets."""
    x = np.linspace(0.001, 6.28, 200000).astype(np.float32)
    s, _ = ref.libm_sincosf(x)
    assert 0 < (s != np.sin(x.astype(np.float64)).astype(np.float32)).sum() < 0.02 * len(x)


def test_umax_table():
    umax = np.zeros(16, np.int32)
    lib = capi.load_library()
    lib.lorb_orb_umax(umax.ctypes.data_as(C.c_void_p))
    assert np.array_equal(umax, OC.golden()["orb/umax"])


def _oracle_stages(img):
    w, h, _, _ = capi_level_sizes(img.shape[1], img.shape[0])
    raw = ref.orb_pyramid(img, list(zip(w, h)))
    return dict(raw=raw, blur=[ref.gaussian7(a) for a in raw], cand=lambda lv: ref.orb_level_candidates(raw[lv]))


def capi_level_sizes(width, height, nfeatures=1000, nlevels=8):
    """lorb_orb_level_sizes is host arithmetic: callable without a GPU."""
    prm = capi.OrbParams(nfeatures, 1.2, nlevels, 20, 7)
    w, h, nf = np.zeros(nlevels, np.int32), np.zeros(nlevels, np.int32), np.zeros(nlevels, np.int32)
    sf = np.zeros(nlevels, np.float32)
    rc = capi.load_library().lorb_orb_level_sizes(C.byref(prm), width, height, w.ctypes.data_as(C.c_void_p),
                                                  h.ctypes.data_as(C.c_void_p), nf.ctypes.data_as(C.c_void_p),
                                                  sf.ctypes.data_as(C.c_void_p))
    assert rc == 0
    return w, h, nf, sf


@pytest.mark.parametrize("c", RC.ORB_EXTRACT[:3], ids=[c[0] for c in RC.ORB_EXTRACT[:3]])
def test_oracle_image_ops_match_cv2(c):
    """cv::resize / cv::GaussianBlur / cv::FAST restatements of oracle/orb_ref.cpp == cv2 4.13."""
    OC.check_stages_against_cv2(_oracle_stages, c)


@pytest.mark.parametrize("c", RC.ORB_EXTRACT, ids=[c[0] for c in RC.ORB_EXTRACT])
def test_oracle_extract_matches_reference_golden(c):
    """The whole extractor assembled from the restated stages == the reference's own
    ORBextractor::operator() outputs (ext/<case>/*): the stand-in the GPU tests compare fresh frames
    with where oracle/_ref is not built."""
    OC.check_extract(lambda img, nf: OC.oracle_extract(img, nfeatures=nf), c)


@pytest.mark.parametrize("kw", [dict(nfeatures=1000, scale_factor=1.2, nlevels=8), dict(nfeatures=64, nlevels=8),
                                dict(nfeatures=3000, nlevels=6), dict(nfeatures=1000, scale_factor=1.5, nlevels=4),
                                dict(nfeatures=100, nlevels=1)], ids=["default", "n64", "n3000_l6", "sf1.5_l4", "l1"])
def test_level_plan_restatement(kw):
    """OC.level_plan (the constructor's tables, restated for the oracle extractor) == the library's
    host arithmetic, over frame sizes including odd ones."""
    for width, height in ((640, 480), (752, 480), (161, 241), (1280, 240), (1241, 376), (97, 113)):
        prm = capi.OrbParams(kw["nfeatures"], kw.get("scale_factor", 1.2), kw["nlevels"], 20, 7)
        nl = kw["nlevels"]
        w, h, nf = (np.zeros(nl, np.int32) for _ in range(3))
        sf = np.zeros(nl, np.float32)
        p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        rc = capi.load_library().lorb_orb_level_sizes(C.byref(prm), width, height, p(w), p(h), p(nf), p(sf))
        if rc != 0:
            continue  # a level smaller than the blur kernel: refused by the library, never extracted
        ow, oh, onf, osf = OC.level_plan(width, height, kw["nfeatures"], kw.get("scale_factor", 1.2), nl)
        assert (ow, oh, onf) == (list(w), list(h), list(nf)) and np.array_equal(osf, sf), (width, height)


def test_level_plan():
    w, h, nf, sf = capi_level_sizes(640, 480)
    assert list(w) == [640, 533, 444, 370, 309, 257, 214, 179] and list(h) == [480, 400, 333, 278, 231, 193, 161, 134]
    assert nf.sum() == 1000 and list(nf[:3]) == [217, 181, 151]  # mnFeaturesPerLevel of the reference run
    assert sf[0] == 1.0 and sf[1] == np.float32(1.2) and sf[2] == np.float32(1.2) * np.float32(1.2)
    prm = capi.OrbParams(1000, 1.2, 8, 20, 7)
    z = np.zeros(8, np.int32)
    p = z.ctypes.data_as(C.c_void_p)
    # levels below one 30 px cell stay in the pyramid (they yield no keypoints, as in the reference) ...
    assert capi.load_library().lorb_orb_level_sizes(C.byref(prm), 100, 100, p, p, None, None) == 0
    # ... but a level smaller than the 7 x 7 blur kernel is refused
    assert capi.load_library().lorb_orb_level_sizes(C.byref(prm), 20, 20, p, p, None, None) != 0


@pytest.mark.parametrize("c", RC.QUADTREE, ids=[c[0] for c in RC.QUADTREE])
def test_quadtree_matches_reference(c):
    """The CPU restatement of the quadtree (oracle/orb_quadtree_ref.h, the oracle of the device
    quadtree) picks exactly the keypoints the compiled reference's DistributeOctTree picks, in the
    same order."""
    args = RC.quadtree_case(c)
    g = OC.golden()
    k = "qt/" + c[0]
    assert str(g[k + "/digest"]) == RC.digest(*args)
    idx = ref.orb_distribute(*args)
    x, y, r = args[:3]
    assert np.array_equal(x[idx], g[k + "/x"]) and np.array_equal(y[idx], g[k + "/y"])
    assert np.array_equal(r[idx], g[k + "/response"])
    assert len(idx) == len(set(idx.tolist())) and len(idx) <= len(x)


def test_quadtree_fresh_vs_compiled_reference():
    from oracle import reflib
    if not reflib.available():
        pytest.skip("oracle/_ref not built")
    rng = np.random.default_rng(123)
    for _ in range(60):
        n, w, h = int(rng.integers(1, 2500)), int(rng.integers(100, 1300)), int(rng.integers(60, 700))
        if round(np.float32(w) / np.float32(h)) < 1:
            continue  # the reference divides by zero (nIni = 0)
        x = rng.integers(0, w - 6, n).astype(np.float32)
        y = rng.integers(0, h - 6, n).astype(np.float32)
        r = rng.integers(7, 60, n).astype(np.float32)
        nf = int(rng.integers(1, 1500))
        idx = ref.orb_distribute(x, y, r, 16, 16 + w, 16, 16 + h, nf)
        ox, oy, orr = reflib.distribute_octree(x, y, r, 16, 16 + w, 16, 16 + h, nf)
        assert len(idx) == len(ox) and np.array_equal(x[idx], ox) and np.array_equal(y[idx], oy)
        assert np.array_equal(r[idx], orr)
