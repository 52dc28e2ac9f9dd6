"""GPU parity of the ORBextractor stages (SURVEY 8(f) rank 5) through the C ABI: bit-exact against
the compiled reference's outputs (tests/golden/orb_golden.npz) and against the oracle on fresh
inputs; the device's sinf/cosf/fastAtan2 against the host's."""
import numpy as np
import pytest

import orb_checks as OC
import ref_cases as RC
from lorb_slam_b200 import capi, synth
from oracle import ref

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("c", RC.ORB_DESCRIBE, ids=[c[0] for c in RC.ORB_DESCRIBE])
def test_cuda_orb_describe_golden(ctx, c):
    OC.check_orb_describe(ctx.orb_describe, c)


@pytest.mark.parametrize("seed", range(4))
def test_cuda_orb_describe_fresh(ctx, seed):
    g = OC.golden()
    oi = synth.make_orb_inputs(4000 + 500 * seed, 100 + seed, width=752 if seed % 2 else 640)
    a, d = ctx.orb_describe(oi, OC.pattern())
    oa, od = ref.orb_describe(oi, OC.pattern(), g["orb/umax"])
    assert np.array_equal(a.view(np.uint32), oa.view(np.uint32)) and np.array_equal(d, od)
    # describing with given angles (computeDescriptors after computeOrientation) is the same thing
    _, d2 = ctx.orb_describe(oi, OC.pattern(), angle_in=oa)
    assert np.array_equal(d2, od)


def test_cuda_orb_describe_edges(ctx):
    oi = synth.make_orb_inputs(0, 5)
    a, d = ctx.orb_describe(oi, OC.pattern())
    assert a.shape == (0,) and d.shape == (0, 32)
    oi = synth.make_orb_inputs(10, 6)
    oi["kx"][3] = 5.0  # closer than EDGE_THRESHOLD to the border
    with pytest.raises(capi.LorbError):
        ctx.orb_describe(oi, OC.pattern())
    # keypoints exactly on the EDGE_THRESHOLD ring of every level: the patch touches the border
    oi = synth.make_orb_inputs(64, 7)
    w = np.array([oi["pyr_raw"][l].shape[1] for l in oi["klevel"]])
    h = np.array([oi["pyr_raw"][l].shape[0] for l in oi["klevel"]])
    oi["kx"] = np.where(np.arange(64) % 2 == 0, 19, w - 20).astype(np.float32)
    oi["ky"] = np.where(np.arange(64) % 4 < 2, 19, h - 20).astype(np.float32)
    a, d = ctx.orb_describe(oi, OC.pattern())
    oa, od = ref.orb_describe(oi, OC.pattern(), OC.golden()["orb/umax"])
    assert np.array_equal(a.view(np.uint32), oa.view(np.uint32)) and np.array_equal(d, od)


def test_device_sincosf_and_atan2_bits(ctx):
    rng = np.random.default_rng(3)
    # every float of [0, 2*pi] that a degree angle times factorPI can produce is a float: sample
    # 8 M of them uniformly in bit pattern plus a dense linear sweep
    hi = int(np.float32(6.3).view(np.uint32))
    x = np.concatenate([rng.integers(0, hi, 6_000_000).astype(np.uint32).view(np.float32),
                        np.linspace(0, 6.3, 2_000_000).astype(np.float32),
                        -np.linspace(0, 100.0, 100_000).astype(np.float32)])
    y = rng.integers(-2700000, 2700000, len(x)).astype(np.float32)
    s, c, _ = ctx.orb_selftest(x, y)
    hs, hc = ref.libm_sincosf(x)
    assert np.array_equal(s.view(np.uint32), hs.view(np.uint32))
    assert np.array_equal(c.view(np.uint32), hc.view(np.uint32))
    g = OC.golden()
    _, _, t = ctx.orb_selftest(g["atan2/y"], g["atan2/x"])
    assert np.array_equal(t.view(np.uint32), g["atan2/deg"].view(np.uint32))


def _cuda_stages(ctx):
    def run(img):
        st = ctx.orb_stages(img)
        ls = st["level_start"]
        return dict(raw=st["raw"], blur=st["blur"],
                    cand=lambda lv: (st["cand_x"][ls[lv]:ls[lv + 1]], st["cand_y"][ls[lv]:ls[lv + 1]],
                                     st["cand_response"][ls[lv]:ls[lv + 1]]))
    return run


@pytest.mark.parametrize("c", RC.ORB_EXTRACT[:3], ids=[c[0] for c in RC.ORB_EXTRACT[:3]])
def test_cuda_image_ops_match_cv2(ctx, c):
    OC.check_stages_against_cv2(_cuda_stages(ctx), c)


@pytest.mark.parametrize("c", RC.ORB_EXTRACT, ids=[c[0] for c in RC.ORB_EXTRACT])
def test_cuda_orb_extract_golden(ctx, c):
    OC.check_extract(lambda img, nf: ctx.orb_extract(img, OC.pattern(), nfeatures=nf), c)


@pytest.mark.parametrize("seed,w,h", [(10, 640, 480), (11, 1241, 376), (12, 200, 150), (13, 97, 113)])
def test_cuda_stages_fresh(ctx, seed, w, h):
    """Every level of fresh images (odd sizes, KITTI-like aspect) against the oracle restatements."""
    img = synth.make_orb_image(seed, w, h)
    nl = 8 if min(w, h) >= 300 else 3
    st = ctx.orb_stages(img, nlevels=nl)
    lw, lh, _, _ = ctx.orb_level_sizes(w, h, nlevels=nl)
    raw = ref.orb_pyramid(img, list(zip(lw, lh)))
    ls = st["level_start"]
    for lv in range(nl):
        assert np.array_equal(st["raw"][lv], raw[lv]), lv
        assert np.array_equal(st["blur"][lv], ref.gaussian7(raw[lv])), lv
        x, y, r = ref.orb_level_candidates(raw[lv])
        assert np.array_equal(st["cand_x"][ls[lv]:ls[lv + 1]], x), lv
        assert np.array_equal(st["cand_y"][ls[lv]:ls[lv + 1]], y) and np.array_equal(st["cand_response"][ls[lv]:ls[lv + 1]], r)


@pytest.mark.parametrize("seed", range(3))
def test_cuda_orb_extract_fresh_vs_reference(ctx, seed):
    """Against the compiled reference where oracle/_ref is built, else against the oracle extractor
    (pinned to the reference's outputs by test_orb_cpu)."""
    img = synth.make_orb_image(40 + seed, 640 + 16 * seed, 480)
    for nf in (1000, 150):
        a, b = ctx.orb_extract(img, OC.pattern(), nfeatures=nf), OC.reference_extract(img, nfeatures=nf)
        assert a["n"] == b["n"]
        for f in ("x", "y", "octave", "angle", "response", "size", "desc"):
            assert np.array_equal(a[f], b[f]), f


def test_cuda_orb_extract_flat_image(ctx):
    img = np.full((480, 640), 77, np.uint8)
    r = ctx.orb_extract(img, OC.pattern())
    assert r["n"] == 0
    # every level below one 30 px cell: a pyramid without keypoints, as in the reference
    assert ctx.orb_extract(synth.make_orb_image(3, 40, 40), OC.pattern())["n"] == 0
    with pytest.raises(capi.LorbError):  # the last level would be 2 x 2: smaller than the blur kernel
        ctx.orb_extract(np.zeros((8, 8), np.uint8), OC.pattern())


def test_config0_extract_then_match(ctx):
    """BASELINE config 0 (reference example/test.cpp): ORB features of a frame pair, brute-force
    Hamming match with cross-check; most matches must agree with the known warp."""
    img = synth.make_orb_image(0)
    a = ctx.orb_extract(img, OC.pattern())
    b = ctx.orb_extract(synth.warp_orb_image(img), OC.pattern())
    m = ctx.match_bf_crosscheck(a["desc"], b["desc"])
    assert m["n_kept"] > 300
    kept = m["keep"].astype(bool)
    q, t = m["q"][kept], m["t"][kept]
    ang = np.deg2rad(3.0)
    xc, yc = a["x"][q] - 320, a["y"][q] - 240
    px = 1.02 * (np.cos(ang) * xc - np.sin(ang) * yc) + 320 + 4.0
    py = 1.02 * (np.sin(ang) * xc + np.cos(ang) * yc) + 240 - 3.0
    err = np.hypot(px - b["x"][t], py - b["y"][t])
    assert np.median(err) < 3.0


@pytest.mark.parametrize("seed", range(2))
def test_stereo_frame_front_end(ctx, seed):
    """lorb_stereo_frame (Frame's stereo constructor on the device) == the separately verified
    pieces chained through host buffers, and == the compiled reference's extractor + its
    Frame::ComputeStereoMatches when oracle/_ref travelled."""
    st0 = synth.make_stereo_pair(8, 20 + seed)
    left, right = st0["pyr_left"][0], st0["pyr_right"][0]
    mbf, mb = float(st0["mbf"]), float(st0["mb"])
    L, R, ur, dp, nm = ctx.stereo_frame(left, right, OC.pattern(), mbf, mb)
    a, b = ctx.orb_extract(left, OC.pattern()), ctx.orb_extract(right, OC.pattern())
    for got, want in ((L, a), (R, b)):
        assert got["n"] == want["n"] > 500
        for f in ("x", "y", "octave", "angle", "response", "size", "desc"):
            assert np.array_equal(got[f], want[f]), f
    _, _, _, sf = ctx.orb_level_sizes(left.shape[1], left.shape[0])
    st = dict(n_levels=8, pyr_left=ctx.orb_stages(left)["raw"], pyr_right=ctx.orb_stages(right)["raw"],
              scale_factors=sf, inv_scale_factors=(np.float32(1.0) / sf).astype(np.float32), mbf=mbf, mb=mb,
              fx=float(st0["fx"]),
              n_left=a["n"], lx=a["x"], ly=a["y"], loct=a["octave"], ldesc=a["desc"],
              n_right=b["n"], rx=b["x"], ry=b["y"], roct=b["octave"], rdesc=b["desc"])
    s = ctx.stereo_matches(st)
    assert nm == s["n_matched"] and nm > 100
    assert np.array_equal(ur, s["uright"]) and np.array_equal(dp, s["depth"])
    o = ref.stereo_matches(st)
    assert nm == o["n_matched"] and np.array_equal(ur, o["uright"]) and np.array_equal(dp, o["depth"])
    from oracle import reflib
    if reflib.available():
        ra, rb = reflib.orb_extract(left), reflib.orb_extract(right)
        assert np.array_equal(ra["desc"], L["desc"]) and np.array_equal(rb["x"], R["x"])
        rs = reflib.stereo_matches(st)
        assert nm == rs["n_matched"] and np.array_equal(ur, rs["uright"]) and np.array_equal(dp, rs["depth"])


@pytest.mark.parametrize("kw", [dict(nlevels=1), dict(nlevels=4, scale_factor=1.5), dict(ini_th=40, min_th=12),
                                dict(ini_th=9, min_th=9), dict(nfeatures=64), dict(nfeatures=3000, nlevels=6)],
                         ids=["one_level", "sf1.5", "th40_12", "th9_9", "n64", "n3000_l6"])
def test_cuda_orb_extract_parameters_vs_reference(ctx, kw):
    """Non-default ORBextractor constructor arguments, and a strided (non-contiguous) input image."""
    img = synth.make_orb_image(77, 700, 500)
    view = img[6:486, 20:660]  # 640x480 window of a 700-px-wide buffer: step 700
    assert not view.flags["C_CONTIGUOUS"]
    prm = dict(nfeatures=1000, scale_factor=1.2, nlevels=8, ini_th=20, min_th=7)
    prm.update(kw)
    b = OC.reference_extract(np.ascontiguousarray(view), **prm)
    cap = prm["nfeatures"] + 64
    # the ctypes wrapper makes arrays contiguous; call the C ABI with the strided view directly
    import ctypes as C
    p = capi.OrbParams(prm["nfeatures"], prm["scale_factor"], prm["nlevels"], prm["ini_th"], prm["min_th"])
    pat = np.ascontiguousarray(OC.pattern(), np.int32).reshape(-1)
    kx, ky, ka, kr, ks = (np.zeros(cap, np.float32) for _ in range(5))
    ko, desc, n = np.zeros(cap, np.int32), np.zeros((cap, 32), np.uint8), C.c_int(0)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    rc = ctx._lib.lorb_orb_extract(ctx._h, C.c_void_p(view.ctypes.data), 640, 480, int(view.strides[0]), C.byref(p),
                                   vp(pat), cap, vp(kx), vp(ky), vp(ko), vp(ka), vp(kr), vp(ks), vp(desc), C.byref(n),
                                   None)
    assert rc == 0 and n.value == b["n"] > 0
    m = n.value
    assert np.array_equal(kx[:m], b["x"]) and np.array_equal(ky[:m], b["y"]) and np.array_equal(ko[:m], b["octave"])
    assert np.array_equal(ka[:m], b["angle"]) and np.array_equal(kr[:m], b["response"])
    assert np.array_equal(ks[:m], b["size"]) and np.array_equal(desc[:m], b["desc"])


def test_cuda_orb_extract_repeatable_and_reentrant(ctx):
    """Same frame twice, a different frame size in between (graph re-capture), a second context on
    another host thread at the same time: always the same bits."""
    import threading
    img, other = synth.make_orb_image(3), synth.make_orb_image(4, 752, 480)
    a = ctx.orb_extract(img, OC.pattern())
    ctx.orb_extract(other, OC.pattern(), nfeatures=500)
    b = ctx.orb_extract(img, OC.pattern())
    res = {}

    def worker():
        with capi.Context(0) as c2:
            for _ in range(5):
                res["t"] = c2.orb_extract(img, OC.pattern())

    t = threading.Thread(target=worker)
    t.start()
    for _ in range(5):
        c = ctx.orb_extract(img, OC.pattern())
    t.join()
    for r in (b, c, res["t"]):
        assert r["n"] == a["n"] and np.array_equal(r["desc"], a["desc"]) and np.array_equal(r["x"], a["x"])
        assert np.array_equal(r["angle"], a["angle"])


def test_device_quadtree_matches_host_quadtree(ctx):
    """orb_quadtree_gpu.cuh (one CTA, parallel rounds) == oracle/orb_quadtree_ref.h (the sequential CPU
    restatement, itself pinned to the compiled reference): golden cases + random ones incl. pixel clusters, wide
    levels whose first pass overshoots the budget, and budgets of 1."""
    g = OC.golden()
    for c in RC.QUADTREE:
        args = RC.quadtree_case(c)
        idx = ctx.orb_distribute(*args)
        x, y, r = args[:3]
        k = "qt/" + c[0]
        assert np.array_equal(x[idx], g[k + "/x"]) and np.array_equal(y[idx], g[k + "/y"])
        assert np.array_equal(idx, ref.orb_distribute(*args))
    rng = np.random.default_rng(11)
    for t in range(150):
        n, w, h = int(rng.integers(1, 3000)), int(rng.integers(100, 1300)), int(rng.integers(60, 700))
        if round(np.float32(w) / np.float32(h)) < 1:
            continue
        span = w - 6 if t % 5 else 30
        x = rng.integers(0, span, n).astype(np.float32)
        y = rng.integers(0, min(span, h - 6), n).astype(np.float32)
        r = rng.integers(7, 60, n).astype(np.float32)
        nf = int(rng.integers(1, 1500)) if t % 7 else 1
        a = ref.orb_distribute(x, y, r, 16, 16 + w, 16, 16 + h, nf)
        b = ctx.orb_distribute(x, y, r, 16, 16 + w, 16, 16 + h, nf)
        assert np.array_equal(a, b), (t, n, w, h, nf)


def test_cuda_orb_extract_soak_vs_reference(ctx):
    """A slice of profiles/scripts/orb_soak.py (300 frames there: 0 differ): varied frame sizes,
    textures (low contrast, pure noise, half flat), budgets, level counts and thresholds, each
    bit-exact against the compiled reference -- including wide frames with small budgets, which
    return more keypoints than nfeatures + a few (lorb_orb_max_keypoints).  Where oracle/_ref is not
    built, the oracle extractor stands in for the reference."""
    rng = np.random.default_rng(99)
    over = 0
    for f in range(28):
        w, h = int(rng.choice([320, 512, 752, 1024, 1280])), int(rng.choice([240, 376, 480]))
        img = synth.make_orb_image(500 + f, w, h)
        if f % 4 == 1:
            img = (128 + (img.astype(np.float32) - 128) * 0.15).astype(np.uint8)
        elif f % 4 == 2:
            img = rng.integers(0, 256, (h, w), dtype=np.uint8)
        elif f % 4 == 3:
            img = img.copy()
            img[:, : w // 2] = 100
        nf, nl = int(rng.choice([100, 500, 2000])), int(rng.choice([4, 8]))
        a = ctx.orb_extract(img, OC.pattern(), nfeatures=nf, nlevels=nl)
        b = OC.reference_extract(img, nfeatures=nf, nlevels=nl)
        assert a["n"] == b["n"] <= ctx.orb_max_keypoints(w, h, nfeatures=nf, nlevels=nl), (f, w, h, nf, nl)
        for k in ("x", "y", "octave", "angle", "response", "size", "desc"):
            assert np.array_equal(a[k], b[k]), (f, k)
        over += a["n"] > nf + 64
    # the case a fixed "nfeatures + 64" capacity misses: a wide frame with a small budget keeps 4 nodes
    # per initial quadtree column on every level
    img = synth.make_orb_image(640, 1280, 240)
    a, b = ctx.orb_extract(img, OC.pattern(), nfeatures=100), OC.reference_extract(img, nfeatures=100)
    assert a["n"] == b["n"] > 100 + 64 and np.array_equal(a["desc"], b["desc"]) and np.array_equal(a["x"], b["x"])
