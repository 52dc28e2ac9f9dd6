"""GPU parity: brute-force Hamming matching through the C ABI vs the oracle,
the cv2-pinned golden vectors, and size-independent properties.
Bar: bit-exact (indices, distances, tie-break order)."""
import numpy as np
import pytest

from lorb_slam_b200 import synth
from oracle import ref

pytestmark = pytest.mark.gpu


def _same(r, o):
    assert np.array_equal(r["q"], o["q"])
    assert np.array_equal(r["t"], o["t"])
    assert np.array_equal(r["dist"], o["dist"])
    assert np.array_equal(r["keep"], o["keep"])
    assert r["n_kept"] == o["n_kept"] and r["min_dist"] == o["min_dist"]


def test_golden_cv2(ctx, golden_dir):
    g = np.load(golden_dir + "/bf_golden.npz")
    for name in g["names"]:
        r = ctx.match_bf_crosscheck(g[f"{name}_q"], g[f"{name}_t"])
        assert np.array_equal(r["q"], g[f"{name}_mq"]), name
        assert np.array_equal(r["t"], g[f"{name}_mt"]), name
        assert np.array_equal(r["dist"], g[f"{name}_md"]), name
        idx, dist, _ = ctx.match_knn2(g[f"{name}_q"], g[f"{name}_t"])
        assert np.array_equal(idx, g[f"{name}_ki"]), name
        assert np.array_equal(dist, g[f"{name}_kd"]), name


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("shape", [(1, 1), (1, 77), (77, 1), (31, 33), (128, 256), (129, 257),
                                   (1000, 1000), (1300, 2100), (2000, 2000), (300, 5000), (5000, 300)])
def test_crosscheck_vs_oracle(ctx, shape, mode):
    rng = np.random.default_rng(hash(shape) % 2**32 + mode)
    for kind in ("uniform", "tie"):
        if kind == "uniform":
            q, t = synth.descriptors_uniform(shape[0], rng), synth.descriptors_uniform(shape[1], rng)
        else:
            q = synth.descriptors_tie_stress(shape[0], rng, 2, 3)
            t = synth.descriptors_tie_stress(shape[1], rng, 2, 3)
        _same(ctx.match_bf_crosscheck(q, t, mode), ref.bf_crosscheck(q, t, mode))


def test_empty_sides(ctx):
    rng = np.random.default_rng(0)
    q = synth.descriptors_uniform(10, rng)
    e = np.zeros((0, 32), np.uint8)
    for a, b in ((q, e), (e, q), (e, e)):
        r = ctx.match_bf_crosscheck(a, b)
        assert len(r["q"]) == 0 and r["n_kept"] == 0 and r["min_dist"] == -1
    idx, dist, ok = ctx.match_knn2(q, e)
    assert (idx == -1).all() and (dist == 256).all() and not ok.any()


def test_wide_tile_path(ctx):
    """Large enough that the 4-queries-per-thread tile variant is chosen."""
    rng = np.random.default_rng(5)
    q, t = synth.descriptors_uniform(9000, rng), synth.descriptors_uniform(9000, rng)
    t[:3000] = synth.descriptors_noisy_copy(q[rng.permutation(9000)[:3000]], rng, 0.05)
    _same(ctx.match_bf_crosscheck(q, t), ref.bf_crosscheck(q, t))
    idx, dist, ok = ctx.match_knn2(q[:4500], t)
    oi, od = ref.knn2(q[:4500], t)
    assert np.array_equal(idx, oi) and np.array_equal(dist, od)


def test_knn2_ratio(ctx):
    rng = np.random.default_rng(3)
    t = synth.descriptors_uniform(700, rng)
    q = synth.descriptors_noisy_copy(t[rng.permutation(700)[:400]], rng, 0.1)
    idx, dist, ok = ctx.match_knn2(q, t, ratio=0.8, max_dist=100)
    oi, od = ref.knn2(q, t)
    assert np.array_equal(idx, oi) and np.array_equal(dist, od)
    exp = (od[:, 0] <= 100) & (od[:, 0].astype(np.float32) < np.float32(0.8) * od[:, 1].astype(np.float32))
    assert np.array_equal(ok.astype(bool), exp)
    # a low-entropy train set: best and second best are decided by the lowest-index rule
    q, t = synth.descriptors_uniform(1300, rng), synth.descriptors_tie_stress(2100, rng, 2, 3)
    idx, dist, _ = ctx.match_knn2(q, t)
    oi, od = ref.knn2(q, t)
    assert np.array_equal(idx, oi) and np.array_equal(dist, od)


def test_properties_full_size(ctx):
    """Size-independent properties at BASELINE config-5 descriptor counts."""
    rng = np.random.default_rng(11)
    a = synth.descriptors_uniform(2000, rng)
    # identical sets: every descriptor matches itself at distance 0
    r = ctx.match_bf_crosscheck(a, a.copy())
    assert np.array_equal(r["q"], np.arange(2000)) and np.array_equal(r["t"], np.arange(2000))
    assert (r["dist"] == 0).all() and r["n_kept"] == 2000 and r["min_dist"] == 0
    # permuted train set: matches follow the permutation
    perm = rng.permutation(2000)
    r = ctx.match_bf_crosscheck(a, a[perm])
    inv = np.argsort(perm)
    assert np.array_equal(r["t"], inv)
    # symmetry of mutual cross-check: swapping sides transposes the match set
    b = synth.descriptors_noisy_copy(a[rng.permutation(2000)], rng, 0.2)
    r1, r2 = ctx.match_bf_crosscheck(a, b), ctx.match_bf_crosscheck(b, a)
    s1 = set(zip(r1["q"].tolist(), r1["t"].tolist()))
    s2 = set(zip(r2["t"].tolist(), r2["q"].tolist()))
    assert s1 == s2 and r1["min_dist"] == r2["min_dist"]


@pytest.fixture(params=["popc", "tensor"])
def sweep_impl(ctx, request):
    """Both sweep kernels (XOR/POPC and tcgen05 int8) must give the oracle's numbers."""
    ctx.sweep_set_impl(request.param)
    yield request.param
    ctx.sweep_set_impl("default")


@pytest.mark.parametrize("n_desc", [1, 7, 100, 256, 257, 512, 513, 1000, 2000, 2048])
def test_sweep_vs_oracle(ctx, sweep_impl, n_desc):
    n_kf = 6
    bank = synth.kf_bank(n_kf, n_desc, seed=n_desc)
    pa, pb = synth.all_pairs(n_kf)
    # also unordered / repeated pairs and a self pair
    pa = np.concatenate([pa, [3, 5, 2]]).astype(np.int32)
    pb = np.concatenate([pb, [1, 5, 0]]).astype(np.int32)
    kept, mt, md = ctx.match_sweep(bank, pa, pb)
    ok, om, od = ref.sweep(bank, pa, pb)
    assert np.array_equal(kept, ok) and np.array_equal(mt, om) and np.array_equal(md, od)
    # per-pair equality with the single-pair entry point
    r = ctx.match_bf_crosscheck(bank[pa[1]], bank[pb[1]])
    assert r["n_kept"] == kept[1] and len(r["q"]) == mt[1] and r["min_dist"] == md[1]


@pytest.mark.parametrize("n_desc,nbytes,nvals", [(300, 1, 2), (777, 2, 4), (2000, 3, 4), (2048, 1, 3)])
def test_sweep_tie_stress(ctx, sweep_impl, n_desc, nbytes, nvals):
    """Low-entropy banks: almost every distance is tied many times over, so the three numbers
    per pair depend on the lowest-index rule of both argmins inside the sweep kernels' own
    mutual-test epilogues (VERDICT r1: only the tile kernel had seen such a bank)."""
    rng = np.random.default_rng(n_desc + nbytes)
    n_kf = 5
    bank = np.stack([synth.descriptors_tie_stress(n_desc, rng, nbytes, nvals) for _ in range(n_kf)])
    bank[3] = bank[1]  # identical keyframes: every row ties with its own copy and many others
    pa, pb = synth.all_pairs(n_kf)
    pa = np.concatenate([pa, [4, 2]]).astype(np.int32)
    pb = np.concatenate([pb, [0, 2]]).astype(np.int32)
    kept, mt, md = ctx.match_sweep(bank, pa, pb)
    ok, om, od = ref.sweep(bank, pa, pb)
    assert np.array_equal(kept, ok) and np.array_equal(mt, om) and np.array_equal(md, od)
    for k in (0, 5):  # and the single-pair entry point agrees match by match
        r = ctx.match_bf_crosscheck(bank[pa[k]], bank[pb[k]])
        o = ref.bf_crosscheck(bank[pa[k]], bank[pb[k]])
        assert np.array_equal(r["q"], o["q"]) and np.array_equal(r["t"], o["t"])
        assert r["n_kept"] == kept[k] and len(r["q"]) == mt[k]


def test_sweep_many_pairs_resident(ctx, sweep_impl):
    """More pairs than SMs, exercising the persistent loop, A reuse and B double buffering."""
    n_kf, n_desc = 24, 700
    bank = synth.kf_bank(n_kf, n_desc, seed=1)
    pa, pb = synth.all_pairs(n_kf)
    ctx.bank_upload(bank)
    kept, mt, md = ctx.match_sweep_resident(pa, pb)
    ok, om, od = ref.sweep(bank, pa, pb)
    assert np.array_equal(kept, ok) and np.array_equal(mt, om) and np.array_equal(md, od)
    ctx.sweep_plan_upload(pa[:50], pb[:50])
    ctx.sweep_plan_run()
    ctx.sweep_plan_run()
    k2, m2, d2 = ctx.sweep_plan_download()
    assert np.array_equal(k2, ok[:50]) and np.array_equal(m2, om[:50]) and np.array_equal(d2, od[:50])
    # the same plan shifted along the bank (what bench.py does block after block)
    ctx.sweep_plan_upload(pa[:40] % 8, pb[:40] % 8)
    ctx.sweep_plan_run(kf_base=9)
    k3, m3, d3 = ctx.sweep_plan_download()
    o3 = ref.sweep(bank, pa[:40] % 8 + 9, pb[:40] % 8 + 9)
    assert np.array_equal(k3, o3[0]) and np.array_equal(m3, o3[1]) and np.array_equal(d3, o3[2])


def test_sweep_long_plan(ctx, sweep_impl):
    """A plan longer than one launch of the tensor-core kernel handles (16 384 keyframe pairs): the
    chunks must tile the pair list without a seam, runs of equal `a` cut by a chunk border included."""
    n_kf, n_desc = 200, 40
    bank = synth.kf_bank(n_kf, n_desc, seed=11)
    pa, pb = synth.all_pairs(n_kf)
    assert len(pa) == 19900
    ctx.bank_upload(bank)
    kept, mt, md = ctx.match_sweep_resident(pa, pb)
    ok, om, od = ref.sweep(bank, pa, pb)
    assert np.array_equal(kept, ok) and np.array_equal(mt, om) and np.array_equal(md, od)


@pytest.mark.parametrize("n_kf,blk,n_desc", [(11, 4, 300), (9, 4, 130), (8, 8, 64)])
def test_sweep_all_tile_grid(ctx, sweep_impl, n_kf, blk, n_desc):
    """The whole sweep as a tile grid split over ranks (SURVEY 8(e) row 1): the union of the ranks'
    results is the oracle's count for every unordered pair, ragged last block included."""
    bank = synth.kf_bank(n_kf, n_desc, seed=n_kf)
    ctx.bank_upload(bank)
    pa, pb = synth.all_pairs(n_kf)
    want = ref.sweep(bank, pa, pb)[0]
    one, done = ctx.match_sweep_all(n_kf, blk)
    assert done == len(pa) and np.array_equal(one, want)
    world = 3
    parts = [ctx.match_sweep_all(n_kf, blk, r, world) for r in range(world)]
    assert sum(d for _, d in parts) == len(pa)
    assert np.array_equal(sum(k for k, _ in parts), want)


def test_compute_descriptors(ctx):
    """SURVEY 8(f) rank 4: MapPoint::ComputeDescriptor batched, bit-exact vs the oracle."""
    rng = np.random.default_rng(17)
    sizes = np.concatenate([[0, 1, 2, 3, 128], rng.integers(1, 40, 400)]).astype(np.int32)
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    desc = np.zeros((offsets[-1], 32), np.uint8)
    for k, m in enumerate(sizes):
        if m == 0:
            continue
        base = synth.descriptors_uniform(1, rng)
        if k % 3 == 0:   # tie-heavy points
            desc[offsets[k]:offsets[k + 1]] = synth.descriptors_tie_stress(m, rng, 1, 3)
        else:
            desc[offsets[k]:offsets[k + 1]] = synth.descriptors_noisy_copy(np.repeat(base, m, 0), rng, 0.1)
    best, med = ctx.compute_descriptors(offsets, desc)
    ob, om = ref.compute_descriptors(offsets, desc)
    assert np.array_equal(best, ob) and np.array_equal(med, om)
    assert best[0] == -1 and best[1] == 0
    with pytest.raises(Exception):
        ctx.compute_descriptors(np.array([0, 129], np.int32), np.zeros((129, 32), np.uint8))
