"""ctypes binding of include/lorb_cuda.h — the call a Python user (tests,
bench.py) makes.  It is a thin, copy-free view over the C ABI: numpy arrays go
in as host pointers, exactly as the C++ Matcher/BA wrappers pass them.

There is no fallback: if liblorb_cuda.so is missing or a call fails, this
raises (LorbError); nothing here computes on the CPU.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "liblorb_cuda.so")

OK = 0
CROSSCHECK_MUTUAL, CROSSCHECK_LEGACY = 0, 1
SWEEP_POPC, SWEEP_TENSOR, SWEEP_DEFAULT = 0, 1, -1
# robust losses of the BA solvers (lorb_ba_set_loss): plain least squares, ceres::HuberLoss,
# SoftLOneLoss, CauchyLoss
LOSS_TRIVIAL, LOSS_HUBER, LOSS_SOFTLONE, LOSS_CAUCHY = 0, 1, 2, 3
TERMINATION = {0: "NO_CONVERGENCE", 1: "CONV_FUNCTION", 2: "CONV_GRADIENT", 3: "CONV_PARAMETER",
               4: "CONV_RADIUS", 5: "FAILURE"}

# every symbol include/lorb_cuda.h declares (tests check the .so exports all of them)
EXPORTS = [
    "lorb_ctx_create", "lorb_ctx_destroy", "lorb_ctx_sync", "lorb_ctx_stream",
    "lorb_ctx_launch_count", "lorb_last_error", "lorb_version",
    "lorb_match_bf_crosscheck", "lorb_match_knn2", "lorb_match_sweep", "lorb_bank_upload",
    "lorb_match_sweep_resident", "lorb_sweep_plan_upload", "lorb_sweep_plan_run",
    "lorb_sweep_plan_download", "lorb_sweep_plan_run_at", "lorb_sweep_set_impl", "lorb_sweep_plan_run_at2", "lorb_sweep_tile_count", "lorb_sweep_rank_tiles",
    "lorb_sweep_pair_index", "lorb_match_sweep_all", "lorb_search_proj_points", "lorb_search_proj_frame", "lorb_frustum_project", "lorb_compute_descriptors",
    "lorb_stereo_matches", "lorb_orb_describe", "lorb_orb_umax", "lorb_orb_selftest",
    "lorb_orb_extract", "lorb_orb_level_sizes", "lorb_orb_stages", "lorb_stereo_frame", "lorb_orb_distribute", "lorb_orb_max_keypoints",
    "lorb_ba_default_options", "lorb_ba_pose_only", "lorb_ba_local", "lorb_ba_local_batched", "lorb_ba_local_shard",
    "lorb_ba_problem_create", "lorb_ba_problem_create_batched", "lorb_ba_problem_create_sharded", "lorb_shard_range", "lorb_ba_shard_points", "lorb_set_host_threads", "lorb_ba_problem_reset", "lorb_ba_problem_solve",
    "lorb_ba_problem_download", "lorb_ba_problem_destroy", "lorb_ba_set_loss", "lorb_ba_get_loss",
    "lorb_dist_get_unique_id",
    "lorb_dist_init", "lorb_dist_finalize", "lorb_dist_allreduce_f64", "lorb_microbench_popc",
    "lorb_microbench_fp64", "lorb_microbench_tensor_i8", "lorb_ctx_profile", "lorb_ctx_profile_read",
]


class LorbError(RuntimeError):
    pass


class BAOptions(C.Structure):
    _fields_ = [("max_num_iterations", C.c_int), ("jacobi_scaling", C.c_int),
                ("max_consecutive_invalid_steps", C.c_int), ("reserved0", C.c_int),
                ("function_tolerance", C.c_double), ("gradient_tolerance", C.c_double),
                ("parameter_tolerance", C.c_double), ("initial_trust_region_radius", C.c_double),
                ("max_trust_region_radius", C.c_double), ("min_trust_region_radius", C.c_double),
                ("min_relative_decrease", C.c_double), ("min_lm_diagonal", C.c_double),
                ("max_lm_diagonal", C.c_double)]


class BALoss(C.Structure):
    _fields_ = [("kind", C.c_int), ("reserved", C.c_int), ("scale", C.c_double)]


class BASummary(C.Structure):
    _fields_ = [("initial_cost", C.c_double), ("final_cost", C.c_double),
                ("final_radius", C.c_double), ("final_gradient_max_norm", C.c_double),
                ("iterations", C.c_int), ("num_successful_steps", C.c_int),
                ("num_unsuccessful_steps", C.c_int), ("termination", C.c_int)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class FrameView(C.Structure):
    _fields_ = [("n_kp", C.c_int), ("kp_x", C.c_void_p), ("kp_y", C.c_void_p),
                ("kp_octave", C.c_void_p), ("kp_angle", C.c_void_p), ("kp_uright", C.c_void_p),
                ("desc", C.c_void_p), ("kp_claim_obs", C.c_void_p), ("min_x", C.c_float),
                ("max_x", C.c_float), ("min_y", C.c_float), ("max_y", C.c_float),
                ("n_levels", C.c_int), ("scale_factors", C.c_void_p)]


class OrbParams(C.Structure):
    _fields_ = [("nfeatures", C.c_int), ("scale_factor", C.c_float), ("nlevels", C.c_int),
                ("ini_th_fast", C.c_int), ("min_th_fast", C.c_int)]


class OrbKeypoints(C.Structure):
    _fields_ = [("n", C.c_int), ("x", C.c_void_p), ("y", C.c_void_p), ("octave", C.c_void_p),
                ("angle", C.c_void_p), ("response", C.c_void_p), ("size", C.c_void_p), ("desc", C.c_void_p),
                ("raw_levels", C.c_void_p)]


class PyramidView(C.Structure):
    _fields_ = [("n_levels", C.c_int), ("width", C.c_void_p), ("height", C.c_void_p),
                ("step", C.c_void_p), ("data", C.c_void_p)]


def _pyramid_view(pyr):
    lv = [np.ascontiguousarray(a, dtype=np.uint8) for a in pyr]
    w = np.array([a.shape[1] for a in lv], np.int32)
    h = np.array([a.shape[0] for a in lv], np.int32)
    st = np.array([a.strides[0] for a in lv], np.int32)
    ptrs = (C.c_void_p * len(lv))(*[a.ctypes.data for a in lv])
    v = PyramidView(len(lv), _ptr(w), _ptr(h), _ptr(st), C.cast(ptrs, C.c_void_p))
    return v, (lv, w, h, st, ptrs)


class Intrinsics(C.Structure):
    _fields_ = [("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float),
                ("mbf", C.c_float), ("mb", C.c_float)]


_lib = None


def load_library():
    """dlopen the C-ABI library; raise if it was not built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LorbError(
                "liblorb_cuda.so is not built (%s). Run `python -m lorb_slam_b200.build`; "
                "this package has no CPU fallback." % LIB_PATH)
        _lib = C.CDLL(LIB_PATH)
        _lib.lorb_last_error.restype = C.c_char_p
        _lib.lorb_version.restype = C.c_char_p
        _lib.lorb_ctx_stream.restype = C.c_void_p
        _lib.lorb_ctx_stream.argtypes = [C.c_void_p]
        _lib.lorb_ctx_launch_count.restype = C.c_longlong
        _lib.lorb_ctx_launch_count.argtypes = [C.c_void_p]
    return _lib


def _check(rc):
    if rc != OK:
        raise LorbError("lorb error %d: %s" % (rc, load_library().lorb_last_error().decode()))


def _ptr(a):
    return C.c_void_p(a.ctypes.data) if a is not None and a.size else C.c_void_p(0)


def _arr(a, dt, shape=None):
    a = np.ascontiguousarray(a, dtype=dt)
    return a.reshape(shape) if shape is not None else a


def ba_options(**kw):
    o = BAOptions()
    load_library().lorb_ba_default_options(C.byref(o))
    for k, v in kw.items():
        if not hasattr(o, k):
            raise AttributeError(k)
        setattr(o, k, v)
    return o


def _frame_view(fr):
    keep = [_arr(fr["kp_x"], np.float32), _arr(fr["kp_y"], np.float32),
            _arr(fr["kp_octave"], np.int32), _arr(fr["kp_angle"], np.float32),
            _arr(fr["kp_uright"], np.float32), _arr(fr["desc"], np.uint8),
            _arr(fr["kp_claim_obs"], np.int32), _arr(fr["scale_factors"], np.float32)]
    v = FrameView(int(fr["n_kp"]), _ptr(keep[0]), _ptr(keep[1]), _ptr(keep[2]), _ptr(keep[3]),
                  _ptr(keep[4]), _ptr(keep[5]), _ptr(keep[6]), float(fr["min_x"]),
                  float(fr["max_x"]), float(fr["min_y"]), float(fr["max_y"]),
                  int(fr["n_levels"]), _ptr(keep[7]))
    return v, keep


def sweep_rank_tiles(n_kf, block_kf, rank, world):
    """[(block row, block column)] of the tiles of `rank` (host logic only; no device needed)."""
    lib = load_library()
    n = C.c_int()
    _check(lib.lorb_sweep_rank_tiles(int(n_kf), int(block_kf), int(rank), int(world), 0, C.c_void_p(0),
                                     C.c_void_p(0), C.byref(n)))
    bi, bj = np.zeros(max(1, n.value), np.int32), np.zeros(max(1, n.value), np.int32)
    _check(lib.lorb_sweep_rank_tiles(int(n_kf), int(block_kf), int(rank), int(world), n.value, _ptr(bi),
                                     _ptr(bj), C.byref(n)))
    return list(zip(bi[:n.value].tolist(), bj[:n.value].tolist()))


def set_host_threads(n):
    _check(load_library().lorb_set_host_threads(int(n)))


def shard_range(n, rank, world):
    """Contiguous [lo, hi) slice of n units owned by `rank` (lorb_shard_range; host logic only)."""
    lo, hi = C.c_longlong(), C.c_longlong()
    _check(load_library().lorb_shard_range(C.c_longlong(int(n)), int(rank), int(world), C.byref(lo), C.byref(hi)))
    return int(lo.value), int(hi.value)


def ba_shard_points(P, obs_cam, obs_pt, rank, world):
    """Point indices of `rank` in the point-sharded large BA (lorb_ba_shard_points; host logic only)."""
    oc, op = _arr(obs_cam, np.int32), _arr(obs_pt, np.int32)
    ids = np.zeros(max(1, int(P)), np.int32)
    n = C.c_int()
    _check(load_library().lorb_ba_shard_points(int(P), len(oc), _ptr(oc), _ptr(op), int(rank), int(world),
                                               _ptr(ids), C.byref(n)))
    return ids[:n.value].copy()


def sweep_pair_index(n_kf, a, b):
    lib = load_library()
    lib.lorb_sweep_pair_index.restype = C.c_longlong
    return int(lib.lorb_sweep_pair_index(int(n_kf), int(a), int(b)))


class Context:
    """One lorb_ctx: a CUDA stream plus device/pinned scratch.  Not thread-safe;
    make one per calling thread (the reference runs Matcher on the tracking
    thread and local BA on the mapper thread, example/main.cpp:36-37)."""

    def __init__(self, device=0):
        self._lib = load_library()
        h = C.c_void_p()
        _check(self._lib.lorb_ctx_create(int(device), C.byref(h)))
        self._h = h
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            self._lib.lorb_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- plumbing
    def sync(self):
        _check(self._lib.lorb_ctx_sync(self._h))

    @property
    def stream(self):
        return self._lib.lorb_ctx_stream(self._h)

    @property
    def launch_count(self):
        return int(self._lib.lorb_ctx_launch_count(self._h))

    # -- brute force
    def match_bf_crosscheck(self, q, t, mode=CROSSCHECK_MUTUAL):
        q, t = _arr(q, np.uint8).reshape(-1, 32), _arr(t, np.uint8).reshape(-1, 32)
        cap = max(1, min(len(q), len(t)))
        oq, ot, od = (np.zeros(cap, np.int32) for _ in range(3))
        keep = np.zeros(cap, np.uint8)
        n, nk, md = C.c_int(), C.c_int(), C.c_int()
        _check(self._lib.lorb_match_bf_crosscheck(
            self._h, _ptr(q), len(q), _ptr(t), len(t), int(mode), _ptr(oq), _ptr(ot), _ptr(od),
            _ptr(keep), C.byref(n), C.byref(nk), C.byref(md)))
        k = n.value
        return dict(q=oq[:k], t=ot[:k], dist=od[:k], keep=keep[:k], n_kept=nk.value,
                    min_dist=md.value)

    def match_knn2(self, q, t, ratio=0.8, max_dist=100):
        q, t = _arr(q, np.uint8).reshape(-1, 32), _arr(t, np.uint8).reshape(-1, 32)
        n = max(1, len(q))
        idx, dist = np.zeros((n, 2), np.int32), np.zeros((n, 2), np.int32)
        ok = np.zeros(n, np.uint8)
        _check(self._lib.lorb_match_knn2(self._h, _ptr(q), len(q), _ptr(t), len(t),
                                         C.c_float(ratio), int(max_dist), _ptr(idx), _ptr(dist),
                                         _ptr(ok)))
        return idx[:len(q)], dist[:len(q)], ok[:len(q)]

    def sweep_set_impl(self, impl):
        """SWEEP_POPC / SWEEP_TENSOR / SWEEP_DEFAULT (or "popc" / "tensor" / "default")."""
        impl = {"popc": SWEEP_POPC, "tensor": SWEEP_TENSOR, "default": SWEEP_DEFAULT}.get(impl, impl)
        _check(self._lib.lorb_sweep_set_impl(self._h, int(impl)))

    def ba_set_loss(self, kind, scale=1.0):
        """Robust loss (LOSS_*, scale a in pixels) of every later BA solve on this ctx."""
        _check(self._lib.lorb_ba_set_loss(self._h, C.byref(BALoss(int(kind), 0, float(scale)))))

    def ba_get_loss(self):
        """-> (kind, scale) of the ctx's BA loss."""
        lo = BALoss()
        _check(self._lib.lorb_ba_get_loss(self._h, C.byref(lo)))
        return lo.kind, lo.scale

    def bank_upload(self, bank):
        bank = _arr(bank, np.uint8)
        assert bank.ndim == 3 and bank.shape[2] == 32
        _check(self._lib.lorb_bank_upload(self._h, _ptr(bank), bank.shape[0], bank.shape[1]))

    def match_sweep(self, bank, pair_a, pair_b):
        bank = _arr(bank, np.uint8)
        pa, pb = _arr(pair_a, np.int32), _arr(pair_b, np.int32)
        n = len(pa)
        kept, mt, md = (np.zeros(max(1, n), np.int32) for _ in range(3))
        _check(self._lib.lorb_match_sweep(self._h, _ptr(bank), bank.shape[0], bank.shape[1],
                                          _ptr(pa), _ptr(pb), n, _ptr(kept), _ptr(mt), _ptr(md)))
        return kept[:n], mt[:n], md[:n]

    def match_sweep_resident(self, pair_a, pair_b):
        pa, pb = _arr(pair_a, np.int32), _arr(pair_b, np.int32)
        n = len(pa)
        kept, mt, md = (np.zeros(max(1, n), np.int32) for _ in range(3))
        _check(self._lib.lorb_match_sweep_resident(self._h, _ptr(pa), _ptr(pb), n, _ptr(kept),
                                                   _ptr(mt), _ptr(md)))
        return kept[:n], mt[:n], md[:n]

    def sweep_plan_upload(self, pair_a, pair_b):
        pa, pb = _arr(pair_a, np.int32), _arr(pair_b, np.int32)
        self._plan_n = len(pa)
        _check(self._lib.lorb_sweep_plan_upload(self._h, _ptr(pa), _ptr(pb), len(pa)))

    def sweep_plan_run(self, kf_base=0, kf_base_b=None):
        if kf_base_b is None:
            _check(self._lib.lorb_sweep_plan_run_at(self._h, int(kf_base)))
        else:
            _check(self._lib.lorb_sweep_plan_run_at2(self._h, int(kf_base), int(kf_base_b)))

    def match_sweep_all(self, n_kf, block_kf, rank=0, world=1, out=None):
        """Every unordered keyframe pair of the resident bank, this rank's tiles of the keyframe
        grid (lorb_match_sweep_all).  -> (kept counts [n_kf (n_kf - 1) / 2], pairs done)."""
        n = n_kf * (n_kf - 1) // 2
        if out is None:
            out = np.zeros(max(1, n), np.int32)
        done = C.c_longlong()
        _check(self._lib.lorb_match_sweep_all(self._h, int(block_kf), int(rank), int(world), _ptr(out),
                                              C.byref(done)))
        return out[:n], done.value

    def sweep_plan_download(self):
        n = self._plan_n
        kept, mt, md = (np.zeros(max(1, n), np.int32) for _ in range(3))
        _check(self._lib.lorb_sweep_plan_download(self._h, _ptr(kept), _ptr(mt), _ptr(md)))
        return kept[:n], mt[:n], md[:n]

    # -- projection-guided search
    def search_proj_points(self, fr, pts, th):
        v, keep = _frame_view(fr)
        n_pts = int(pts["n_pts"])
        a = [_arr(pts["proj_x"], np.float32), _arr(pts["proj_y"], np.float32),
             _arr(pts["proj_xr"], np.float32), _arr(pts["level"], np.int32),
             _arr(pts["view_cos"], np.float32), _arr(pts["active"], np.uint8),
             _arr(pts["mp_desc"], np.uint8), _arr(pts["mp_nobs"], np.int32)]
        kfp = np.full(max(1, n_pts), -1, np.int32)
        pfk = np.full(max(1, v.n_kp), -1, np.int32)
        nm, nc = C.c_int(), C.c_longlong()
        _check(self._lib.lorb_search_proj_points(
            self._h, C.byref(v), n_pts, *[_ptr(x) for x in a], C.c_float(th), _ptr(kfp), _ptr(pfk),
            C.byref(nm), C.byref(nc)))
        return dict(kp_for_point=kfp[:n_pts], point_for_kp=pfk[:v.n_kp], n_matches=nm.value,
                    n_candidates=nc.value)

    def search_proj_frame(self, cur, last, th):
        v, keep = _frame_view(cur)
        n_last = int(last["n_last"])
        K = last["K"]
        Ks = Intrinsics(K["fx"], K["fy"], K["cx"], K["cy"], K["mbf"], K["mb"])
        tc, tl = _arr(last["tcw_cur"], np.float32), _arr(last["tcw_last"], np.float32)
        a = [_arr(last["valid"], np.uint8), _arr(last["xw"], np.float32),
             _arr(last["octave"], np.int32), _arr(last["angle"], np.float32),
             _arr(last["mp_desc"], np.uint8), _arr(last["mp_nobs"], np.int32)]
        kfi = np.full(max(1, n_last), -1, np.int32)
        sfk = np.full(max(1, v.n_kp), -1, np.int32)
        nm, nc = C.c_int(), C.c_longlong()
        _check(self._lib.lorb_search_proj_frame(
            self._h, C.byref(v), _ptr(tc), _ptr(tl), C.byref(Ks), n_last, *[_ptr(x) for x in a],
            C.c_float(th), _ptr(kfi), _ptr(sfk), C.byref(nm), C.byref(nc)))
        return dict(kp_for_item=kfi[:n_last], state_for_kp=sfk[:v.n_kp], n_matches=nm.value,
                    n_candidates=nc.value)

    def compute_descriptors(self, offsets, desc):
        offsets = _arr(offsets, np.int32)
        desc = _arr(desc, np.uint8).reshape(-1, 32)
        n = len(offsets) - 1
        best, med = np.zeros(max(1, n), np.int32), np.zeros(max(1, n), np.int32)
        _check(self._lib.lorb_compute_descriptors(self._h, n, _ptr(offsets), _ptr(desc), _ptr(best),
                                                  _ptr(med)))
        return best[:n], med[:n]

    def stereo_matches(self, st):
        """Frame::ComputeStereoMatches; st as produced by synth.make_stereo_pair."""
        vl, kl = _pyramid_view(st["pyr_left"])
        vr, kr = _pyramid_view(st["pyr_right"])
        n, nr = int(st["n_left"]), int(st["n_right"])
        a = [_arr(st["scale_factors"], np.float32), _arr(st["inv_scale_factors"], np.float32),
             _arr(st["lx"], np.float32), _arr(st["ly"], np.float32), _arr(st["loct"], np.int32),
             _arr(st["ldesc"], np.uint8), _arr(st["rx"], np.float32), _arr(st["ry"], np.float32),
             _arr(st["roct"], np.int32), _arr(st["rdesc"], np.uint8)]
        ur, dp = np.zeros(max(1, n), np.float32), np.zeros(max(1, n), np.float32)
        nm = C.c_int(0)
        _check(self._lib.lorb_stereo_matches(
            self._h, C.byref(vl), C.byref(vr), int(st["n_levels"]), _ptr(a[0]), _ptr(a[1]),
            C.c_float(st["mbf"]), C.c_float(st["mb"]), n, _ptr(a[2]), _ptr(a[3]), _ptr(a[4]), _ptr(a[5]),
            nr, _ptr(a[6]), _ptr(a[7]), _ptr(a[8]), _ptr(a[9]), _ptr(ur), _ptr(dp), C.byref(nm)))
        return dict(uright=ur[:n], depth=dp[:n], n_matched=nm.value)

    def orb_describe(self, oi, pattern, angle_in=None):
        """IC_Angle + computeOrbDescriptor; oi as produced by synth.make_orb_inputs, pattern
        [512, 2] int32 -> (angle[n], desc[n, 32])."""
        vb, kb = _pyramid_view(oi["pyr_blur"])
        vr, kr = _pyramid_view(oi["pyr_raw"])
        n = int(oi["n_kp"])
        a = [_arr(pattern, np.int32).reshape(-1), _arr(oi["kx"], np.float32), _arr(oi["ky"], np.float32),
             _arr(oi["klevel"], np.int32)]
        ang = np.zeros(max(1, n), np.float32)
        desc = np.zeros((max(1, n), 32), np.uint8)
        ain = None if angle_in is None else _arr(angle_in, np.float32)
        _check(self._lib.lorb_orb_describe(
            self._h, C.byref(vr), C.byref(vb), int(oi["n_levels"]), _ptr(a[0]), n, _ptr(a[1]), _ptr(a[2]),
            _ptr(a[3]), None if ain is None else _ptr(ain), _ptr(ang), _ptr(desc)))
        return ang[:n], desc[:n]

    def orb_level_sizes(self, width, height, nfeatures=1000, scale_factor=1.2, nlevels=8, ini_th=20, min_th=7):
        prm = OrbParams(nfeatures, scale_factor, nlevels, ini_th, min_th)
        w, h, nf = np.zeros(nlevels, np.int32), np.zeros(nlevels, np.int32), np.zeros(nlevels, np.int32)
        sf = np.zeros(nlevels, np.float32)
        _check(self._lib.lorb_orb_level_sizes(C.byref(prm), width, height, _ptr(w), _ptr(h), _ptr(nf), _ptr(sf)))
        return w, h, nf, sf

    def orb_max_keypoints(self, width, height, nfeatures=1000, scale_factor=1.2, nlevels=8, ini_th=20, min_th=7):
        prm = OrbParams(nfeatures, scale_factor, nlevels, ini_th, min_th)
        n = C.c_int(0)
        _check(self._lib.lorb_orb_max_keypoints(C.byref(prm), width, height, C.byref(n)))
        return n.value

    def orb_extract(self, img, pattern, nfeatures=1000, scale_factor=1.2, nlevels=8, ini_th=20, min_th=7):
        """ORBextractor::operator() on one 8-bit image -> dict like oracle.reflib.orb_extract."""
        img = _arr(img, np.uint8)
        prm = OrbParams(nfeatures, scale_factor, nlevels, ini_th, min_th)
        pat = _arr(pattern, np.int32).reshape(-1)
        cap = max(1, self.orb_max_keypoints(img.shape[1], img.shape[0], nfeatures, scale_factor, nlevels, ini_th, min_th))
        kx, ky = np.zeros(cap, np.float32), np.zeros(cap, np.float32)
        ko, ka = np.zeros(cap, np.int32), np.zeros(cap, np.float32)
        kr, ks = np.zeros(cap, np.float32), np.zeros(cap, np.float32)
        desc = np.zeros((cap, 32), np.uint8)
        n = C.c_int(0)
        _check(self._lib.lorb_orb_extract(
            self._h, _ptr(img), img.shape[1], img.shape[0], img.strides[0], C.byref(prm), _ptr(pat), cap,
            _ptr(kx), _ptr(ky), _ptr(ko), _ptr(ka), _ptr(kr), _ptr(ks), _ptr(desc), C.byref(n), None))
        n = n.value
        return dict(n=n, x=kx[:n], y=ky[:n], octave=ko[:n], angle=ka[:n], response=kr[:n], size=ks[:n],
                    desc=desc[:n], n_per_level=np.bincount(ko[:n], minlength=nlevels).astype(np.int32))

    def stereo_frame(self, left, right, pattern, mbf, mb, nfeatures=1000, scale_factor=1.2, nlevels=8, ini_th=20,
                     min_th=7):
        """Frame's stereo constructor on the device: both extractions + ComputeStereoMatches.
        -> (left dict, right dict, uright, depth, n_matched)"""
        left, right = _arr(left, np.uint8), _arr(right, np.uint8)
        assert left.shape == right.shape
        prm = OrbParams(nfeatures, scale_factor, nlevels, ini_th, min_th)
        pat = _arr(pattern, np.int32).reshape(-1)
        cap = max(1, self.orb_max_keypoints(left.shape[1], left.shape[0], nfeatures, scale_factor, nlevels, ini_th, min_th))
        keep, views = [], []
        for _ in range(2):
            a = dict(x=np.zeros(cap, np.float32), y=np.zeros(cap, np.float32), octave=np.zeros(cap, np.int32),
                     angle=np.zeros(cap, np.float32), response=np.zeros(cap, np.float32),
                     size=np.zeros(cap, np.float32), desc=np.zeros((cap, 32), np.uint8))
            keep.append(a)
            views.append(OrbKeypoints(0, _ptr(a["x"]), _ptr(a["y"]), _ptr(a["octave"]), _ptr(a["angle"]),
                                      _ptr(a["response"]), _ptr(a["size"]), _ptr(a["desc"]), None))
        ur, dp = np.zeros(cap, np.float32), np.zeros(cap, np.float32)
        nm = C.c_int(0)
        _check(self._lib.lorb_stereo_frame(
            self._h, _ptr(left), _ptr(right), left.shape[1], left.shape[0], left.strides[0], right.strides[0],
            C.byref(prm), _ptr(pat), C.c_float(mbf), C.c_float(mb), cap, C.byref(views[0]), C.byref(views[1]),
            _ptr(ur), _ptr(dp), C.byref(nm)))
        res = []
        for a, v in zip(keep, views):
            n = v.n
            d = {k: a[k][:n] for k in a}
            d["n"] = n
            res.append(d)
        return res[0], res[1], ur[:res[0]["n"]], dp[:res[0]["n"]], nm.value

    def orb_stages(self, img, nfeatures=1000, scale_factor=1.2, nlevels=8, ini_th=20, min_th=7):
        """Pyramid, blurred pyramid and the candidate keypoints handed to the quadtree."""
        img = _arr(img, np.uint8)
        prm = OrbParams(nfeatures, scale_factor, nlevels, ini_th, min_th)
        w, h, _, _ = self.orb_level_sizes(img.shape[1], img.shape[0], nfeatures, scale_factor, nlevels, ini_th, min_th)
        raw = [np.zeros((h[l], w[l]), np.uint8) for l in range(nlevels)]
        blur = [np.zeros((h[l], w[l]), np.uint8) for l in range(nlevels)]
        pr = (C.c_void_p * nlevels)(*[a.ctypes.data for a in raw])
        pb = (C.c_void_p * nlevels)(*[a.ctypes.data for a in blur])
        cap = int(sum(int(w[l]) * int(h[l]) for l in range(nlevels)) // 4 + 1024)
        cx, cy, cr = np.zeros(cap, np.float32), np.zeros(cap, np.float32), np.zeros(cap, np.float32)
        ls = np.zeros(nlevels + 1, np.int32)
        _check(self._lib.lorb_orb_stages(
            self._h, _ptr(img), img.shape[1], img.shape[0], img.strides[0], C.byref(prm), pr, pb, cap,
            _ptr(cx), _ptr(cy), _ptr(cr), _ptr(ls)))
        t = int(ls[-1])
        return dict(raw=raw, blur=blur, cand_x=cx[:t], cand_y=cy[:t], cand_response=cr[:t], level_start=ls)

    def orb_distribute(self, x, y, response, min_x, max_x, min_y, max_y, n_features):
        """ORBextractor::DistributeOctTree alone (device quadtree) -> chosen indices."""
        x, y, r = (_arr(a, np.float32) for a in (x, y, response))
        out = np.zeros(max(n_features + 16, len(x) + 16), np.int32)
        n = C.c_int(0)
        _check(self._lib.lorb_orb_distribute(self._h, len(x), _ptr(x), _ptr(y), _ptr(r), min_x, max_x, min_y,
                                                 max_y, n_features, _ptr(out), C.byref(n)))
        return out[:n.value]

    def orb_selftest(self, a, b):
        a, b = _arr(a, np.float32), _arr(b, np.float32)
        n = len(a)
        s, c, t = np.zeros(n, np.float32), np.zeros(n, np.float32), np.zeros(n, np.float32)
        _check(self._lib.lorb_orb_selftest(self._h, n, _ptr(a), _ptr(b), _ptr(s), _ptr(c), _ptr(t)))
        return s, c, t

    def frustum_project(self, fp):
        n = int(fp["n"])
        K = fp["K"]
        Ks = Intrinsics(K["fx"], K["fy"], K["cx"], K["cy"], K["mbf"], K.get("mb", 0.0))
        a = [_arr(fp["tcw"], np.float32), _arr(fp["ow"], np.float32), _arr(fp["xw"], np.float32),
             _arr(fp["normal"], np.float32), _arr(fp["min_dist"], np.float32),
             _arr(fp["max_dist"], np.float32)]
        out = dict(in_view=np.zeros(max(1, n), np.uint8), proj_x=np.full(max(1, n), -7.0, np.float32),
                   proj_y=np.full(max(1, n), -7.0, np.float32),
                   proj_xr=np.full(max(1, n), -7.0, np.float32),
                   level=np.full(max(1, n), -7, np.int32),
                   view_cos=np.full(max(1, n), -7.0, np.float32))
        _check(self._lib.lorb_frustum_project(
            self._h, _ptr(a[0]), _ptr(a[1]), C.byref(Ks), C.c_float(fp["min_x"]),
            C.c_float(fp["max_x"]), C.c_float(fp["min_y"]), C.c_float(fp["max_y"]), n, _ptr(a[2]),
            _ptr(a[3]), _ptr(a[4]), _ptr(a[5]), C.c_float(fp["cos_limit"]), C.c_float(fp["log_sf"]),
            int(fp["n_levels"]), _ptr(out["in_view"]), _ptr(out["proj_x"]), _ptr(out["proj_y"]),
            _ptr(out["proj_xr"]), _ptr(out["level"]), _ptr(out["view_cos"])))
        return {k: v[:n] for k, v in out.items()}

    # -- bundle adjustment
    def ba_pose_only(self, xw, uv, K, rt, opt=None):
        xw, uv = _arr(xw, np.float32).reshape(-1, 3), _arr(uv, np.float32).reshape(-1, 2)
        K = _arr(K, np.float32).reshape(4)
        rt = _arr(rt, np.float64).reshape(6).copy()
        opt = opt or ba_options()
        s = BASummary()
        _check(self._lib.lorb_ba_pose_only(self._h, len(xw), _ptr(xw), _ptr(uv), _ptr(K), _ptr(rt),
                                           C.byref(opt), C.byref(s)))
        return rt, s.as_dict()

    def ba_local_shard(self, pb, opt=None):
        """lorb_ba_local_shard: `pb` is this rank's shard; collective over the ctx communicator."""
        return self.ba_local(pb, opt, _entry="lorb_ba_local_shard")

    def ba_local(self, pb, opt=None, _entry="lorb_ba_local"):
        cams = _arr(pb["cams"], np.float64).copy()
        pts = _arr(pb["pts"], np.float64).copy()
        oc, op = _arr(pb["obs_cam"], np.int32), _arr(pb["obs_pt"], np.int32)
        ouv = _arr(pb["obs_uv"], np.float32)
        fp = _arr(pb.get("fix_pt", np.zeros(0)), np.int32)
        fuv = _arr(pb.get("fix_uv", np.zeros((0, 2))), np.float32)
        frt = _arr(pb.get("fix_rt", np.zeros((0, 6))), np.float32)
        K = _arr(pb["K"], np.float32).reshape(4)
        opt = opt or ba_options()
        s = BASummary()
        _check(getattr(self._lib, _entry)(self._h, len(cams), _ptr(cams), len(pts), _ptr(pts), len(oc),
                                       _ptr(oc), _ptr(op), _ptr(ouv), len(fp), _ptr(fp), _ptr(fuv),
                                       _ptr(frt), _ptr(K), C.byref(opt), C.byref(s)))
        return cams, pts, s.as_dict()

    def ba_local_batched(self, bt, opt=None, inplace=False):
        """inplace: bt["cams"] / bt["pts"] (contiguous float64) are updated where they lie, as a C++
        caller's arrays would be; otherwise they are copied first."""
        if inplace:
            cams, pts = bt["cams"], bt["pts"]
            assert cams.dtype == np.float64 and pts.dtype == np.float64
            assert cams.flags.c_contiguous and pts.flags.c_contiguous
        else:
            cams = _arr(bt["cams"], np.float64).copy()
            pts = _arr(bt["pts"], np.float64).copy()
        co, po, oo = (_arr(bt[k], np.int32) for k in ("cam_off", "pt_off", "obs_off"))
        oc, op = _arr(bt["obs_cam"], np.int32), _arr(bt["obs_pt"], np.int32)
        ouv = _arr(bt["obs_uv"], np.float32)
        K = _arr(bt["K"], np.float32).reshape(4)
        nw = int(bt["n_windows"])
        opt = opt or ba_options()
        sums = (BASummary * nw)()
        null = C.c_void_p(0)
        fo = fp = fuv = frt = None
        if "fix_off" in bt:
            fo, fp = _arr(bt["fix_off"], np.int32), _arr(bt["fix_pt"], np.int32)
            fuv, frt = _arr(bt["fix_uv"], np.float32), _arr(bt["fix_rt"], np.float32)
        _check(self._lib.lorb_ba_local_batched(
            self._h, nw, _ptr(co), _ptr(cams), _ptr(po), _ptr(pts), _ptr(oo), _ptr(oc), _ptr(op),
            _ptr(ouv), _ptr(fo) if fo is not None else null, _ptr(fp) if fo is not None else null,
            _ptr(fuv) if fo is not None else null, _ptr(frt) if fo is not None else null, _ptr(K),
            C.byref(opt), sums))
        return cams, pts, [s.as_dict() for s in sums]

    def ba_problem(self, pb):
        return BAProblem(self, pb)

    def ba_problem_batched(self, bt):
        return BAProblem(self, None, batch=bt)

    def ba_problem_sharded(self, pb, rank, world):
        """This rank's point shard of the whole problem `pb` (lorb_ba_problem_create_sharded)."""
        return BAProblem(self, pb, shard=(rank, world))

    # -- multi-GPU
    @staticmethod
    def dist_unique_id():
        buf = (C.c_uint8 * 128)()
        _check(load_library().lorb_dist_get_unique_id(buf))
        return bytes(buf)

    def dist_init(self, uid, rank, world):
        buf = (C.c_uint8 * 128).from_buffer_copy(uid)
        _check(self._lib.lorb_dist_init(self._h, buf, int(rank), int(world)))

    def dist_finalize(self):
        _check(self._lib.lorb_dist_finalize(self._h))

    def dist_allreduce_f64(self, a):
        a = _arr(a, np.float64).copy()
        _check(self._lib.lorb_dist_allreduce_f64(self._h, _ptr(a), a.size))
        return a

    # -- diagnostics
    def microbench_fp64(self, kind=0, iters=4096):
        """flop/s of independent DFMA chains (kind 0) or DMMA m8n8k4 (kind 1), whole GPU."""
        v = C.c_double()
        _check(self._lib.lorb_microbench_fp64(self._h, int(kind), int(iters), C.byref(v)))
        return v.value

    def profile(self, enable=True):
        _check(self._lib.lorb_ctx_profile(self._h, 1 if enable else 0))

    def profile_read(self, slot):
        """-> (total milliseconds, launches) of a bracketed kernel slot (see lorb_cuda.h)."""
        ms, n = C.c_double(), C.c_longlong()
        _check(self._lib.lorb_ctx_profile_read(self._h, int(slot), C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def microbench_tensor_i8(self, tiles=4096):
        r = C.c_double()
        _check(self._lib.lorb_microbench_tensor_i8(self._h, int(tiles), C.byref(r)))
        return r.value

    def microbench_popc(self, kind=0, iters=4096):
        r = C.c_double()
        _check(self._lib.lorb_microbench_popc(self._h, int(kind), int(iters), C.byref(r)))
        return r.value


class BAProblem:
    """Device-resident local-BA problem (lorb_ba_problem_*)."""

    def __init__(self, ctx, pb, batch=None, shard=None):
        self._ctx = ctx
        self._lib = ctx._lib
        self.nw = 1
        if batch is not None:
            bt = batch
            cams, pts = _arr(bt["cams"], np.float64), _arr(bt["pts"], np.float64)
            co, po, oo = (_arr(bt[k], np.int32) for k in ("cam_off", "pt_off", "obs_off"))
            oc, op = _arr(bt["obs_cam"], np.int32), _arr(bt["obs_pt"], np.int32)
            ouv = _arr(bt["obs_uv"], np.float32)
            K = _arr(bt["K"], np.float32).reshape(4)
            self.C, self.P, self.nw = len(cams), len(pts), int(bt["n_windows"])
            h = C.c_void_p()
            fix = [C.c_void_p(0)] * 4
            if "fix_off" in bt:
                self._fix = (_arr(bt["fix_off"], np.int32), _arr(bt["fix_pt"], np.int32),
                             _arr(bt["fix_uv"], np.float32), _arr(bt["fix_rt"], np.float32))
                fix = [_ptr(a) for a in self._fix]
            _check(self._lib.lorb_ba_problem_create_batched(
                ctx._h, self.nw, _ptr(co), _ptr(cams), _ptr(po), _ptr(pts), _ptr(oo), _ptr(oc),
                _ptr(op), _ptr(ouv), fix[0], fix[1], fix[2], fix[3], _ptr(K), C.byref(h)))
            self._h = h
            return
        cams, pts = _arr(pb["cams"], np.float64), _arr(pb["pts"], np.float64)
        oc, op = _arr(pb["obs_cam"], np.int32), _arr(pb["obs_pt"], np.int32)
        ouv = _arr(pb["obs_uv"], np.float32)
        fp = _arr(pb.get("fix_pt", np.zeros(0)), np.int32)
        fuv = _arr(pb.get("fix_uv", np.zeros((0, 2))), np.float32)
        frt = _arr(pb.get("fix_rt", np.zeros((0, 6))), np.float32)
        K = _arr(pb["K"], np.float32).reshape(4)
        self.C, self.P = len(cams), len(pts)
        h = C.c_void_p()
        if shard is not None:
            ids, n = np.zeros(max(1, len(pts)), np.int32), C.c_int()
            _check(self._lib.lorb_ba_problem_create_sharded(
                ctx._h, len(cams), _ptr(cams), len(pts), _ptr(pts), len(oc), _ptr(oc), _ptr(op),
                _ptr(ouv), len(fp), _ptr(fp), _ptr(fuv), _ptr(frt), _ptr(K), int(shard[0]), int(shard[1]),
                C.byref(h), _ptr(ids), C.byref(n)))
            self.point_ids = ids[:n.value].copy()
            self.P = n.value
            self._h = h
            return
        _check(self._lib.lorb_ba_problem_create(
            ctx._h, len(cams), _ptr(cams), len(pts), _ptr(pts), len(oc), _ptr(oc), _ptr(op),
            _ptr(ouv), len(fp), _ptr(fp), _ptr(fuv), _ptr(frt), _ptr(K), C.byref(h)))
        self._h = h

    def reset(self):
        _check(self._lib.lorb_ba_problem_reset(self._h))

    def solve(self, opt=None, sharded=False):
        opt = opt or ba_options()
        if self.nw > 1:
            sums = (BASummary * self.nw)()
            _check(self._lib.lorb_ba_problem_solve(self._h, C.byref(opt), 0, sums))
            return [x.as_dict() for x in sums]
        s = BASummary()
        _check(self._lib.lorb_ba_problem_solve(self._h, C.byref(opt), int(bool(sharded)),
                                               C.byref(s)))
        return s.as_dict()

    def download(self):
        cams = np.zeros((self.C, 6), np.float64)
        pts = np.zeros((self.P, 3), np.float64)
        _check(self._lib.lorb_ba_problem_download(self._h, _ptr(cams), _ptr(pts)))
        return cams, pts

    def close(self):
        if getattr(self, "_h", None):
            self._lib.lorb_ba_problem_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
