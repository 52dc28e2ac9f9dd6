"""TEST INFRASTRUCTURE ONLY: the BA oracle with a robust loss (ba_robust_ref.cpp), for the tests and
profiles of lorb_ba_set_loss.  The library is the oracle's own source (oracle/ba_ref.cpp) with its
linearize() / eval_cost() replaced by the loss-corrected forms of ba_robust_ref.cpp; it is compiled
on first use into the temporary directory (keyed by the sources' hash), never into the tree.

loss: None (plain least squares, the reference) or (LOSS_*, scale a)."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import ref

LOSS_TRIVIAL, LOSS_HUBER, LOSS_SOFTLONE, LOSS_CAUCHY = 0, 1, 2, 3

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_ORACLE = os.path.join(_ROOT, "oracle", "ba_ref.cpp")
_PATCH = os.path.join(_HERE, "ba_robust_ref.cpp")
_lib = None


def _source():
    src, patch = open(_ORACLE).read(), open(_PATCH).read()
    part1, part2 = patch.split("// ---- part 2: appended after the oracle's C entry points\n")
    for name, sig in (("eval_cost", "(const Problem& pb, const double* cams, const double* pts) {"),
                      ("linearize", "(const Problem& pb, Lin& L) {")):
        old = "\ndouble %s%s" % (name, sig)
        assert src.count(old) == 1, name
        src = src.replace(old, "\ndouble plain_%s%s" % (name, sig))
    anchor = "\ninline bool has_cam("
    assert src.count(anchor) == 1
    src = src.replace(anchor, "\n" + part1 + anchor)
    return src + "\n" + part2


def _load():
    global _lib
    if _lib is None:
        src = _source()
        key = hashlib.sha256(src.encode()).hexdigest()[:16]
        out = os.path.join(tempfile.gettempdir(), "lorb_ba_robust_ref_%s_%d.so" % (key, os.getuid()))
        if not os.path.exists(out):
            cpp = out[:-3] + ".cpp"
            with open(cpp, "w") as f:
                f.write(src)
            tmp = out + ".%d" % os.getpid()
            subprocess.run(["/usr/bin/g++", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
                            "-fopenmp", "-std=c++14", "-I", os.path.join(_ROOT, "oracle"), "-o", tmp, cpp, "-lm"],
                           check=True, capture_output=True)
            os.replace(tmp, out)
        _lib = C.CDLL(out)
        _lib.orc_ba_local_cost.restype = C.c_double
        _lib.orc_ba_set_loss.argtypes = [C.c_int, C.c_double]
        _lib.orc_ba_loss_eval.argtypes = [C.c_int, C.c_double, C.c_double, C.POINTER(C.c_double)]
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def _arr(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


def _set_loss(loss):
    kind, scale = (LOSS_TRIVIAL, 1.0) if loss is None else (int(loss[0]), float(loss[1]))
    _load().orc_ba_set_loss(kind, scale)


def loss_eval(kind, scale, s):
    """(rho, rho', rho'') of the loss at s = |r|^2."""
    out = np.zeros(3)
    _load().orc_ba_loss_eval(int(kind), float(scale), float(s), _p(out, C.c_double))
    return tuple(float(v) for v in out)


def ba_pose_only(xw, uv, K, rt, opt=None, loss=None):
    xw, uv, K = _arr(xw, np.float32).reshape(-1, 3), _arr(uv, np.float32).reshape(-1, 2), _arr(K, np.float32).reshape(4)
    rt = _arr(rt, np.float64).reshape(6).copy()
    opt = opt or ref.ba_options()
    s = ref.BASummary()
    _set_loss(loss)
    rc = _load().orc_ba_pose_only(len(xw), _p(xw, C.c_float), _p(uv, C.c_float), _p(K, C.c_float),
                                  _p(rt, C.c_double), C.byref(opt), C.byref(s))
    assert rc == 0
    return rt, s.as_dict()


def _local_args(pb, cams, pts):
    oc, op, ouv = _arr(pb["obs_cam"], np.int32), _arr(pb["obs_pt"], np.int32), _arr(pb["obs_uv"], np.float32)
    fp, fuv = _arr(pb.get("fix_pt", []), np.int32), _arr(pb.get("fix_uv", []), np.float32)
    frt, K = _arr(pb.get("fix_rt", []), np.float32), _arr(pb["K"], np.float32).reshape(4)
    keep = (cams, pts, oc, op, ouv, fp, fuv, frt, K)
    args = (len(cams), _p(cams, C.c_double), len(pts), _p(pts, C.c_double), len(oc), _p(oc, C.c_int),
            _p(op, C.c_int), _p(ouv, C.c_float), len(fp), _p(fp, C.c_int), _p(fuv, C.c_float),
            _p(frt, C.c_float), _p(K, C.c_float))
    return args, keep


def ba_local(pb, opt=None, loss=None):
    """pb: dict(cams[C,6], pts[P,3], obs_cam, obs_pt, obs_uv, fix_pt, fix_uv, fix_rt, K)."""
    cams, pts = _arr(pb["cams"], np.float64).copy(), _arr(pb["pts"], np.float64).copy()
    args, _keep = _local_args(pb, cams, pts)
    opt = opt or ref.ba_options()
    s = ref.BASummary()
    _set_loss(loss)
    assert _load().orc_ba_local(*args, C.byref(opt), C.byref(s)) == 0
    return cams, pts, s.as_dict()


def ba_local_cost(pb, cams=None, pts=None, loss=None):
    """1/2 sum rho(|r|^2) of a local-BA state."""
    cams = _arr(pb["cams"] if cams is None else cams, np.float64)
    pts = _arr(pb["pts"] if pts is None else pts, np.float64)
    args, _keep = _local_args(pb, cams, pts)
    _set_loss(loss)
    return float(_load().orc_ba_local_cost(*args))


def ba_local_batched(cam_off, cams, pt_off, pts, obs_off, obs_cam, obs_pt, obs_uv, K, opt=None, loss=None):
    cam_off, pt_off, obs_off = _arr(cam_off, np.int32), _arr(pt_off, np.int32), _arr(obs_off, np.int32)
    cams, pts = _arr(cams, np.float64).copy(), _arr(pts, np.float64).copy()
    oc, op, ouv, K = _arr(obs_cam, np.int32), _arr(obs_pt, np.int32), _arr(obs_uv, np.float32), _arr(K, np.float32)
    nw = len(cam_off) - 1
    opt = opt or ref.ba_options()
    sums = (ref.BASummary * nw)()
    _set_loss(loss)
    _load().orc_ba_local_batched(nw, _p(cam_off, C.c_int), _p(cams, C.c_double), _p(pt_off, C.c_int),
                                 _p(pts, C.c_double), _p(obs_off, C.c_int), _p(oc, C.c_int), _p(op, C.c_int),
                                 _p(ouv, C.c_float), _p(K, C.c_float), C.byref(opt), sums)
    return cams, pts, [s.as_dict() for s in sums]
