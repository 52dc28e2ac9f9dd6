"""TEST INFRASTRUCTURE ONLY: the BA oracle extended with robust losses, per-residual weights and
outlier rounds (ba_oracle_ext.cpp), for the tests and profiles of lorb_ba_set_loss,
lorb_ba_pose_rounds_batched and lorb_ba_local_rounds_batched.  The library is the oracle's own source
(oracle/ba_ref.cpp) with its linearize() / eval_cost() replaced by the weighted, loss-corrected forms
of ba_oracle_ext.cpp and the round drivers appended; it is compiled on first use into the temporary
directory (keyed by the sources' hash), never into the tree.

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
_PATCH = os.path.join(_HERE, "ba_oracle_ext.cpp")
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
        out = os.path.join(tempfile.gettempdir(), "lorb_ba_oracle_ext_%s_%d.so" % (key, os.getuid()))
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
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


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
    """pb's window at (cams, pts) -> (orc_ba_local's arguments C .. K, the arrays they point into)."""
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


def ba_pose_rounds(xw, uv, K, rt, info=None, n_rounds=4, robust_rounds=3, chi2=5.991, opt=None, loss=None):
    """One frame -> (rt, inlier[n] bool, chi2[n], n_inliers, rounds_run, summaries[n_rounds])."""
    xw, uv, K = _arr(xw, np.float32).reshape(-1, 3), _arr(uv, np.float32).reshape(-1, 2), _arr(K, np.float32).reshape(4)
    rt = _arr(rt, np.float64).reshape(6).copy()
    n = len(xw)
    w = None if info is None else _arr(info, np.float32).reshape(n)
    opt = opt or ref.ba_options()
    inl, c2 = np.zeros(max(n, 1), np.uint8), np.zeros(max(n, 1), np.float64)
    n_in, run = C.c_int(), C.c_int()
    sums = (ref.BASummary * n_rounds)()
    _set_loss(loss)
    assert _load().orc_ba_pose_rounds(n, _p(xw, C.c_float), _p(uv, C.c_float), _p(w, C.c_float), _p(K, C.c_float),
                                      _p(rt, C.c_double), int(n_rounds), int(robust_rounds), C.c_double(chi2),
                                      C.byref(opt), _p(inl, C.c_ubyte), _p(c2, C.c_double), C.byref(n_in),
                                      C.byref(run), sums) == 0
    return rt, inl[:n].astype(bool), c2[:n], n_in.value, run.value, [s.as_dict() for s in sums]


def ba_pose_rounds_batched(obs_off, xw, uv, K, rt, info=None, **kw):
    """Frame by frame; the same tuple as Context.ba_pose_rounds_batched."""
    obs_off = np.asarray(obs_off)
    xw, uv = _arr(xw, np.float32).reshape(-1, 3), _arr(uv, np.float32).reshape(-1, 2)
    rt = _arr(rt, np.float64).reshape(-1, 6)
    outs = []
    for f in range(len(rt)):
        a, b = int(obs_off[f]), int(obs_off[f + 1])
        outs.append(ba_pose_rounds(xw[a:b], uv[a:b], K, rt[f], None if info is None else np.asarray(info)[a:b], **kw))
    if not outs:
        return np.zeros((0, 6)), np.zeros(0, bool), np.zeros(0), np.zeros(0, np.int32), np.zeros(0, np.int32), []
    return (np.stack([o[0] for o in outs]), np.concatenate([o[1] for o in outs]), np.concatenate([o[2] for o in outs]),
            np.array([o[3] for o in outs], np.int32), np.array([o[4] for o in outs], np.int32), [o[5] for o in outs])


def budgets(n_rounds, opt):
    """opt: None (5 + 10 iterations for two rounds, else default options), one options struct for every
    round, or a list of n_rounds of them."""
    if opt is None:
        return [ref.ba_options(max_num_iterations=5), ref.ba_options(max_num_iterations=10)] if n_rounds == 2 \
            else [ref.ba_options() for _ in range(n_rounds)]
    if isinstance(opt, (list, tuple)):
        assert len(opt) == n_rounds
        return list(opt)
    return [opt] * n_rounds


def ba_local_rounds(pb, w=None, fix_w=None, n_rounds=2, robust_rounds=1, chi2=5.991, depth_check=1, opt=None,
                    loss=None):
    """One window (the dict of ba_local) -> (cams, pts, obs_inlier[O] bool, obs_chi2[O], fix_inlier[F] bool,
    fix_chi2[F], n_inliers, summaries[n_rounds]) as Context.ba_local_rounds."""
    cams, pts = _arr(pb["cams"], np.float64).copy(), _arr(pb["pts"], np.float64).copy()
    args, _keep = _local_args(pb, cams, pts)
    O, F = args[4], args[8]
    w = None if w is None else _arr(w, np.float32).reshape(O)
    fw = None if fix_w is None else _arr(fix_w, np.float32).reshape(F)
    opts = budgets(n_rounds, opt)
    inl, c2 = np.zeros(max(O, 1), np.uint8), np.zeros(max(O, 1), np.float64)
    finl, fc2 = np.zeros(max(F, 1), np.uint8), np.zeros(max(F, 1), np.float64)
    n_in = C.c_int()
    sums = (ref.BASummary * n_rounds)()
    optarr = (type(opts[0]) * n_rounds)(*opts)
    _set_loss(loss)
    # orc_ba_local's window arguments with the weights after obs_uv and after fix_rt
    rc = _load().orc_ba_local_rounds(*args[:8], _p(w, C.c_float), *args[8:12], _p(fw, C.c_float), args[12],
                                     int(n_rounds), int(robust_rounds), C.c_double(chi2), int(depth_check), optarr,
                                     _p(inl, C.c_ubyte), _p(c2, C.c_double), _p(finl, C.c_ubyte), _p(fc2, C.c_double),
                                     C.byref(n_in), sums)
    assert rc == 0
    return (cams, pts, inl[:O].astype(bool), c2[:O], finl[:F].astype(bool), fc2[:F], n_in.value,
            [s.as_dict() for s in sums])
