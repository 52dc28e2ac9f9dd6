"""TEST INFRASTRUCTURE ONLY: the pose-only BA oracle with outlier rounds (ba_rounds_ref.cpp), for the
tests and profiles of lorb_ba_pose_rounds_batched.  The library is the robust oracle of robust_ref.py
(oracle/ba_ref.cpp with ba_robust_ref.cpp spliced in) with per-observation weights added to its
linearize() / eval_cost() and a C++ round driver; it is compiled on first use into the temporary
directory (keyed by the sources' hash), never into the tree.

loss: None (plain least squares) or (LOSS_*, scale a)."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import robust_ref
from oracle import ref

_HERE = os.path.dirname(os.path.abspath(__file__))
_PATCH = os.path.join(_HERE, "ba_rounds_ref.cpp")
_lib = None


def _source():
    src, patch = robust_ref._source(), open(_PATCH).read()
    part1, part2 = patch.split("// ---- part 2: appended after the oracle's C entry points\n")
    for name, sig in (("eval_cost", "(const Problem& pb, const double* cams, const double* pts) {"),
                      ("linearize", "(const Problem& pb, Lin& L) {")):
        old = "\ndouble %s%s" % (name, sig)
        assert src.count(old) == 1, name
        src = src.replace(old, "\ndouble robust_%s%s" % (name, sig))
    anchor = "\ninline bool has_cam("
    assert src.count(anchor) == 1
    src = src.replace(anchor, "\n" + part1 + anchor)
    return src + "\n" + part2


def _load():
    global _lib
    if _lib is None:
        src = _source()
        key = hashlib.sha256(src.encode()).hexdigest()[:16]
        out = os.path.join(tempfile.gettempdir(), "lorb_ba_rounds_ref_%s_%d.so" % (key, os.getuid()))
        if not os.path.exists(out):
            cpp = out[:-3] + ".cpp"
            with open(cpp, "w") as f:
                f.write(src)
            tmp = out + ".%d" % os.getpid()
            subprocess.run(["/usr/bin/g++", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
                            "-fopenmp", "-std=c++14", "-I", os.path.join(os.path.dirname(_HERE), "oracle"),
                            "-o", tmp, cpp, "-lm"], check=True, capture_output=True)
            os.replace(tmp, out)
        _lib = C.CDLL(out)
        _lib.orc_ba_set_loss.argtypes = [C.c_int, C.c_double]
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def _arr(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


def _set_loss(loss):
    kind, scale = (robust_ref.LOSS_TRIVIAL, 1.0) if loss is None else (int(loss[0]), float(loss[1]))
    _load().orc_ba_set_loss(kind, scale)


def ba_pose_only(xw, uv, K, rt, opt=None, loss=None):
    """One unweighted solve of this library (no rounds) -> (rt, summary)."""
    xw, uv, K = _arr(xw, np.float32).reshape(-1, 3), _arr(uv, np.float32).reshape(-1, 2), _arr(K, np.float32).reshape(4)
    rt = _arr(rt, np.float64).reshape(6).copy()
    opt = opt or ref.ba_options()
    s = ref.BASummary()
    _set_loss(loss)
    assert _load().orc_ba_pose_only(len(xw), _p(xw, C.c_float), _p(uv, C.c_float), _p(K, C.c_float),
                                    _p(rt, C.c_double), C.byref(opt), C.byref(s)) == 0
    return rt, s.as_dict()


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
    assert _load().orc_ba_pose_rounds(n, _p(xw, C.c_float), _p(uv, C.c_float),
                                      _p(w, C.c_float) if w is not None else None, _p(K, C.c_float),
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
