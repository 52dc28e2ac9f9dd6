"""TEST INFRASTRUCTURE ONLY: the local BA oracle with outlier rounds (ba_local_rounds_ref.cpp), for the
tests and profiles of lorb_ba_local_rounds_batched.  The library is the robust oracle of robust_ref.py
(oracle/ba_ref.cpp with ba_robust_ref.cpp spliced in) with per-residual weights added to its
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
_PATCH = os.path.join(_HERE, "ba_local_rounds_ref.cpp")
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
        out = os.path.join(tempfile.gettempdir(), "lorb_ba_local_rounds_ref_%s_%d.so" % (key, os.getuid()))
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
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


def _arr(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


def _set_loss(loss):
    kind, scale = (robust_ref.LOSS_TRIVIAL, 1.0) if loss is None else (int(loss[0]), float(loss[1]))
    _load().orc_ba_set_loss(kind, scale)


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
    """One window (the dict of robust_ref.ba_local) -> (cams, pts, obs_inlier[O] bool, obs_chi2[O],
    fix_inlier[F] bool, fix_chi2[F], n_inliers, summaries[n_rounds]) as Context.ba_local_rounds."""
    cams, pts = _arr(pb["cams"], np.float64).copy(), _arr(pb["pts"], np.float64).copy()
    oc, op, ouv = _arr(pb["obs_cam"], np.int32), _arr(pb["obs_pt"], np.int32), _arr(pb["obs_uv"], np.float32)
    fp, fuv = _arr(pb.get("fix_pt", []), np.int32), _arr(pb.get("fix_uv", []), np.float32)
    frt, K = _arr(pb.get("fix_rt", []), np.float32), _arr(pb["K"], np.float32).reshape(4)
    O, F = len(oc), len(fp)
    w = None if w is None else _arr(w, np.float32).reshape(O)
    fw = None if fix_w is None else _arr(fix_w, np.float32).reshape(F)
    opts = budgets(n_rounds, opt)
    inl, c2 = np.zeros(max(O, 1), np.uint8), np.zeros(max(O, 1), np.float64)
    finl, fc2 = np.zeros(max(F, 1), np.uint8), np.zeros(max(F, 1), np.float64)
    n_in = C.c_int()
    sums = (ref.BASummary * n_rounds)()
    optarr = (type(opts[0]) * n_rounds)(*opts)
    _set_loss(loss)
    rc = _load().orc_ba_local_rounds(
        len(cams), _p(cams, C.c_double), len(pts), _p(pts, C.c_double), O, _p(oc, C.c_int), _p(op, C.c_int),
        _p(ouv, C.c_float), _p(w, C.c_float), F, _p(fp, C.c_int), _p(fuv, C.c_float), _p(frt, C.c_float),
        _p(fw, C.c_float), _p(K, C.c_float), int(n_rounds), int(robust_rounds), C.c_double(chi2), int(depth_check),
        optarr, _p(inl, C.c_ubyte), _p(c2, C.c_double), _p(finl, C.c_ubyte), _p(fc2, C.c_double), C.byref(n_in),
        sums)
    assert rc == 0
    return (cams, pts, inl[:O].astype(bool), c2[:O], finl[:F].astype(bool), fc2[:F], n_in.value,
            [s.as_dict() for s in sums])
