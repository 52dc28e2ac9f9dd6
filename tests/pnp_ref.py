"""TEST INFRASTRUCTURE ONLY: the host restatement of lorb_pnp_ransac_batched (pnp_ref.cpp), compiled on first use
into the temporary directory (keyed by the sources' hash, never into the tree) with -O2 -ffp-contract=off, so its
arithmetic is the device's correctly rounded, uncontracted fp64."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(os.path.dirname(_HERE), "lorb_slam_b200", "csrc")
_SRC = os.path.join(_HERE, "pnp_ref.cpp")
_HDR = os.path.join(_CSRC, "pnp_math.cuh")
_lib = None


def _load():
    global _lib
    if _lib is None:
        key = hashlib.sha256(open(_SRC, "rb").read() + open(_HDR, "rb").read()).hexdigest()[:16]
        out = os.path.join(tempfile.gettempdir(), "lorb_pnp_ref_%s_%d.so" % (key, os.getuid()))
        if not os.path.exists(out):
            tmp = out + ".%d" % os.getpid()
            subprocess.run(["/usr/bin/g++", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
                            "-fopenmp", "-std=c++14", "-I", _CSRC, "-o", tmp, _SRC, "-lm"], check=True,
                           capture_output=True)
            os.replace(tmp, out)
        _lib = C.CDLL(out)
        _lib.pnr_draw4.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p]
        _lib.pnr_ransac.argtypes = [C.c_int] + [C.c_void_p] * 6 + [C.c_int, C.c_double] + [C.c_void_p] * 5
    return _lib


def _p(a):
    return C.c_void_p(a.ctypes.data) if a is not None and a.size else C.c_void_p(0)


def draw4(seed, h, n):
    """The four sample indices of hypothesis h, or None if the hypothesis is invalid."""
    idx = np.zeros(4, np.int32)
    ok = _load().pnr_draw4(int(seed), int(h), int(n), _p(idx))
    return idx if ok else None


def p3p(xw, uv, K):
    """Every P3P solution of three correspondences -> (R [k,3,3], t [k,3]) in solver order."""
    xw, uv = np.ascontiguousarray(xw, np.float32).reshape(3, 3), np.ascontiguousarray(uv, np.float32).reshape(3, 2)
    K = np.ascontiguousarray(K, np.float32).reshape(4)
    R, t = np.zeros((4, 9)), np.zeros((4, 3))
    k = _load().pnr_p3p(_p(xw), _p(uv), _p(K), _p(R), _p(t))
    return R[:k].reshape(k, 3, 3), t[:k]


def rotation_to_angle_axis(R):
    R = np.ascontiguousarray(R, np.float64).reshape(9)
    aa = np.zeros(3)
    _load().pnr_rotation_to_angle_axis(_p(R), _p(aa))
    return aa


def ransac(corr_off, xw, uv, K, info=None, seeds=None, n_hypotheses=300, chi2=5.991):
    """The same tuple as Context.pnp_ransac_batched: (rt[B,6], best_hyp[B], n_inliers[B], inlier[O] bool, chi2[O])."""
    co = np.ascontiguousarray(corr_off, np.int32).reshape(-1)
    xw, uv = np.ascontiguousarray(xw, np.float32).reshape(-1, 3), np.ascontiguousarray(uv, np.float32).reshape(-1, 2)
    K = np.ascontiguousarray(K, np.float32).reshape(4)
    w = None if info is None else np.ascontiguousarray(info, np.float32).reshape(-1)
    sd = None if seeds is None else np.ascontiguousarray(seeds, np.uint64).reshape(-1)
    B, O = len(co) - 1, len(xw)
    rt, best, n_in = np.zeros((B, 6)), np.zeros(B, np.int32), np.zeros(B, np.int32)
    inl, c2 = np.zeros(max(O, 1), np.uint8), np.zeros(max(O, 1))
    _load().pnr_ransac(B, _p(co), _p(xw), _p(uv), _p(w), _p(K), _p(sd), int(n_hypotheses), float(chi2), _p(rt),
                       _p(best), _p(n_in), _p(inl), _p(c2))
    return rt, best, n_in, inl[:O].astype(bool), c2[:O]
