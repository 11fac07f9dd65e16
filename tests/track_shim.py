"""TEST INFRASTRUCTURE: numpy-facing wrapper of tests/hostshim/libdfb_track_shim.so -- the host build of the per-pixel functions
of rigid point-to-TSDF tracking (csrc/dfb_track.h, see tests/hostshim/track_shim.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "hostshim", "track_shim.cpp")
_SO = os.path.join(_HERE, "hostshim", "libdfb_track_shim.so")
_ROOT = os.path.dirname(_HERE)


def build(force=False):
    csrc = os.path.join(_ROOT, "dynamicfusion_body_b200", "csrc")
    deps = [_SRC, os.path.join(csrc, "dfb_math.h"), os.path.join(csrc, "dfb_track.h"), os.path.join(_ROOT, "include", "dfb.h")]
    if not force and os.path.isfile(_SO) and all(os.path.getmtime(_SO) >= os.path.getmtime(d) for d in deps):
        return _SO
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", _SRC, "-o", _SO])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        vp, i, d = C.c_void_p, C.c_int, C.c_double
        _lib.ts_normal_eq.argtypes = [vp, vp, i, i, i, i, d, vp, vp, i, i, vp, vp, i, d, d, vp, vp, vp]
        _lib.ts_normal_eq.restype = i
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def normal_eq(tsdf, weight, tsdf_res, scale, center, depth, Kinv, lw34, stride, tdist, delta):
    """Host run of dfb_track_normal_eq: (sums (29,), residual (rows_s, cols_s) NaN = none, jac (rows_s, cols_s, 6) 0 = none)."""
    T = np.ascontiguousarray(tsdf, dtype=np.float32)
    W = np.ascontiguousarray(weight, dtype=np.float32)
    dm = np.ascontiguousarray(depth, dtype=np.float32)
    rows, cols = dm.shape
    rs, cs = (rows + stride - 1) // stride, (cols + stride - 1) // stride
    ctr = np.ascontiguousarray(center, dtype=np.float64).reshape(3)
    Ki = np.ascontiguousarray(Kinv, dtype=np.float64).reshape(9)
    lw = np.ascontiguousarray(lw34, dtype=np.float64).reshape(12)
    out = np.zeros(29)
    res = np.zeros((rs, cs))
    jac = np.zeros((rs, cs, 6))
    rc = lib().ts_normal_eq(_p(T), _p(W), T.shape[0], T.shape[1], T.shape[2], int(tsdf_res), float(scale), _p(ctr), _p(dm), rows, cols,
                            _p(Ki), _p(lw), int(stride), float(tdist), float(delta), _p(out), _p(res), _p(jac))
    assert rc == 0
    return out, res, jac
