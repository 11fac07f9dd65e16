"""TEST INFRASTRUCTURE: numpy-facing wrapper of tests/hostshim/libdfb_raycast_shim.so -- the host build of the per-ray function
of the raycaster (csrc/dfb_raycast.h and the tracker's functions of csrc/dfb_track.h, see tests/hostshim/raycast_shim.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

from dynamicfusion_body_b200 import _capi, engine

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "hostshim", "raycast_shim.cpp")
_SO = os.path.join(_HERE, "hostshim", "libdfb_raycast_shim.so")
_ROOT = os.path.dirname(_HERE)


def build(force=False):
    csrc = os.path.join(_ROOT, "dynamicfusion_body_b200", "csrc")
    deps = [_SRC, os.path.join(_ROOT, "include", "dfb.h")] + [os.path.join(csrc, h) for h in ("dfb_math.h", "dfb_track.h", "dfb_raycast.h")]
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
        _lib.rc_raycast.argtypes = [vp, vp, i, i, i, i, d, vp, C.POINTER(_capi.Views), d, d, d, d, vp, vp]
        _lib.rc_raycast.restype = i
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def raycast(tsdf, weight, tsdf_res, scale, center, tdist, K, rows, cols, extrinsics=None, step=None, z_near=0.0, z_far=None):
    """Host run of dfb_raycast with the arguments of oracle/raycast.py:raycast (views from engine.camera_views; z_far defaults to
    engine.raycast_far as in engine.raycast): (depth (V,rows,cols) float32, normal (V,rows,cols,3) float32)."""
    T = np.ascontiguousarray(tsdf, dtype=np.float32)
    W = np.ascontiguousarray(weight, dtype=np.float32)
    views = engine.camera_views(K, rows, cols, extrinsics)
    ctr = np.ascontiguousarray(center, dtype=np.float64).reshape(3)
    step = float(scale) if step is None else float(step)
    if z_far is None:
        z_far = max(engine.raycast_far(T.shape, tsdf_res, views, scale, ctr), z_near + step)
    V = views.n_views
    depth = np.zeros((V, rows, cols), np.float32)
    normal = np.zeros((V, rows, cols, 3), np.float32)
    rc = lib().rc_raycast(_p(T), _p(W), *T.shape, int(tsdf_res), float(scale), _p(ctr), C.byref(views), float(tdist), step,
                          float(z_near), float(z_far), _p(depth), _p(normal))
    assert rc == 0
    return depth, normal
