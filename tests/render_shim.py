"""TEST INFRASTRUCTURE: numpy-facing wrapper of tests/hostshim/libdfb_render_shim.so -- the host build of the per-face and
per-pixel functions of the z-buffer rasteriser (csrc/dfb_render.h, see tests/hostshim/render_shim.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

from dynamicfusion_body_b200 import _capi

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "hostshim", "render_shim.cpp")
_SO = os.path.join(_HERE, "hostshim", "libdfb_render_shim.so")
_ROOT = os.path.dirname(_HERE)


def build(force=False):
    csrc = os.path.join(_ROOT, "dynamicfusion_body_b200", "csrc")
    deps = [_SRC, os.path.join(csrc, "dfb_math.h"), os.path.join(csrc, "dfb_render.h"), os.path.join(_ROOT, "include", "dfb.h")]
    if not force and os.path.isfile(_SO) and all(os.path.getmtime(_SO) >= os.path.getmtime(d) for d in deps):
        return _SO
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", _SRC, "-o", _SO])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        vp = C.c_void_p
        _lib.rs_render.argtypes = [vp, C.c_int64, vp, C.c_int64, C.POINTER(_capi.Views), vp, vp, vp, vp]
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def camera_views(K, rows, cols, extrinsics=None, n_views=None):
    """dfb_views for rendering: intrinsics, optional (V,3,4) extrinsics and the image size; no depth maps."""
    v = _capi.Views()
    v.n_views = (1 if n_views is None else int(n_views)) if extrinsics is None else len(extrinsics)
    v.rows, v.cols = int(rows), int(cols)
    K = np.asarray(K, dtype=np.float64).ravel()
    for i in range(9):
        v.K[i] = float(K[i])
    v.has_extrinsics = 0 if extrinsics is None else 1
    if extrinsics is not None:
        E = np.asarray(extrinsics, dtype=np.float64).reshape(-1, 12)
        for j in range(v.n_views):
            for i in range(12):
                v.E[j][i] = float(E[j, i])
    return v


def render(pts, faces, K, rows, cols, extrinsics=None, n_views=None):
    """Host run of dfb_render: (depth (V,rows,cols) float32, face (V,rows,cols) int32, normal (V,rows,cols,3) float32)."""
    P = np.ascontiguousarray(pts, dtype=np.float64).reshape(-1, 3)
    F = np.ascontiguousarray(faces, dtype=np.int32).reshape(-1, 3)
    views = camera_views(K, rows, cols, extrinsics, n_views)
    V = views.n_views
    zbuf = np.zeros(V * rows * cols, np.uint64)
    depth = np.zeros((V, rows, cols), np.float32)
    face = np.zeros((V, rows, cols), np.int32)
    normal = np.zeros((V, rows, cols, 3), np.float32)
    rc = lib().rs_render(_p(P), len(P), _p(F), len(F), C.byref(views), _p(zbuf), _p(depth), _p(face), _p(normal))
    assert rc == 0
    return depth, face, normal
