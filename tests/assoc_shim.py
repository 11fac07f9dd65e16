"""TEST INFRASTRUCTURE: numpy-facing wrapper of tests/hostshim/libdfb_assoc_shim.so -- the host build of the per-vertex
function of projective data association (csrc/dfb_math.h assoc_projective_ref, see tests/hostshim/assoc_shim.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

import hostshim_api as hs
from dynamicfusion_body_b200 import _capi

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "hostshim", "assoc_shim.cpp")
_SO = os.path.join(_HERE, "hostshim", "libdfb_assoc_shim.so")
_ROOT = os.path.dirname(_HERE)


def build(force=False):
    deps = [_SRC, os.path.join(_ROOT, "dynamicfusion_body_b200", "csrc", "dfb_math.h"), os.path.join(_ROOT, "include", "dfb.h")]
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
        _lib.as_corr_projective.argtypes = [vp, vp, C.c_int64, C.POINTER(_capi.Views), C.c_double, C.c_double, vp, vp, vp]
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def corr_projective(warped_pts, warped_normals, depths, K, Kinv, max_distance, min_normal_dot, extrinsics=None):
    """Host run of dfb_corr_projective: (view (m,) int32, cost (m,) float64, corr (m,3) float64)."""
    wp = np.ascontiguousarray(warped_pts, dtype=np.float64).reshape(-1, 3)
    wn = np.ascontiguousarray(warped_normals, dtype=np.float64).reshape(-1, 3)
    views, keep = hs.make_views(depths, K, Kinv, extrinsics)
    m = len(wp)
    view = np.zeros(m, np.int32)
    cost = np.zeros(m)
    corr = np.zeros((m, 3))
    rc = lib().as_corr_projective(_p(wp), _p(wn), m, C.byref(views), float(max_distance), float(min_normal_dot), _p(view), _p(cost), _p(corr))
    assert rc == 0
    return view, cost, corr
