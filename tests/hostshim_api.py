"""TEST INFRASTRUCTURE: numpy-facing wrapper of tests/hostshim/libdfb_hostshim.so -- the host build of the kernels' per-element
logic and of the entry points' own argument checks and parameter set-up (see tests/hostshim/*.cpp).  Lets the CPU suite check the
arithmetic against the oracle without a GPU."""
import ctypes as C
import glob
import os
import subprocess

import numpy as np

from dynamicfusion_body_b200 import _capi, engine

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "hostshim", "libdfb_hostshim.so")
_ROOT = os.path.dirname(_HERE)


def build(force=False):
    srcs = sorted(glob.glob(os.path.join(_HERE, "hostshim", "*.cpp")))
    deps = [f for f in glob.glob(os.path.join(_HERE, "hostshim", "*")) if not f.endswith(".so")]
    deps += glob.glob(os.path.join(_ROOT, "dynamicfusion_body_b200", "csrc", "*.h")) + [os.path.join(_ROOT, "include", "dfb.h")]
    if not force and os.path.isfile(_SO) and all(os.path.getmtime(_SO) >= os.path.getmtime(d) for d in deps):
        return _SO
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared"] + srcs + ["-o", _SO])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        vp, i, d = C.c_void_p, C.c_int, C.c_double
        _lib.hs_last_error.restype = C.c_char_p
        _lib.hs_nodes_pack.argtypes = [vp, vp, vp, C.c_int, vp]
        _lib.hs_tsdf_update_projective.argtypes = [C.POINTER(_capi.Volume), C.POINTER(_capi.WarpField), C.POINTER(_capi.Views),
                                                   C.c_double, C.c_double, C.c_int, C.POINTER(_capi.Workspace), vp, vp, vp]
        _lib.hs_fuse_depth_rigid.argtypes = [C.POINTER(_capi.Volume), C.c_int, vp, C.c_int, C.c_int, vp, vp, vp, C.c_double,
                                             vp, C.c_double, C.c_double, C.c_int, C.POINTER(_capi.Workspace), vp, vp, vp]
        _lib.hs_tsdf_update_volume.argtypes = [C.POINTER(_capi.Volume), C.POINTER(_capi.WarpField), vp, C.c_int, C.c_int, C.c_int,
                                               C.c_double, C.c_double, C.c_int, C.POINTER(_capi.Workspace), vp, vp]
        _lib.hs_warp_points.argtypes = [vp, vp, C.c_int64, vp, C.POINTER(_capi.WarpField), vp, vp]
        _lib.hs_corr_projective.argtypes = [vp, vp, C.c_int64, C.POINTER(_capi.Views), d, d, vp, vp, vp]
        _lib.hs_render.argtypes = [vp, C.c_int64, vp, C.c_int64, C.POINTER(_capi.Views), vp, vp, vp]
        _lib.hs_track_normal_eq.argtypes = [C.POINTER(_capi.Volume), i, d, vp, vp, i, i, vp, vp, vp, i, d, d, vp, vp, vp]
        _lib.hs_raycast.argtypes = [C.POINTER(_capi.Volume), i, d, vp, C.POINTER(_capi.Views), d, d, d, d, vp, vp]
    return _lib


def set_bricks(knn=None, k=4, slab_shape=None, enable=True, use_pairs=True, regions=True):
    """Enable/disable the brick-culling emulation.  Returns the per-voxel brick-class array (0xFF = mixed) that the next
    update_projective / fuse_depth_rigid call fills."""
    L = lib()
    L.hs_brick_nodes_build.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    L.hs_set_bricks.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    L.hs_region_dmax.restype = C.c_float
    L.hs_region_valid.restype = C.c_float
    if not enable:
        L.hs_set_bricks(None, None, None, None, 0)
        return None
    sx, ry, rz = slab_shape
    nb = ((sx + 3) // 4) * ((ry + 3) // 4) * ((rz + 31) // 32)
    cls_vox = np.zeros(sx * ry * rz, np.uint8)
    keep = [cls_vox]
    if knn is not None:
        knn = np.ascontiguousarray(knn, dtype=np.uint16)
        nodes = np.zeros((nb, 24), np.uint16); count = np.zeros(nb, np.uint8); pairs = np.zeros((nb, 10), np.uint32)
        L.hs_brick_nodes_build(_p(knn), k, sx, ry, rz, _p(nodes), _p(count), _p(pairs))
        L.hs_set_bricks(_p(nodes), _p(count), _p(pairs) if use_pairs else None, _p(cls_vox), 1 if regions else 0)
        keep += [knn, nodes, count, pairs]
    else:
        L.hs_set_bricks(None, None, None, _p(cls_vox), 0)
    set_bricks._keep = keep
    return cls_vox


def region_stats():
    """(largest deviation bound among valid regions, fraction of valid regions) of the last region-enabled call."""
    return float(lib().hs_region_dmax()), float(lib().hs_region_valid())


def regions_resolved():
    """Number of regions the last region-enabled call classified as a whole (all their bricks inherit the class)."""
    return int(lib().hs_region_resolved())


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _check(rc):
    if rc != 0:
        raise RuntimeError("hostshim error %d: %s" % (rc, lib().hs_last_error().decode()))


class HostWarpField:
    def __init__(self, node_pos, node_dq, node_w, k, knn=None, lw=None):
        self.node_pos = np.ascontiguousarray(node_pos, dtype=np.float32)
        self.node_dq = np.ascontiguousarray(node_dq, dtype=np.float32)
        n = len(self.node_pos)
        self.node_w = np.ascontiguousarray(np.broadcast_to(np.asarray(node_w, dtype=np.float32), (n,)))
        self.rec = np.zeros((n, 12), dtype=np.float32)
        if n:
            lib().hs_nodes_pack(_p(self.node_pos), _p(self.node_dq), _p(self.node_w), n, _p(self.rec))
        self.k = k
        self.knn = None if knn is None else np.ascontiguousarray(knn, dtype=np.uint16)
        self.lw = lw

    def struct(self):
        s = _capi.WarpField()
        s.node_rec = self.rec.ctypes.data
        s.node_pos = self.node_pos.ctypes.data
        s.node_dq = self.node_dq.ctypes.data
        s.node_w = self.node_w.ctypes.data
        s.n_nodes = len(self.node_pos)
        s.k = self.k
        s.knn = self.knn.ctypes.data if self.knn is not None else None
        s.has_lw = 0 if self.lw is None else 1
        if self.lw is not None:
            s.lw_is_f32 = 1 if np.asarray(self.lw).dtype == np.float32 else 0
            for i in range(8):
                s.lw[i] = float(self.lw[i])
        return s


def _vol(tsdf, w, res, x0, x1):
    v = _capi.Volume()
    v.tsdf = tsdf.ctypes.data
    v.weight = w.ctypes.data
    v.rx, v.ry, v.rz = res
    v.x0, v.x1 = x0, x1
    return v


def _ws():
    counters = np.zeros(8, dtype=np.uint32)
    w = _capi.Workspace()
    w.list = None
    w.capacity = 0
    w.counters = counters.ctypes.data
    return w, counters


def _views(depths, K, Kinv, extrinsics=None):
    """engine.views_struct over host depth maps; returns it with the arrays it points into."""
    depths = [np.ascontiguousarray(d, dtype=np.float32) for d in depths]
    rows, cols = depths[0].shape
    return engine.views_struct(len(depths), rows, cols, K, Kinv, extrinsics, [d.ctypes.data for d in depths]), depths


def update_projective(tsdf, w, res, wf, depths, K, Kinv, tdist, extrinsics=None, wmax=100.0, mode=0, x0=0, x1=None):
    """tsdf, w: float32 slab arrays (modified in place). Returns (mask, frustum, cls, n_uncertain)."""
    x1 = res[0] if x1 is None else x1
    views, keep = _views(depths, K, Kinv, extrinsics)
    ws, counters = _ws()
    n = tsdf.size
    mask = np.zeros(n, np.uint8); frus = np.zeros(n, np.uint8); cls = np.zeros(n, np.uint8)
    vol = _vol(tsdf, w, res, x0, x1)
    s = wf.struct()
    _check(lib().hs_tsdf_update_projective(C.byref(vol), C.byref(s), C.byref(views), tdist, wmax, mode, C.byref(ws),
                                           _p(mask), _p(frus), _p(cls)))
    return mask, frus, cls, int(counters[0])


def fuse_depth_rigid(tsdf, w, res, tsdf_res, depth, lw34, K, Kinv, scale, center, tdist, wmax=100.0, mode=0, x0=0, x1=None):
    x1 = res[0] if x1 is None else x1
    depth = np.ascontiguousarray(depth, dtype=np.float32)
    lw34 = np.ascontiguousarray(lw34, dtype=np.float64); K = np.ascontiguousarray(K, dtype=np.float64)
    Kinv = np.ascontiguousarray(Kinv, dtype=np.float64); center = np.ascontiguousarray(center, dtype=np.float64)
    ws, counters = _ws()
    n = tsdf.size
    mask = np.zeros(n, np.uint8); frus = np.zeros(n, np.uint8); cls = np.zeros(n, np.uint8)
    vol = _vol(tsdf, w, res, x0, x1)
    _check(lib().hs_fuse_depth_rigid(C.byref(vol), tsdf_res, _p(depth), depth.shape[0], depth.shape[1], _p(lw34), _p(K), _p(Kinv),
                                     scale, _p(center), tdist, wmax, mode, C.byref(ws), _p(mask), _p(frus), _p(cls)))
    return mask, frus, cls, int(counters[0])


def update_volume(tsdf, w, res, wf, curr, tdist, wmax=100.0, mode=0, x0=0, x1=None):
    x1 = res[0] if x1 is None else x1
    curr = np.ascontiguousarray(curr, dtype=np.float32)
    ws, counters = _ws()
    n = tsdf.size
    mask = np.zeros(n, np.uint8); cls = np.zeros(n, np.uint8)
    vol = _vol(tsdf, w, res, x0, x1)
    s = wf.struct()
    _check(lib().hs_tsdf_update_volume(C.byref(vol), C.byref(s), _p(curr), curr.shape[0], curr.shape[1], curr.shape[2], tdist, wmax,
                                       mode, C.byref(ws), _p(mask), _p(cls)))
    return mask, cls, int(counters[0])


def warp_points(pts, normals, idx, wf):
    pts = np.ascontiguousarray(pts, dtype=np.float32)
    normals = None if normals is None else np.ascontiguousarray(normals, dtype=np.float32)
    idx = np.ascontiguousarray(idx, dtype=np.int32)
    out = np.zeros((len(pts), 3)); outn = np.zeros((len(pts), 3))
    s = wf.struct()
    _check(lib().hs_warp_points(_p(pts), _p(normals), len(pts), _p(idx), C.byref(s), _p(out), _p(outn)))
    return (out, outn) if normals is not None else out


def corr_projective(warped_pts, warped_normals, depths, K, Kinv, max_distance, min_normal_dot, extrinsics=None):
    """Host run of dfb_corr_projective: (view (m,) int32, cost (m,) float64, corr (m,3) float64)."""
    wp = np.ascontiguousarray(warped_pts, dtype=np.float64).reshape(-1, 3)
    wn = np.ascontiguousarray(warped_normals, dtype=np.float64).reshape(-1, 3)
    views, keep = _views(depths, K, Kinv, extrinsics)
    m = len(wp)
    view = np.zeros(m, np.int32)
    cost = np.zeros(m)
    corr = np.zeros((m, 3))
    _check(lib().hs_corr_projective(_p(wp), _p(wn), m, C.byref(views), float(max_distance), float(min_normal_dot), _p(view), _p(cost),
                                    _p(corr)))
    return view, cost, corr


def render(pts, faces, K, rows, cols, extrinsics=None, n_views=None):
    """Host run of dfb_render: (depth (V,rows,cols) float32, face (V,rows,cols) int32, normal (V,rows,cols,3) float32)."""
    P = np.ascontiguousarray(pts, dtype=np.float64).reshape(-1, 3)
    F = np.ascontiguousarray(faces, dtype=np.int32).reshape(-1, 3)
    views = engine.camera_views(K, rows, cols, extrinsics, n_views)
    V = views.n_views
    depth = np.zeros((V, rows, cols), np.float32)
    face = np.zeros((V, rows, cols), np.int32)
    normal = np.zeros((V, rows, cols, 3), np.float32)
    _check(lib().hs_render(_p(P), len(P), _p(F), len(F), C.byref(views), _p(depth), _p(face), _p(normal)))
    return depth, face, normal


def normal_eq(tsdf, weight, tsdf_res, scale, center, depth, Kinv, lw34, stride, tdist, delta):
    """Host run of dfb_track_normal_eq: (sums (29,), residual (rows_s, cols_s) NaN = none, jac (rows_s, cols_s, 6) 0 = none)."""
    T = np.ascontiguousarray(tsdf, dtype=np.float32)
    W = np.ascontiguousarray(weight, dtype=np.float32)
    dm = np.ascontiguousarray(depth, dtype=np.float32)
    rows, cols = dm.shape
    rs, cs = (rows + stride - 1) // stride, (cols + stride - 1) // stride
    ctr = np.ascontiguousarray(center, dtype=np.float64).reshape(3)
    Ki = np.ascontiguousarray(Kinv, dtype=np.float64).reshape(3, 3)
    K = np.linalg.inv(Ki)
    lw = np.ascontiguousarray(lw34, dtype=np.float64).reshape(12)
    out = np.zeros(29)
    res = np.zeros((rs, cs))
    jac = np.zeros((rs, cs, 6))
    vol = _vol(T, W, T.shape, 0, T.shape[0])
    _check(lib().hs_track_normal_eq(C.byref(vol), int(tsdf_res), float(scale), _p(ctr), _p(dm), rows, cols, _p(K), _p(Ki), _p(lw),
                                    int(stride), float(tdist), float(delta), _p(out), _p(res), _p(jac)))
    return out, res, jac


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
    vol = _vol(T, W, T.shape, 0, T.shape[0])
    _check(lib().hs_raycast(C.byref(vol), int(tsdf_res), float(scale), _p(ctr), C.byref(views), float(tdist), step, float(z_near),
                            float(z_far), _p(depth), _p(normal)))
    return depth, normal


# ---- Gauss-Newton path ------------------------------------------------------------------------------------------
class HostGN:
    """Host arrays + dfb_gn_problem struct for the hostshim GN entry points."""

    def __init__(self, vertices, normals, corr, vert_knn, node_pos, node_w, node_vertex_idx, lw, rw, huber=False, f_scale=1.0):
        self.vertices = np.ascontiguousarray(vertices, dtype=np.float32)
        self.normals = np.ascontiguousarray(normals, dtype=np.float32)
        self.corr = np.ascontiguousarray(corr, dtype=np.float64)
        self.vert_knn = np.ascontiguousarray(vert_knn, dtype=np.int32)
        self.node_pos = np.ascontiguousarray(node_pos, dtype=np.float32)
        n = len(self.node_pos)
        self.node_w = np.ascontiguousarray(np.broadcast_to(np.asarray(node_w, dtype=np.float32), (n,)))
        self.node_nbr = np.ascontiguousarray(self.vert_knn[np.asarray(node_vertex_idx)], dtype=np.int32)
        p = _capi.GNProblem()
        p.n_vert = len(self.vertices)
        p.vertices = self.vertices.ctypes.data; p.normals = self.normals.ctypes.data; p.corr = self.corr.ctypes.data
        p.vert_knn = self.vert_knn.ctypes.data
        p.n_nodes = n; p.k = self.vert_knn.shape[1]
        p.node_pos = self.node_pos.ctypes.data; p.node_w = self.node_w.ctypes.data; p.node_nbr = self.node_nbr.ctypes.data
        lw = np.asarray(lw)
        for i in range(8):
            p.lw[i] = float(lw[i])
        p.lw_is_f32 = 1 if lw.dtype == np.float32 else 0
        p.rw = rw; p.huber = 1 if huber else 0; p.f_scale = f_scale
        self.p = p
        L = lib()
        vp = C.c_void_p
        L.hs_gn_residuals.argtypes = [C.POINTER(_capi.GNProblem), vp, C.c_int, vp]
        L.hs_gn_residuals_lw.argtypes = [C.POINTER(_capi.GNProblem), vp, C.c_int, vp, C.c_int, vp]
        L.hs_gn_normal_eq_dense.argtypes = [C.POINTER(_capi.GNProblem), vp, vp, vp, vp]
        L.hs_gn_lw_normal_eq.argtypes = [C.POINTER(_capi.GNProblem), vp, vp, vp, vp, vp]

    def residuals(self, x):
        x = np.asarray(x)
        xd = np.ascontiguousarray(x, dtype=np.float64)
        f = np.zeros(self.p.n_vert + 3 * self.p.k * self.p.n_nodes)
        lib().hs_gn_residuals(C.byref(self.p), _p(xd), 1 if x.dtype == np.float32 else 0, _p(f))
        return f

    def residuals_lw(self, node_dq, lw):
        node_dq = np.asarray(node_dq); lw = np.asarray(lw)
        dqd = np.ascontiguousarray(node_dq, dtype=np.float64); lwd = np.ascontiguousarray(lw, dtype=np.float64)
        f = np.zeros(self.p.n_vert)
        lib().hs_gn_residuals_lw(C.byref(self.p), _p(dqd), 1 if node_dq.dtype == np.float32 else 0, _p(lwd),
                                 1 if lw.dtype == np.float32 else 0, _p(f))
        return f

    def normal_eq_dense(self, x):
        xd = np.ascontiguousarray(x, dtype=np.float64)
        n8 = 8 * self.p.n_nodes
        H = np.zeros((n8, n8)); g = np.zeros(n8); cost = np.zeros(2)
        lib().hs_gn_normal_eq_dense(C.byref(self.p), _p(xd), _p(H), _p(g), _p(cost))
        return H, g, cost

    def lw_normal_eq(self, node_dq, lw):
        dqd = np.ascontiguousarray(node_dq, dtype=np.float64); lwd = np.ascontiguousarray(lw, dtype=np.float64)
        H = np.zeros((8, 8)); g = np.zeros(8); cost = np.zeros(2)
        lib().hs_gn_lw_normal_eq(C.byref(self.p), _p(dqd), _p(lwd), _p(H), _p(g), _p(cost))
        return H, g, cost


def marching_cubes(vol, step_size=1, level=None, x_origin=0, plane_offsets=False):
    """Host run of csrc/dfb_mc.h in the composition of mc.cu (count -> scan -> emit); same arguments as engine.marching_cubes."""
    L = lib()
    vp = C.c_void_p
    vol = np.ascontiguousarray(vol, dtype=np.float32)
    rx, ry, rz = vol.shape
    s = int(step_size)
    L.hs_mc_level.restype = C.c_float
    L.hs_mc_level.argtypes = [vp, C.c_int64]
    L.hs_mc_count.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, vp, vp, vp]
    L.hs_mc_emit.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, vp, vp, vp, vp, vp, vp, vp]
    lv = L.hs_mc_level(_p(vol), vol.size) if level is None else float(np.float32(level))
    nx, ny, nz = (rx - 1) // s + 1, (ry - 1) // s + 1, (rz - 1) // s + 1
    rows, ncz = nx * ny, (nz + 31) // 32
    chunks = np.zeros((rows * ncz, 4), dtype=np.int32)
    voff = np.zeros(rows + 1, dtype=np.int32); toff = np.zeros(rows + 1, dtype=np.int32)
    L.hs_mc_count(_p(vol), rx, ry, rz, s, int(x_origin), lv, _p(chunks), _p(voff), _p(toff))
    nv, nt = int(voff[-1]), int(toff[-1])
    verts = np.zeros((nv, 3), np.float32); normals = np.zeros((nv, 3), np.float32); values = np.zeros(nv, np.float32)
    faces = np.zeros((nt, 3), np.int32)
    L.hs_mc_emit(_p(vol), rx, ry, rz, s, int(x_origin), lv, _p(chunks), _p(voff), _p(toff), _p(verts), _p(normals), _p(values), _p(faces))
    if plane_offsets:
        return verts, faces, normals, values, voff[::ny].astype(np.int64), toff[::ny].astype(np.int64)
    return verts, faces, normals, values
