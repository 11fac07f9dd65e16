"""Device-resident state and thin launch wrappers over the C ABI (include/dfb.h).

torch is used for what it is good at here -- owning device memory, streams, and (in dist.py)
torch.distributed -- never for the arithmetic of the hot path.  Every function below ends in a call
into libdfb_b200.so on the current CUDA stream; there is no eager/torch/CPU fallback.
"""
import ctypes as C
import os

import numpy as np
import torch

from . import _capi


USE_REGIONS = True   # region reference maps (dfb_brick.h); False = per-brick pairwise hull + per-voxel DQB tier (validation)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _require_cuda(device):
    if not torch.cuda.is_available():
        raise RuntimeError("dynamicfusion_body_b200 needs a CUDA device (B200); there is no CPU path")
    return torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())


def _to_dev(a, dtype, device):
    if isinstance(a, torch.Tensor):
        return a.to(device=device, dtype=dtype).contiguous()
    a = np.ascontiguousarray(a)
    if not a.flags.writeable:
        a = a.copy()            # torch.from_numpy refuses to alias read-only buffers silently
    return torch.from_numpy(a).to(device=device, dtype=dtype).contiguous()


class Workspace:
    """Deferred-voxel list for the exact pass.  capacity defaults to 1/4 of the slab."""

    def __init__(self, n_voxels, device, fraction=0.25, n_bricks=0):
        self.capacity = int(max(1024, n_voxels * fraction))
        self.list = torch.empty(self.capacity, dtype=torch.int32, device=device)
        self.counters = torch.zeros(8, dtype=torch.int32, device=device)
        self.n_bricks = int(n_bricks)
        self.brick_cls = torch.zeros(4 * self.n_bricks, dtype=torch.uint8, device=device) if n_bricks else None
        self.brick_lists = torch.zeros(2 * self.n_bricks, dtype=torch.int32, device=device) if n_bricks else None
        # one bit per voxel for deferred voxels that find the list full (kept all-zero between calls by the exact pass)
        self.overflow_bits = torch.zeros((int(n_voxels) + 31) // 32, dtype=torch.int32, device=device)

    def struct(self, use_bricks=True):
        s = _capi.Workspace()
        s.list = self.list.data_ptr()
        s.capacity = self.capacity
        s.counters = self.counters.data_ptr()
        s.overflow_bits = self.overflow_bits.data_ptr()
        if use_bricks and self.brick_cls is not None:
            s.brick_cls = self.brick_cls.data_ptr()
            s.brick_lists = self.brick_lists.data_ptr()
        return s

    def _decode(self, c):
        c = c.astype(np.int64) & 0xffffffff
        return {"deferred": int(c[0]), "exact_processed": int(c[1]), "bricks_streamed": int(c[2]), "bricks_mixed": int(c[3]),
                "bricks": self.n_bricks, "dqb_voxels": int(c[4])}

    def stats(self):
        return self._decode(self.counters.cpu().numpy())

    def stats_async(self):
        """Start the 32-byte device->host read of the counters on the current stream (pinned buffer) and return a handle
        whose .result() waits for it: a streaming caller reads frame t's counters while frame t+1 is already queued."""
        if not hasattr(self, "_pinned"):
            self._pinned = [torch.empty(8, dtype=torch.int32).pin_memory() for _ in range(4)]
            self._pin_i = 0
        buf = self._pinned[self._pin_i % len(self._pinned)]
        self._pin_i += 1
        buf.copy_(self.counters, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        ws = self

        class _Pending:
            def result(self):
                ev.synchronize()
                return ws._decode(buf.numpy().copy())
        return _Pending()


class DeviceVolume:
    """(tsdf, weight) slab x in [x0,x1) of an (rx,ry,rz) grid, float32, C order (x slowest)."""

    def __init__(self, res, x0=0, x1=None, device=None, tsdf=None, weight=None, fill=None):
        self.device = _require_cuda(device)
        self.res = tuple(int(r) for r in res)
        self.x0 = int(x0)
        self.x1 = int(self.res[0] if x1 is None else x1)
        shape = (self.x1 - self.x0, self.res[1], self.res[2])
        if tsdf is not None:
            self.tsdf = _to_dev(tsdf, torch.float32, self.device).reshape(shape)
        else:
            self.tsdf = torch.full(shape, float(fill if fill is not None else 0.0), dtype=torch.float32, device=self.device)
        if weight is not None:
            self.weight = _to_dev(weight, torch.float32, self.device).reshape(shape)
        else:
            self.weight = torch.zeros(shape, dtype=torch.float32, device=self.device)
        nb = int(_capi.lib().dfb_brick_count(self.x1 - self.x0, self.res[1], self.res[2]))
        self.workspace = Workspace(self.n_voxels, self.device, n_bricks=nb)

    @property
    def n_voxels(self):
        return (self.x1 - self.x0) * self.res[1] * self.res[2]

    def struct(self):
        s = _capi.Volume()
        s.tsdf = self.tsdf.data_ptr()
        s.weight = self.weight.data_ptr()
        s.rx, s.ry, s.rz = self.res
        s.x0, s.x1 = self.x0, self.x1
        return s


class DeviceWarpField:
    """Deformation nodes (dg_v, dg_se3, dg_w of core/fusion.py:113-116) as device SoA + packed records,
    and the cached voxel kNN table (valid until the node POSITIONS change, i.e. until update_graph)."""

    def __init__(self, k, device=None):
        self.device = _require_cuda(device)
        self.k = int(k)
        self.n_nodes = 0
        self.node_pos = self.node_dq = self.node_w = self.node_rec = None
        self._knn = {}
        self._knn_radii = {}
        self._bricks = {}

    def set_nodes(self, node_pos, node_dq, node_w):
        n = len(node_pos)
        self.node_pos = _to_dev(node_pos, torch.float32, self.device).reshape(n, 3)
        w = np.broadcast_to(np.asarray(node_w, dtype=np.float32), (n,)) if not isinstance(node_w, torch.Tensor) else node_w
        self.node_w = _to_dev(w, torch.float32, self.device).reshape(n)
        self.n_nodes = n
        self._knn = {}
        self._knn_radii = {}
        self._bricks = {}
        self.node_dq = None
        self.set_dq(node_dq)

    def set_dq(self, node_dq):
        """Only the transforms changed (e.g. after solve): repack records, keep the kNN tables.  The device buffers keep their
        addresses while the node count stays the same (a captured frame step refers to them)."""
        if (self.node_dq is not None and tuple(self.node_dq.shape) == (self.n_nodes, 8)
                and (isinstance(node_dq, torch.Tensor) or isinstance(node_dq, np.ndarray))):
            src = node_dq if isinstance(node_dq, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(node_dq, dtype=np.float32))
            if src.data_ptr() != self.node_dq.data_ptr():
                self.node_dq.copy_(src.reshape(self.n_nodes, 8), non_blocking=True)
        else:
            self.node_dq = _to_dev(node_dq, torch.float32, self.device).reshape(self.n_nodes, 8)
        self.repack()

    def repack(self):
        if self.node_rec is None or self.node_rec.shape[0] != self.n_nodes:
            self.node_rec = torch.empty((self.n_nodes, _capi.DFB_NODE_REC_FLOATS), dtype=torch.float32, device=self.device)
        _capi.check(_capi.lib().dfb_nodes_pack(_ptr(self.node_pos), _ptr(self.node_dq), _ptr(self.node_w), self.n_nodes,
                                               _ptr(self.node_rec), _stream()))

    def knn_table(self, res, x0, x1):
        """uint16 [(x1-x0)*ry*rz, k] (stored in an int16 tensor), built on first use (with the per-brick search radii that
        `append_nodes` needs to bring it up to date incrementally)."""
        key = (tuple(res), x0, x1)
        t = self._knn.get(key)
        if t is None:
            n = (x1 - x0) * res[1] * res[2]
            t = torch.empty((n, self.k), dtype=torch.int16, device=self.device)
            L = _capi.lib()
            if os.environ.get("DFB_KNN_BRUTE"):                     # validation: the O(voxels * nodes) kernel, no radii
                _capi.check(L.dfb_knn_build_volume(_ptr(self.node_pos), self.n_nodes, self.k, res[0], res[1], res[2], x0, x1, _ptr(t), _stream()))
            else:
                radii = torch.empty(int(L.dfb_knn_brick_count(x1 - x0, res[1], res[2])), dtype=torch.float32, device=self.device)
                _capi.check(L.dfb_knn_build_volume_radii(_ptr(self.node_pos), self.n_nodes, self.k, res[0], res[1], res[2], x0, x1, _ptr(t),
                                                         _ptr(radii), _stream()))
                self._knn_radii[key] = radii
            self._knn[key] = t
        return t

    def append_nodes(self, node_pos, node_dq, node_w):
        """A graph revision that only APPENDS nodes (what update_graph does, core/fusion.py:216-229): the cached voxel kNN tables and
        the brick / region candidate sets are brought up to date incrementally -- only the 8^3 bricks a new node can reach are
        rebuilt (dfb_knn_update_volume), everything else stays.  Same tables as a full rebuild, bit for bit."""
        m = len(node_pos)
        if m == 0:
            return
        n_old = self.n_nodes
        new_pos = _to_dev(node_pos, torch.float32, self.device).reshape(m, 3)
        new_dq = _to_dev(node_dq, torch.float32, self.device).reshape(m, 8)
        w = np.broadcast_to(np.asarray(node_w, dtype=np.float32), (m,)) if not isinstance(node_w, torch.Tensor) else node_w
        new_w = _to_dev(w, torch.float32, self.device).reshape(m)
        self.node_pos = torch.cat([self.node_pos, new_pos]).contiguous()
        self.node_w = torch.cat([self.node_w, new_w]).contiguous()
        dq = torch.cat([self.node_dq, new_dq]).contiguous()
        self.n_nodes = n_old + m
        self.node_dq = None
        self.set_dq(dq)
        L = _capi.lib()
        for key, t in list(self._knn.items()):
            res, x0, x1 = key
            radii = self._knn_radii.get(key)
            if radii is None or n_old < self.k:                      # no radii on record (brute-force build): rebuild on demand
                del self._knn[key]
                self._bricks.pop(key, None)
                continue
            dirty = torch.empty(radii.numel(), dtype=torch.uint8, device=self.device)
            _capi.check(L.dfb_knn_update_volume(_ptr(self.node_pos), n_old, self.n_nodes, self.k, res[0], res[1], res[2], x0, x1, _ptr(t),
                                                _ptr(radii), _ptr(dirty), _stream()))
            self.last_dirty = dirty
            b = self._bricks.get(key)
            if b is not None:
                nodes, count, pairs, rnodes, rcount, rpairs, rrec = b
                _capi.check(L.dfb_brick_nodes_update(_ptr(t), self.k, res[0], res[1], res[2], x0, x1, _ptr(dirty), _ptr(nodes), _ptr(count),
                                                     _ptr(pairs), _stream()))
                _capi.check(L.dfb_region_update(_ptr(t), self.k, res[0], res[1], res[2], x0, x1, _ptr(dirty), _ptr(rnodes), _ptr(rcount),
                                                _ptr(rpairs), _stream()))

    def brick_nodes(self, res, x0, x1):
        """(nodes uint16 [n_bricks,24], count uint8 [n_bricks]): union of the kNN sets of each 4x4x32 brick; cached with
        the kNN table (same validity: until the node positions change)."""
        key = (tuple(res), x0, x1)
        t = self._bricks.get(key)
        if t is None:
            knn = self.knn_table(res, x0, x1)
            nb = int(_capi.lib().dfb_brick_count(x1 - x0, res[1], res[2]))
            nodes = torch.zeros((nb, 24), dtype=torch.int16, device=self.device)
            count = torch.zeros(nb, dtype=torch.uint8, device=self.device)
            pairs = torch.zeros((nb, 10), dtype=torch.int32, device=self.device)
            _capi.check(_capi.lib().dfb_brick_nodes_build(_ptr(knn), self.k, res[0], res[1], res[2], x0, x1, _ptr(nodes), _ptr(count),
                                                          _ptr(pairs), _stream()))
            nr = int(_capi.lib().dfb_region_count(x1 - x0, res[1], res[2]))
            rnodes = torch.zeros((nr, 64), dtype=torch.int16, device=self.device)
            rcount = torch.zeros(nr, dtype=torch.uint8, device=self.device)
            rpairs = torch.zeros((nr, 65), dtype=torch.int32, device=self.device)
            rrec = torch.zeros((nr, 32), dtype=torch.float32, device=self.device)
            _capi.check(_capi.lib().dfb_region_build(_ptr(knn), self.k, res[0], res[1], res[2], x0, x1, _ptr(rnodes), _ptr(rcount),
                                                     _ptr(rpairs), _stream()))
            t = (nodes, count, pairs, rnodes, rcount, rpairs, rrec)
            self._bricks[key] = t
        return t

    def knn_points(self, pts, k=None):
        k = self.k if k is None else k
        p = _to_dev(pts, torch.float32, self.device).reshape(-1, 3)
        out = torch.empty((p.shape[0], k), dtype=torch.int32, device=self.device)
        _capi.check(_capi.lib().dfb_knn_points(_ptr(p), p.shape[0], _ptr(self.node_pos), self.n_nodes, k, _ptr(out), _stream()))
        return out

    def struct(self, lw=None, knn=None, k=None, bricks=None):
        s = _capi.WarpField()
        if bricks is not None:
            s.brick_nodes = bricks[0].data_ptr()
            s.brick_count = bricks[1].data_ptr()
            s.brick_pairs = bricks[2].data_ptr()
            if USE_REGIONS:
                s.region_nodes = bricks[3].data_ptr()
                s.region_count = bricks[4].data_ptr()
                s.region_pairs = bricks[5].data_ptr()
                s.region_rec = bricks[6].data_ptr()
        k = self.k if k is None else k
        if k > 0:
            s.node_rec = self.node_rec.data_ptr()
            s.node_pos = self.node_pos.data_ptr()
            s.node_dq = self.node_dq.data_ptr()
            s.node_w = self.node_w.data_ptr()
        s.n_nodes = self.n_nodes
        s.k = k
        s.knn = knn.data_ptr() if knn is not None else None
        fill_lw(s, lw)
        return s


def fill_lw(s, lw):
    """lw: None, or an 8-vector; a float32 numpy array keeps the reference's float32 dtype flow (Q3)."""
    s.has_lw = 0 if lw is None else 1
    s.lw_is_f32 = 0
    if lw is not None:
        if isinstance(lw, torch.Tensor):
            lw = lw.detach().cpu().numpy()
        lw = np.asarray(lw)
        s.lw_is_f32 = 1 if lw.dtype == np.float32 else 0
        for i in range(8):
            s.lw[i] = float(lw[i])


def make_views(depths, K, Kinv=None, extrinsics=None):
    """depths: CUDA float32 tensor (V,rows,cols) (negative depth, 0 = no data)."""
    if depths.dim() == 2:
        depths = depths[None]
    assert depths.is_cuda and depths.dtype == torch.float32 and depths.is_contiguous()
    K = np.asarray(K, dtype=np.float64)
    Kinv = np.linalg.inv(K) if Kinv is None else np.asarray(Kinv, dtype=np.float64)
    v = _capi.Views()
    v.n_views = depths.shape[0]
    if v.n_views > _capi.DFB_MAX_VIEWS:
        raise ValueError("at most %d views per pass" % _capi.DFB_MAX_VIEWS)
    for i in range(v.n_views):
        v.depth[i] = depths[i].data_ptr()
    v.rows, v.cols = int(depths.shape[1]), int(depths.shape[2])
    for i in range(9):
        v.K[i] = float(K.ravel()[i])
        v.Kinv[i] = float(Kinv.ravel()[i])
    v.has_extrinsics = 0 if extrinsics is None else 1
    if extrinsics is not None:
        E = np.asarray(extrinsics, dtype=np.float64).reshape(v.n_views, 12)
        for j in range(v.n_views):
            for i in range(12):
                v.E[j][i] = float(E[j, i])
    return v


def _mask_bufs(vol, want):
    if not want:
        return None, None
    return (torch.zeros(vol.n_voxels, dtype=torch.uint8, device=vol.device),
            torch.zeros(vol.n_voxels, dtype=torch.uint8, device=vol.device))


def update_projective(vol, wf, lw, depths, K, Kinv=None, extrinsics=None, tdist=1.0, wmax=100.0,
                      mode=_capi.MODE_HYBRID, want_masks=False, views=None, use_bricks=True):
    """a3: warped projective TSDF update of the slab `vol` in place; returns (mask, frustum) bit-arrays or None."""
    views = views if views is not None else make_views(depths, K, Kinv, extrinsics)
    knn = wf.knn_table(vol.res, vol.x0, vol.x1)
    bricks = wf.brick_nodes(vol.res, vol.x0, vol.x1) if use_bricks else None
    ws = vol.workspace.struct(use_bricks)
    mask, frus = _mask_bufs(vol, want_masks)
    v = vol.struct()
    s = wf.struct(lw, knn, bricks=bricks)
    _capi.check(_capi.lib().dfb_tsdf_update_projective(C.byref(v), C.byref(s), C.byref(views), float(tdist), float(wmax),
                                                       int(mode), C.byref(ws), _ptr(mask), _ptr(frus), _stream()))
    return (mask, frus) if want_masks else None


def update_volume(vol, wf, lw, curr, tdist, wmax=100.0, mode=_capi.MODE_HYBRID, want_masks=False, rigid=False):
    """a1: Fusion.updateTSDF (or FusionDM.updateTSDF when rigid=True) on the slab in place."""
    assert curr.is_cuda and curr.dtype == torch.float32 and curr.is_contiguous() and curr.dim() == 3
    k = 0 if rigid else wf.k
    knn = None if rigid else wf.knn_table(vol.res, vol.x0, vol.x1)
    ws = vol.workspace.struct(False)
    mask = torch.zeros(vol.n_voxels, dtype=torch.uint8, device=vol.device) if want_masks else None
    v = vol.struct()
    s = wf.struct(lw, knn, k=k) if wf is not None else _rigid_struct(lw)
    _capi.check(_capi.lib().dfb_tsdf_update_volume(C.byref(v), C.byref(s), _ptr(curr), curr.shape[0], curr.shape[1],
                                                   curr.shape[2], float(tdist), float(wmax), int(mode), C.byref(ws),
                                                   _ptr(mask), _stream()))
    return mask


def _rigid_struct(lw):
    s = _capi.WarpField()
    s.k = 0
    fill_lw(s, lw)
    return s


def fuse_depth_rigid(vol, tsdf_res, depth, lw34, K, Kinv=None, scale=1.0, center=None, tdist=1.0, wmax=100.0,
                     mode=_capi.MODE_HYBRID, want_masks=False, use_bricks=True):
    """a2: FusionDM.fuseDepths on the slab in place."""
    assert depth.is_cuda and depth.dtype == torch.float32 and depth.is_contiguous() and depth.dim() == 2
    K = np.ascontiguousarray(K, dtype=np.float64)
    Kinv = np.ascontiguousarray(np.linalg.inv(K) if Kinv is None else Kinv, dtype=np.float64)
    lw34 = np.ascontiguousarray(lw34, dtype=np.float64).reshape(12)
    center = np.ascontiguousarray(np.zeros(3) if center is None else center, dtype=np.float64)
    ws = vol.workspace.struct(use_bricks)
    mask, frus = _mask_bufs(vol, want_masks)
    v = vol.struct()
    f64 = _capi.c_f64p
    _capi.check(_capi.lib().dfb_fuse_depth_rigid(C.byref(v), int(tsdf_res), _ptr(depth), depth.shape[0], depth.shape[1],
                                                 lw34.ctypes.data_as(f64), K.ctypes.data_as(f64), Kinv.ctypes.data_as(f64),
                                                 float(scale), center.ctypes.data_as(f64), float(tdist), float(wmax), int(mode),
                                                 C.byref(ws), _ptr(mask), _ptr(frus), _stream()))
    return (mask, frus) if want_masks else None


def warp_points(wf, lw, pts, normals=None, idx=None, k=None):
    """a4: Fusion.warp for float32 points; returns float64 CUDA tensors."""
    dev = wf.device
    p = _to_dev(pts, torch.float32, dev).reshape(-1, 3)
    n = None if normals is None else _to_dev(normals, torch.float32, dev).reshape(-1, 3)
    k = wf.k if k is None else k
    if k > 0:
        idx = wf.knn_points(p, k) if idx is None else _to_dev(idx, torch.int32, dev).reshape(-1, k)
    out = torch.empty((p.shape[0], 3), dtype=torch.float64, device=dev)
    outn = torch.empty((p.shape[0], 3), dtype=torch.float64, device=dev) if n is not None else None
    s = wf.struct(lw, None, k=k)
    _capi.check(_capi.lib().dfb_warp_points(_ptr(p), _ptr(n), p.shape[0], _ptr(idx), C.byref(s), _ptr(out), _ptr(outn), _stream()))
    return (out, outn) if n is not None else out


# ---- SURVEY 8f ranks 1-2: point-set search, correspondences, graph maintenance (csrc/graph.cu) -----------------
class PointGrid:
    """Uniform search grid over a float32 point set on the device: the stand-in for the scipy KDTree the reference
    builds over live / canonical surface vertices (core/fusion.py:204,255,308; core/fusion_dm.py:226).  Exact results
    (float64 distances, ties by lower id); the cell size only affects speed."""

    MAX_CELLS = 1 << 24

    def __init__(self, pts, cell=None, device=None):
        dev = _require_cuda(device)
        self.device = dev
        self.pts = _to_dev(pts, torch.float32, dev).reshape(-1, 3)
        n = self.pts.shape[0]
        if n:
            lo = self.pts.amin(0).double().cpu().numpy()
            hi = self.pts.amax(0).double().cpu().numpy()
        else:
            lo = hi = np.zeros(3)
        ext = np.maximum(hi - lo, 1e-6)
        if cell is None:
            # surface samples: about sqrt(n) of them along the longest extent -> a few points per occupied cell ...
            cell = float(ext.max()) / float(min(256, max(4, int(round(np.sqrt(max(n, 1)) / 2)))))
            # ... but no more than ~8 cells per point (most cells of a surface's bounding box are empty; measured at
            # 300 k points: 13.7 M cells -> build 6.5 ms, query 0.52 ms; 1.9 M cells -> 1.0 / 0.64 ms)
            cell = max(cell, float(np.cbrt(ext.prod() / (8.0 * max(n, 1)))))
        cell = float(cell)
        while True:
            dims = np.floor(ext / cell).astype(np.int64) + 1
            if int(dims.prod()) <= self.MAX_CELLS:
                break
            cell *= 1.26
        self.cell, self.origin, self.dims = cell, lo, [int(d) for d in dims]
        cells = int(dims.prod())
        self.cell_start = torch.empty(cells + 1, dtype=torch.int32, device=dev)
        self.order = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
        scratch = torch.empty(int(_capi.lib().dfb_point_grid_scratch_ints(cells)), dtype=torch.int32, device=dev)
        if n == 0:
            self.pts = torch.zeros((1, 3), dtype=torch.float32, device=dev)   # a valid pointer; n stays 0
        self.n = n
        _capi.check(_capi.lib().dfb_point_grid_build(C.byref(self.struct()), _ptr(self.cell_start), _ptr(self.order), _ptr(scratch), _stream()))

    def struct(self):
        s = _capi.PointGrid()
        s.pts = self.pts.data_ptr()
        s.n = self.n
        for i in range(3):
            s.origin[i] = float(self.origin[i])
            s.dims[i] = self.dims[i]
        s.cell = self.cell
        s.cell_start = self.cell_start.data_ptr()
        s.order = self.order.data_ptr()
        return s

    def knn(self, queries, k, want_d2=False):
        """KDTree.query(q, k)[1] for (m,3) float64 queries: (m,k) int32, ascending distance."""
        q = _to_dev(queries, torch.float64, self.device).reshape(-1, 3)
        idx = torch.empty((q.shape[0], k), dtype=torch.int32, device=self.device)
        d2 = torch.empty((q.shape[0], k), dtype=torch.float64, device=self.device) if want_d2 else None
        _capi.check(_capi.lib().dfb_point_grid_knn(C.byref(self.struct()), _ptr(q), q.shape[0], k, _ptr(idx), _ptr(d2), _stream()))
        return (idx, d2) if want_d2 else idx


def corr_select(warped_pts, warped_normals, live_verts, nn):
    """Best-of-k point-to-plane candidate (core/fusion.py:264-274): returns (best index (m,) int32, best cost (m,) float64)."""
    dev = nn.device
    wv = _to_dev(warped_pts, torch.float64, dev).reshape(-1, 3)
    wn = _to_dev(warped_normals, torch.float64, dev).reshape(-1, 3)
    lv = _to_dev(live_verts, torch.float32, dev).reshape(-1, 3)
    best = torch.empty(wv.shape[0], dtype=torch.int32, device=dev)
    cost = torch.empty(wv.shape[0], dtype=torch.float64, device=dev)
    _capi.check(_capi.lib().dfb_corr_select(_ptr(wv), _ptr(wn), wv.shape[0], _ptr(lv), _ptr(nn), nn.shape[1], _ptr(best), _ptr(cost), _stream()))
    return best, cost


def corr_projective(warped_pts, warped_normals, views, max_distance, min_normal_dot):
    """Projective data association of warped canonical points / normals (float64, as `warp_points` returns them) against the
    depth views of `make_views`: returns (view (m,) int32, -1 = none; cost (m,) float64, +inf = none; corr (m,3) float64, the
    live point in the frame of the warped points, 0 = none) as CUDA tensors."""
    dev = warped_pts.device if isinstance(warped_pts, torch.Tensor) and warped_pts.is_cuda else _require_cuda(None)
    wv = _to_dev(warped_pts, torch.float64, dev).reshape(-1, 3)
    wn = _to_dev(warped_normals, torch.float64, dev).reshape(-1, 3)
    m = wv.shape[0]
    view = torch.empty(m, dtype=torch.int32, device=dev)
    cost = torch.empty(m, dtype=torch.float64, device=dev)
    corr = torch.empty((m, 3), dtype=torch.float64, device=dev)
    _capi.check(_capi.lib().dfb_corr_projective(_ptr(wv), _ptr(wn), m, C.byref(views), float(max_distance), float(min_normal_dot),
                                                _ptr(view), _ptr(cost), _ptr(corr), _stream()))
    return view, cost, corr


def graph_unsupported(wf, verts, vert_knn):
    """core/fusion.py:211-215: bool (m,) -- surface points no node of `wf` supports."""
    dev = wf.device
    v = _to_dev(verts, torch.float32, dev).reshape(-1, 3)
    kn = _to_dev(vert_knn, torch.int32, dev).reshape(v.shape[0], -1)
    out = torch.empty(v.shape[0], dtype=torch.uint8, device=dev)
    _capi.check(_capi.lib().dfb_graph_unsupported(_ptr(v), v.shape[0], _ptr(kn), kn.shape[1], _ptr(wf.node_pos), _ptr(wf.node_w), _ptr(out), _stream()))
    return out.bool()


def uniform_sample(pts, radius, device=None, rounds_per_call=16):
    """`uniform_sample` (core/util.py:27-47) on the device: returns (samples (s,3) float32 numpy, indices (s,) int64 numpy),
    identical to the sequential greedy sampler (parallel lexicographic maximal independent set, csrc/graph.cu)."""
    dev = _require_cuda(device)
    p = _to_dev(pts, torch.float32, dev).reshape(-1, 3)
    n = p.shape[0]
    if n == 0:
        return np.zeros((0, 3), np.float32), np.zeros(0, np.int64)
    grid = PointGrid(p, cell=float(radius) * 1.001, device=dev)      # just above the radius: the 3x3x3 cell neighbourhood covers the ball
    state = torch.zeros(n, dtype=torch.uint8, device=dev)
    undecided = torch.ones(1, dtype=torch.int32, device=dev)
    s = grid.struct()
    while True:
        _capi.check(_capi.lib().dfb_graph_sample_rounds(C.byref(s), float(radius), rounds_per_call, _ptr(state), _ptr(undecided), _stream()))
        if int(undecided.item()) == 0:
            break
    idx = torch.nonzero(state == 1).reshape(-1)
    return p[idx].cpu().numpy(), idx.cpu().numpy().astype(np.int64)


def marching_cubes(vol, step_size=1, level=None, x_origin=0, plane_offsets=False, keep_on_device=False):
    """Surface extraction on the device (SURVEY 8f rank 3; include/dfb.h `dfb_mc_*`): the call the reference makes as
    measure.marching_cubes_lewiner(volume, step_size=..., allow_degenerate=False) (core/fusion.py:554-568, 579).
    vol: (rx, ry, rz) CUDA tensor or host array; level None = 0.5 * (min + max) like skimage.  Returns host arrays
    (verts (V,3) float32 voxel coordinates, faces (F,3) int32, normals (V,3) float32, values (V,) float32).
    x_origin: sample index (voxel x / step) of vol[0] in the whole grid when `vol` is an x-slab -- coordinates and degenerate-triangle
    decisions are then those of the whole grid.  plane_offsets=True appends (plane_voff, plane_toff), int64 [nx + 1]: first vertex /
    triangle of every sample x-plane (vertices are ordered by owning sample, triangles by cell, x slowest) -- what
    dist.extract_surface_slab cuts the halo planes off with.  keep_on_device=True returns CUDA tensors instead of host arrays."""
    if not isinstance(vol, torch.Tensor):
        vol = _to_dev(np.asarray(vol), torch.float32, _require_cuda(None))
    if vol.dim() != 3:
        raise ValueError("marching_cubes needs a 3-D volume")
    step = int(step_size)
    if step < 1:
        raise ValueError("step_size must be >= 1")
    if not vol.is_cuda:
        vol = vol.to(_require_cuda(None))
    vol = vol.to(dtype=torch.float32).contiguous()
    rx, ry, rz = (int(n) for n in vol.shape)
    if min(rx, ry, rz) < 2:
        raise ValueError("marching_cubes needs at least 2 samples per axis")
    L = _capi.lib()
    dev = vol.device
    with torch.cuda.device(dev):
        lv = torch.empty(3, dtype=torch.float32, device=dev)
        if level is None:
            scratch = torch.empty(int(L.dfb_mc_level_scratch_floats()), dtype=torch.float32, device=dev)
            _capi.check(L.dfb_mc_level(_ptr(vol), vol.numel(), _ptr(scratch), _ptr(lv), _stream()))
        else:
            lv.fill_(float(np.float32(level)))
        rows = int(L.dfb_mc_rows(rx, ry, step))
        chunks = torch.empty((int(L.dfb_mc_chunks(rx, ry, rz, step)), 4), dtype=torch.int32, device=dev)
        offs = torch.empty((2, rows + 1), dtype=torch.int32, device=dev)
        _capi.check(L.dfb_mc_count(_ptr(vol), rx, ry, rz, step, int(x_origin), _ptr(lv), _ptr(chunks), _ptr(offs[0]), _ptr(offs[1]), _stream()))
        nv, nt = (int(x) for x in offs[:, rows].tolist())            # the one synchronisation: sizes of the outputs
        verts = torch.empty((nv, 3), dtype=torch.float32, device=dev)
        normals = torch.empty((nv, 3), dtype=torch.float32, device=dev)
        values = torch.empty(nv, dtype=torch.float32, device=dev)
        faces = torch.empty((nt, 3), dtype=torch.int32, device=dev)
        if nv or nt:
            _capi.check(L.dfb_mc_emit(_ptr(vol), rx, ry, rz, step, int(x_origin), _ptr(lv), _ptr(chunks), _ptr(offs[0]), _ptr(offs[1]),
                                      _ptr(verts), _ptr(normals), _ptr(values), _ptr(faces), _stream()))
        if keep_on_device:      # CUDA tensors: the mesh stays where update_graph / setupCorrespondences / solve consume it
            out = (verts, faces, normals, values)
        else:
            out = (verts.cpu().numpy(), faces.cpu().numpy(), normals.cpu().numpy(), values.cpu().numpy())
        if plane_offsets:
            ny = (ry - 1) // step + 1
            po = offs[:, ::ny].cpu().numpy().astype(np.int64)        # rows are (x, y) pairs: every ny-th entry starts an x-plane; [rows] = total
            out += (po[0], po[1])
        return out


# ---- SURVEY 8b item 9 / 8e: NCCL communicator and the one-launch frame step (csrc/comm.cu, csrc/step.cu) ----------------
class Comm:
    """dfb_comm: one NCCL communicator per process / GPU, created from a unique id.  `from_torch` distributes the id with
    torch.distributed (any backend) -- a host without torch hands the DFB_COMM_ID_BYTES bytes around by its own means."""

    def __init__(self, unique_id, world, rank, device=None):
        dev = _require_cuda(device)
        self.device = dev
        self.world, self.rank = int(world), int(rank)
        self._h = C.c_void_p()
        buf = (C.c_char * _capi.DFB_COMM_ID_BYTES).from_buffer_copy(bytes(unique_id))
        _capi.check(_capi.lib().dfb_comm_init(C.byref(self._h), buf, self.world, self.rank, dev.index if dev.index is not None else torch.cuda.current_device()))

    @staticmethod
    def unique_id():
        buf = (C.c_char * _capi.DFB_COMM_ID_BYTES)()
        _capi.check(_capi.lib().dfb_comm_unique_id(buf))
        return bytes(buf)

    @classmethod
    def from_torch(cls, device=None, group=None):
        import torch.distributed as dist
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        box = [cls.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        return cls(box[0], world, rank, device)

    @property
    def handle(self):
        return self._h

    def broadcast(self, t, root=0):
        assert t.is_cuda and t.is_contiguous()
        _capi.check(_capi.lib().dfb_comm_broadcast(self._h, _ptr(t), t.numel() * t.element_size(), int(root), _stream()))
        return t

    def broadcast_frame(self, depths=None, node_dq=None, lw=None, root=0):
        for t, dt in ((depths, torch.float32), (node_dq, torch.float32), (lw, torch.float64)):
            assert t is None or (t.is_cuda and t.is_contiguous() and t.dtype == dt)
        _capi.check(_capi.lib().dfb_comm_broadcast_frame(self._h, _ptr(depths), 0 if depths is None else depths.numel(), _ptr(node_dq),
                                                         0 if node_dq is None else node_dq.shape[0], _ptr(lw), int(root), _stream()))

    def allreduce_f64(self, t, op="sum"):
        assert t.is_cuda and t.is_contiguous() and t.dtype == torch.float64
        _capi.check(_capi.lib().dfb_comm_allreduce_f64(self._h, _ptr(t), t.numel(), 0 if op == "sum" else 1, _stream()))
        return t

    def sendrecv(self, send=None, send_peer=-1, recv=None, recv_peer=-1):
        _capi.check(_capi.lib().dfb_comm_sendrecv(self._h, _ptr(send), 0 if send is None else send.numel() * send.element_size(), int(send_peer),
                                                  _ptr(recv), 0 if recv is None else recv.numel() * recv.element_size(), int(recv_peer), _stream()))

    def close(self):
        if self._h:
            _capi.lib().dfb_comm_destroy(self._h)
            self._h = C.c_void_p()


class FrameStep:
    """dfb_frame_step: one frame of the a3 path (transform upload / broadcast -> node records -> warped projective update ->
    counters read-back, plus the prefetch of the next frame's sensor data as a concurrent branch) as ONE CUDA-graph launch.
    The argument structs are built once; `run` is a single C call."""

    def __init__(self, vol, wf, lw, views, tdist, wmax=100.0):
        self._h = C.c_void_p()
        _capi.check(_capi.lib().dfb_frame_step_create(C.byref(self._h)))
        self.vol, self.wf, self.views = vol, wf, views
        knn = wf.knn_table(vol.res, vol.x0, vol.x1)
        bricks = wf.brick_nodes(vol.res, vol.x0, vol.x1)
        self._keep = (knn, bricks)
        self._v = vol.struct()
        self._w = wf.struct(lw, knn, bricks=bricks)
        self._ws = vol.workspace.struct(True)
        self.tdist, self.wmax = float(tdist), float(wmax)

    def set_lw(self, lw):
        fill_lw(self._w, lw)

    def set_views(self, views):
        self.views = views

    def io(self, comm=None, comm_prefetch=None, root=0, dq_src=None, prefetch_dst=None, prefetch_src=None, counters_host=None):
        io = _capi.FrameIO()
        io.comm = comm.handle if comm is not None else None
        io.comm_prefetch = comm_prefetch.handle if comm_prefetch is not None else None
        io.root = int(root)
        io.dq_src = dq_src.data_ptr() if dq_src is not None else None
        if prefetch_dst is not None:
            io.prefetch_dst = prefetch_dst.data_ptr()
            io.prefetch_bytes = prefetch_dst.numel() * prefetch_dst.element_size()
            io.prefetch_src = prefetch_src.data_ptr() if prefetch_src is not None else None
        io.counters_host = counters_host.data_ptr() if counters_host is not None else None
        io._keep = (comm, comm_prefetch, dq_src, prefetch_dst, prefetch_src, counters_host)
        return io

    def run(self, io=None):
        _capi.check(_capi.lib().dfb_frame_step_run(self._h, C.byref(self._v), C.byref(self._w), C.byref(self.views), self.tdist, self.wmax,
                                                   C.byref(self._ws), C.byref(io) if io is not None else None, _stream()))

    def stats(self):
        out = (C.c_int64 * 5)()
        _capi.check(_capi.lib().dfb_frame_step_stats(self._h, out))
        return {"captures": out[0], "updates": out[1], "replays": out[2], "direct": out[3], "graph_nodes": out[4]}

    def __del__(self):
        try:
            if self._h:
                _capi.lib().dfb_frame_step_destroy(self._h)
        except Exception:
            pass


def slab_cost_profile(vol, unit_planes=16):
    """Estimated cost of every `unit_planes`-thick x-layer of the slab from the brick classes of the LAST projective update
    (Workspace.brick_cls: 0 = SKIP, 0xFF = MIXED, else CLAMP): cost = 0.6 per brick (classification) + 1.6 per CLAMP brick
    (streaming) + 10.7 per MIXED brick (per-voxel tier + its share of the exact pass), in ns on one B200 -- the weights are the
    measured per-brick times of the 512^3 benchmark step.  Feeds dist.balanced_slab_partition.  numpy float64 [n_units]."""
    sx, ry, rz = vol.x1 - vol.x0, vol.res[1], vol.res[2]
    nbx, nby, nbz = (sx + 3) // 4, (ry + 3) // 4, (rz + 31) // 32
    nb = nbx * nby * nbz
    cls = vol.workspace.brick_cls[:nb].view(nbx, nby * nbz)
    mixed = (cls == 0xFF).sum(1).double()
    clamp = ((cls != 0xFF) & (cls != 0)).sum(1).double()
    layer = (0.6 * nby * nbz + 1.6 * clamp + 10.7 * mixed).cpu().numpy()          # per 4-plane brick layer
    per_unit = unit_planes // 4
    n_units = (nbx + per_unit - 1) // per_unit
    pad = np.zeros(n_units * per_unit)
    pad[:nbx] = layer
    return pad.reshape(n_units, per_unit).sum(1)
