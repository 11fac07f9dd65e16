"""Drop-in classes for the reference's hot-path objects, backed by libdfb_b200.so.

The reference replaces a hot method by subclassing and overriding it (`FusionDM_GPU(FusionDM)`,
core/fusion_dm.py:563-600); a driver then only swaps the class name (test.py:158-161).  `Fusion`,
`FusionDM` and `FusionDM_GPU` below keep the reference's method names, argument meaning, attribute names
and error behaviour for the two hot paths (SURVEY 8b), with state living on the GPU:

  * `_tsdf`, `_tsdfw`  -- device-resident float32 slabs; reading the attribute materialises a numpy copy,
                          assigning a numpy array uploads it (the OpenCL path's per-call full-volume
                          upload/readback, core/fusion_dm.py:693-703, is exactly what this avoids);
  * `_nodes`           -- the reference's list of (vertex_idx, pos, dq, w) tuples (core/fusion.py:113-116)
                          on read/assign, SoA tensors + packed records on the device;
  * the per-voxel KD-tree query of `updateTSDF` (core/fusion.py:175) is replaced by an exact kNN table
                          cached per graph revision.

The callers either side of the hot paths (SURVEY 8f ranks 1-2) run on the device too: `setupCorrespondences`
(closest-point correspondences), `update_graph` / `construct_graph` (node sampling, unsupported surface points,
vertex->node tables), and so does surface extraction (8f rank 3, `marching_cubes`; `surface_extractor` swaps it out).
"""
import os

import numpy as np
import torch
from scipy.spatial import KDTree

from . import _capi, engine
from . import dist as ddist
from . import gn as _gn


def _as_np(a):
    if isinstance(a, torch.Tensor):
        return a.detach().cpu().numpy()
    return np.asarray(a)


class _FusionBase:
    """State shared by Fusion and FusionDM."""

    def _init_state(self, trunc_distance, knn, marching_cubes_step_size, verbose, write_warpfield, device):
        self._device = engine._require_cuda(device)
        _capi.lib()                                       # fail loudly now if the CUDA library is missing
        self._itercounter = 0
        self._curr_tsdf = None
        self._tdist = abs(trunc_distance)
        self._knn = knn
        self._marching_cubes_step_size = marching_cubes_step_size
        self._verbose = verbose
        self._write_warpfield = write_warpfield
        self._vol = None
        self._wf = engine.DeviceWarpField(knn, self._device)
        self._node_vertex_idx = np.zeros(0, dtype=np.int64)
        self._neighbor_look_up = []
        self._correspondences = []
        self._vertices = None
        self._normals = None
        self._faces = None
        self._radius = None
        self._sess = None
        self._mode = _capi.MODE_HYBRID
        self._last_views = None
        self._dev_cache = {}

    # ---- device copies of the host arrays the object owns ------------------------------------------
    def _dev(self, arr, dtype=torch.float32):
        """Device copy of a host array held in a reference attribute (`_vertices`, `_normals`, `_neighbor_look_up`), cached by the
        array's identity.  The device surface extractor leaves its output on the GPU and the numpy attribute is its one download, so
        the callers either side of the hot paths (update_graph, setupCorrespondences, solve) never upload the mesh again.  The
        attributes are replaced, never edited in place, by this class (as by the reference); a caller that edits one in place
        must re-assign it."""
        if isinstance(arr, torch.Tensor):
            return arr.to(device=self._device, dtype=dtype)
        key = (id(arr), dtype)
        hit = self._dev_cache.get(key)
        if hit is not None and hit[0] is arr:
            return hit[1]
        t = engine._to_dev(arr, dtype, self._device)
        self._remember(arr, t, dtype)
        return t

    def _remember(self, arr, t, dtype=torch.float32):
        if len(self._dev_cache) >= 12:
            self._dev_cache.pop(next(iter(self._dev_cache)))
        self._dev_cache[(id(arr), dtype)] = (arr, t)       # keeps `arr` alive, so its id cannot be re-used

    # ---- device-resident volume exposed under the reference's attribute names -------------------
    @property
    def _tsdf(self):
        return None if self._vol is None else self._vol.tsdf.cpu().numpy()

    @_tsdf.setter
    def _tsdf(self, value):
        self._set_volume(value, None)

    @property
    def _tsdfw(self):
        return None if self._vol is None else self._vol.weight.cpu().numpy()

    @_tsdfw.setter
    def _tsdfw(self, value):
        self._set_volume(None, value)

    def _set_volume(self, tsdf, weight, shape=None, slab=None):
        if tsdf is not None:
            if not isinstance(tsdf, (np.ndarray, torch.Tensor)) or tsdf.ndim != 3:
                raise ValueError('Only 3D numpy array is accepted as tsdf')
        if self._vol is None or (tsdf is not None and tuple(tsdf.shape) != tuple(self._vol.tsdf.shape)):
            if tsdf is None and weight is None:
                full = tuple(shape)
            else:
                ref = tsdf if tsdf is not None else weight
                full = tuple(shape) if shape is not None else tuple(ref.shape)
            x0, x1 = slab if slab is not None else (0, full[0])
            self._vol = engine.DeviceVolume(full, x0, x1, self._device, tsdf=tsdf, weight=weight, fill=self._tdist)
            return
        if tsdf is not None:
            self._vol.tsdf.copy_(engine._to_dev(tsdf, torch.float32, self._device).reshape(self._vol.tsdf.shape))
        if weight is not None:
            self._vol.weight.copy_(engine._to_dev(weight, torch.float32, self._device).reshape(self._vol.weight.shape))

    # ---- deformation graph under the reference's `_nodes` layout --------------------------------
    @property
    def _nodes(self):
        if self._wf.n_nodes == 0:
            return []
        pos = self._wf.node_pos.cpu().numpy()
        dq = self._wf.node_dq.cpu().numpy()
        w = self._wf.node_w.cpu().numpy()
        return [(int(self._node_vertex_idx[i]), pos[i], dq[i], float(w[i])) for i in range(len(pos))]

    @_nodes.setter
    def _nodes(self, nodes):
        nodes = list(nodes)
        if not nodes:
            self._wf = engine.DeviceWarpField(self._knn, self._device)
            self._node_vertex_idx = np.zeros(0, dtype=np.int64)
            return
        self._node_vertex_idx = np.array([n[0] for n in nodes], dtype=np.int64)
        pos = np.array([n[1] for n in nodes], dtype=np.float32)
        dq = np.array([n[2] for n in nodes], dtype=np.float32)
        w = np.array([n[3] for n in nodes], dtype=np.float32)
        same_pos = (self._wf.n_nodes == len(nodes) and np.array_equal(self._wf.node_pos.cpu().numpy(), pos)
                    and np.array_equal(self._wf.node_w.cpu().numpy(), w))
        if same_pos:
            self._wf.set_dq(dq)                            # transforms only: the cached kNN tables stay valid
        else:
            self._wf.k = self._knn
            self._wf.set_nodes(pos, dq, w)

    def set_node_dqs(self, dq):
        """Fast path for per-frame transform updates: (N,8) float32, host or device."""
        self._wf.set_dq(dq)

    @property
    def _kdtree(self):
        """Host KD-tree over the node positions (what the reference stores, core/fusion.py:119)."""
        return KDTree(self._wf.node_pos.cpu().numpy()) if self._wf.n_nodes else None

    def build_knn(self):
        """Build (or fetch) the cached voxel->k-nearest-node table of this slab.  Called implicitly by the
        update methods; exposed so that a driver can pay for it outside a timed region."""
        t = self._wf.knn_table(self._vol.res, self._vol.x0, self._vol.x1)
        self._wf.brick_nodes(self._vol.res, self._vol.x0, self._vol.x1)
        return t

    def knn_indices(self):
        """(n_voxels, k) int64 node ids == KDTree.query(pos, k+1)[1][:-1] per voxel (core/fusion.py:175-176)."""
        return self.build_knn().cpu().numpy().view(np.uint16).astype(np.int64)

    def frame_stats(self):
        """Counters of the last update call (a 32-byte device->host read)."""
        s = self._vol.workspace.stats()
        return s

    def frame_stats_async(self):
        """Same counters without stalling the stream: returns a handle, .result() waits for the copy."""
        return self._vol.workspace.stats_async()

    # ---- warp helpers (core/fusion.py:502-551), evaluated on the device -------------------------
    def _lookup(self, pos, k):
        return self._wf.knn_points(np.asarray(pos, dtype=np.float32).reshape(-1, 3), k).cpu().numpy()

    def _set_lookup(self, nlu_dev):
        """`_neighbor_look_up` (vertex -> k nearest nodes) from a device int32 table: one download, the device copy is kept."""
        h = nlu_dev.cpu().numpy().astype(np.int64)
        self._remember(h, nlu_dev, torch.int32)
        self._neighbor_look_up = h

    def warp(self, pos, dqs=None, locations=None, normal=None, dmax=None, m_lw=None):
        """Fusion.warp (core/fusion.py:502-520) for one point or an (M,3) batch.  `dqs` given explicitly
        must be the current node transforms of `locations` (the reference always passes those)."""
        p = np.asarray(pos, dtype=np.float32)
        single = p.ndim == 1
        p2 = p.reshape(-1, 3)
        if locations is None:
            # query(k+1)[:-1] (core/fusion.py:504-505) == the k nearest
            loc = self._lookup(p2, self._knn)
        else:
            loc = np.asarray(locations, dtype=np.int32).reshape(len(p2), -1)
        wf = self._wf
        if dqs is not None:
            wf = self._wf_with_dqs(loc, np.asarray(dqs, dtype=np.float32).reshape(len(p2), -1, 8), dmax)
            loc = np.arange(loc.size, dtype=np.int32).reshape(loc.shape)
        elif dmax is not None:
            wf = self._wf_with_dmax(dmax)
        n2 = None if normal is None else np.asarray(normal, dtype=np.float32).reshape(-1, 3)
        out = engine.warp_points(wf, m_lw, p2, n2, idx=loc, k=loc.shape[1])
        if normal is None:
            r = out.cpu().numpy()
            return r[0] if single else r
        r, rn = out[0].cpu().numpy(), out[1].cpu().numpy()
        return (r[0], rn[0]) if single else (r, rn)

    @staticmethod
    def _dmax_w(dmax, n):
        """`exp(-(|pos - dg_v| / dmax)^2)` (core/fusion.py:539-541) is the default weight `exp(-(|pos - dg_v| / (2 dg_w))^2)` with
        2 dg_w replaced by dmax: in the reference both divisors are python floats, i.e. weak operands rounded to float32, and
        halving / doubling a float32 is exact -- so node weights of float32(dmax) / 2 reproduce the dmax variant bit for bit."""
        return np.full(n, np.float32(dmax) / np.float32(2.0), dtype=np.float32)

    def _wf_with_dqs(self, loc, dqs, dmax=None):
        """Temporary warp field whose node j is (pos/w of node loc.flat[j], dq = dqs.flat[j]) -- lets
        `warp`/`dq_blend` honour explicitly passed transforms like the reference does."""
        pos = self._wf.node_pos.cpu().numpy()[loc.reshape(-1)]
        w = self._wf.node_w.cpu().numpy()[loc.reshape(-1)] if dmax is None else self._dmax_w(dmax, loc.size)
        wf = engine.DeviceWarpField(loc.shape[1], self._device)
        wf.set_nodes(pos, dqs.reshape(-1, 8), w)
        return wf

    def _wf_with_dmax(self, dmax):
        """The current graph with every node weight replaced by dmax / 2 (see _dmax_w)."""
        wf = engine.DeviceWarpField(self._wf.k, self._device)
        wf.set_nodes(self._wf.node_pos, self._wf.node_dq, self._dmax_w(dmax, self._wf.n_nodes))
        return wf

    def dq_blend(self, pos, dqs=None, locations=None, dmax=None):
        """Fusion.dq_blend (core/fusion.py:527-551): blended, 8-norm-normalised dual quaternion (Q2)."""
        p = np.asarray(pos, dtype=np.float32).reshape(1, 3)
        loc = self._lookup(p, self._knn) if locations is None else np.asarray(locations, dtype=np.int32).reshape(1, -1)
        wf = self._wf
        if dqs is not None:
            wf = self._wf_with_dqs(loc, np.asarray(dqs, dtype=np.float32).reshape(1, -1, 8), dmax)
            loc = np.arange(loc.size, dtype=np.int32).reshape(loc.shape)
        elif dmax is not None:
            wf = self._wf_with_dmax(dmax)
        return _gn.dq_blend_points(wf, p, loc)[0]

    def write_warp_field(self, path, filename):
        """core/fusion.py:571-573."""
        from . import io
        io.write_warp_field(self._nodes, path, filename, self._itercounter)

    # ---- surface extraction (SURVEY 8f rank 3) ------------------------------------------------------
    surface_extractor = "device"
    """"device" (default): the library's own extractor (`engine.marching_cubes`, include/dfb.h `dfb_mc_*`) on the
    device-resident volume.  A callable(tsdf, step_size) -> (verts, faces, normals, values) -- the contract of
    skimage.measure.marching_cubes_lewiner(tsdf, step_size=..., allow_degenerate=False) that the reference calls
    (core/fusion.py:554-564) -- replaces it (e.g. skimage itself where it is installed).  None: no extraction; the
    methods that need a surface raise NotImplementedError unless the vertices are handed to them."""

    def marching_cubes(self, tsdf=None, step_size=0):
        """core/fusion.py:553-568.  Vertices are in voxel coordinates of the whole grid (a slab's x offset is added)."""
        ext = self.surface_extractor
        if ext is None:
            raise NotImplementedError("no surface extractor configured: set `surface_extractor` (\"device\" or a callable), "
                                      "or pass live_vertices= / vertices= to the caller")
        if step_size < 1:
            step_size = self._marching_cubes_step_size
        step_size = max(1, int(step_size))                            # the reference's test.py:74 passes 0.5; skimage needs an int >= 1
        if tsdf is not None:
            return engine.marching_cubes(tsdf, step_size) if ext == "device" else ext(_as_np(tsdf), step_size)
        if ext == "device":
            v, f, n, _ = self._device_surface(step_size, keep_on_device=True)
        else:
            v, f, n, _ = ext(_as_np(self._tsdf), step_size)
        if isinstance(v, torch.Tensor):                               # the mesh stays on the device; the attributes are its download
            vh, nh = v.cpu().numpy(), n.cpu().numpy()
            self._remember(vh, v)
            self._remember(nh, n)
            v, n, f = vh, nh, f.cpu().numpy()
        self._vertices, self._faces, self._normals = np.asarray(v, dtype=np.float32), f, np.asarray(n, dtype=np.float32)
        if self._verbose:
            print("Marching Cubes result: number of extracted vertices is %d" % (len(self._vertices)))

    def _device_surface(self, step_size, level=None, keep_on_device=False):
        """Surface of the resident canonical volume (level None = 0.5 * (min + max) like skimage's default).  A rank that holds an x-slab of a volume sharded over the process group
        (SURVEY 8e) extracts its share with three halo planes per boundary and every rank receives the whole mesh, identical to the
        single-GPU one (dist.extract_surface_slab); a lone slab is extracted as is, in whole-grid coordinates."""
        vol = self._vol
        rx = int(vol.res[0])
        if ddist.is_dist() and (vol.x0 > 0 or vol.x1 < rx):
            return ddist.allgather_mesh(ddist.extract_surface_slab(vol.tsdf, vol.x0, vol.x1, rx, step_size, level=level))
        if vol.x0 % step_size == 0:
            return engine.marching_cubes(vol.tsdf, step_size, level, x_origin=vol.x0 // step_size, keep_on_device=keep_on_device)
        v, f, n, val = engine.marching_cubes(vol.tsdf, step_size, level)
        v[:, 0] += np.float32(vol.x0)
        return v, f, n, val

    def write_live_frame_mesh(self, path, filename, warpfield_path):
        """core/fusion_dm.py:357-358: an empty method in the reference."""
        pass

    def average_edge_dist_in_face(self, f):
        """core/fusion.py:592-596."""
        v1, v2, v3 = self._vertices[f[0]], self._vertices[f[1]], self._vertices[f[2]]
        return (np.linalg.norm(v1 - v2) + np.linalg.norm(v1 - v3) + np.linalg.norm(v2 - v3)) / 3

    def write_canonical_mesh(self, path, filename):
        """core/fusion.py:577-586 / core/fusion_dm.py:339-354: extract the canonical surface (step size 1) and write it as OBJ; FusionDM maps vertices and normals to world coordinates with `_IND` first."""
        from . import io
        ind = getattr(self, "_IND", None)
        # FusionDM extracts the ZERO level set (`level=0`, core/fusion_dm.py:341-342); Fusion passes no level (core/fusion.py:579),
        # i.e. skimage's default 0.5 * (min + max)
        level = 0.0 if ind is not None else None
        if self.surface_extractor == "device":
            verts, faces, normals, _ = self._device_surface(1, level)
        else:
            ext = self.surface_extractor
            try:
                verts, faces, normals, _ = ext(_as_np(self._tsdf), 1, level) if level is not None else ext(_as_np(self._tsdf), 1)
            except TypeError:
                verts, faces, normals, _ = ext(_as_np(self._tsdf), 1)
            if self._vol.x0:
                verts = np.array(verts); verts[:, 0] += self._vol.x0
        if ind is not None:
            rot, trans = ind[:3, :3], ind[:3, 3]
            verts = np.asarray(verts, dtype=np.float64) @ rot.T + trans
            normals = np.asarray(normals, dtype=np.float64) @ rot.T
        io.write_obj(os.path.join(path, filename), verts, normals, faces, face_normals=ind is not None)

    # ---- SURVEY 8f rank 1: closest-point correspondences ---------------------------------------------
    def _live_vertices(self, curr_tsdf, live_vertices):
        if live_vertices is None:
            live_vertices = self.marching_cubes(curr_tsdf, step_size=1)[0]
        lv = engine._to_dev(live_vertices, torch.float32, self._device).reshape(-1, 3)
        if lv.shape[0] < self._knn:
            raise ValueError('the live surface has fewer vertices than knn')
        return lv

    def _closest_points(self, lv, wv, wn):
        """core/fusion.py:264-274: k nearest live vertices of every warped canonical vertex, best point-to-plane cost."""
        nn = engine.PointGrid(lv, device=self._device).knn(wv, self._knn)
        return engine.corr_select(wv, wn, lv, nn)

    def _relink_nodes(self):
        """node -> index of its nearest canonical vertex (core/fusion.py:204-209,308-313)."""
        if self._wf.n_nodes and self._vertices is not None and len(self._vertices):
            grid = engine.PointGrid(self._dev(self._vertices), device=self._device)
            self._node_vertex_idx = grid.knn(self._wf.node_pos.double(), 1).reshape(-1).cpu().numpy().astype(np.int64)


class Fusion(_FusionBase):
    """Non-rigid fusion object (core/fusion.py:49).  Constructor arguments as in the reference; `device`
    selects the GPU.  `use_cnn` is accepted for signature compatibility (the CNN path is out of scope)."""

    def __init__(self, trunc_distance, subsample_rate=5.0, knn=4, marching_cubes_step_size=3, verbose=False,
                 use_cnn=True, write_warpfield=True, device=None):
        self._init_state(trunc_distance, knn, marching_cubes_step_size, verbose, write_warpfield, device)
        self._lw = np.array([1, 0, 0, 0, 0, 0.1, 0, 0], dtype=np.float32)   # core/fusion.py:57
        self._subsample_rate = subsample_rate
        self._K = None
        self._Kinv = None
        self._curr_depths = None        # depth frame of the last projective association (re-associated by solve)
        self._corridx = None            # vertices the data term covers (None = all of them)

    def InitializeCanonicalSpace(self, tsdf=None, depths=None, lws=None, K=None, tsdf_size=256, *, tsdf_shape=None,
                                 slab=None, vertices=None, normals=None, faces=None, nodes=None, radius=None):
        """core/fusion.py:73-96.  The reference extracts the canonical surface with marching cubes and samples
        the nodes from it; so does this (device extractor, `marching_cubes`) unless the canonical `vertices`/`normals`
        (and optionally ready-made `nodes`) are passed in.  `slab=(x0,x1)` keeps only that x-range of the
        volume on this GPU (multi-GPU sharding); `tsdf_shape` creates the fresh volume (tsdf=+tdist, w=0)."""
        if K is not None:
            self._K = np.asarray(K, dtype=np.float64)
            self._Kinv = np.linalg.inv(self._K)
        if tsdf is not None:
            self._set_volume(tsdf, None, shape=tsdf_shape, slab=slab)
            self._vol.weight.zero_()
        else:
            shape = tuple(tsdf_shape) if tsdf_shape is not None else (tsdf_size,) * 3
            self._vol = None
            self._set_volume(None, None, shape=shape, slab=slab)
            if depths is not None and lws is not None and self._K is not None:
                for dm, lw in zip(depths, lws):
                    d = engine._to_dev(dm, torch.float32, self._device)
                    engine.fuse_depth_rigid(self._vol, shape[0], d, lw, self._K, self._Kinv, 1.0, None, self._tdist, 100.0)
        if vertices is not None:
            self._vertices = np.asarray(vertices, dtype=np.float32)
            self._normals = None if normals is None else np.asarray(normals, dtype=np.float32)
            self._faces = faces
        elif self.surface_extractor is not None and nodes is None and min(self._vol.tsdf.shape) >= 2:
            self.marching_cubes()                                     # core/fusion.py:88 (initial marching cubes)
            faces = self._faces
            if not len(self._vertices):                               # empty volume: nothing to sample a graph from yet
                self._vertices = self._faces = self._normals = faces = None
        if radius is not None:
            self._radius = float(radius)
        elif self._vertices is not None and faces is not None and len(faces):
            f = np.asarray(faces)
            v = self._vertices.astype(np.float64)
            e = (np.linalg.norm(v[f[:, 0]] - v[f[:, 1]], axis=1) + np.linalg.norm(v[f[:, 0]] - v[f[:, 2]], axis=1)
                 + np.linalg.norm(v[f[:, 1]] - v[f[:, 2]], axis=1)) / 3
            self._radius = self._subsample_rate * float(e.mean())     # core/fusion.py:89-92
        if nodes is not None:
            self._nodes = nodes
            if self._vertices is not None:
                self._neighbor_look_up = self._lookup(self._vertices, self._knn).astype(np.int64)
        elif self._vertices is not None and self._radius is not None:
            self.construct_graph()

    def construct_graph(self):
        """core/fusion.py:101-123: radius-based node sampling from the canonical vertices, initial node dq
        [1,0,0,0,0,.01,.01,0] (Q5), w = 2*radius, vertex->node kNN table."""
        nodes_v, nodes_idx = engine.uniform_sample(self._vertices, self._radius, device=self._device)
        dq0 = np.array([1, 0.00, 0.00, 0.00, 0.00, 0.01, 0.01, 0.00], dtype=np.float32)
        self._nodes = [(int(nodes_idx[i]), nodes_v[i], dq0, 2 * self._radius) for i in range(len(nodes_v))]
        self._neighbor_look_up = self._lookup(self._vertices, self._knn).astype(np.int64)

    def update_graph(self, *, vertices=None, normals=None, faces=None):
        """core/fusion.py:201-239.  The reference re-extracts the canonical surface first (`marching_cubes()`); pass
        `vertices` (+ `normals`) to supply it instead.  Then, all on the device: nodes re-linked to their nearest vertex,
        surface points no node supports (min |node - v| / dg_w >= 1 over the k nearest) found, new nodes sampled from
        them with `uniform_sample` and initialised by `dq_blend` over the OLD graph, vertex->node table rebuilt.  As in
        the reference the vertex index stored with a NEW node counts within the unsupported subset (core/fusion.py:217-219)."""
        if vertices is not None:
            self._vertices = np.asarray(vertices, dtype=np.float32)
            self._normals = None if normals is None else np.asarray(normals, dtype=np.float32)
            self._faces = faces
        else:
            self.marching_cubes()
        self._relink_nodes()
        vd = self._dev(self._vertices)
        vknn = self._wf.knn_points(vd, self._knn)
        uns = engine.graph_unsupported(self._wf, vd, vknn)
        new_v, new_idx = engine.uniform_sample(vd[uns], self._radius, device=self._device)
        if len(new_v):
            new_dq = _gn.dq_blend_points(self._wf, new_v, self._wf.knn_points(new_v, self._knn))
            self._node_vertex_idx = np.concatenate([self._node_vertex_idx, new_idx])
            # new graph revision: nodes are only appended, so the cached voxel kNN table / brick / region sets are updated
            # incrementally (the reference rebuilds its KD-tree here, core/fusion.py:229)
            self._wf.append_nodes(new_v, new_dq.astype(np.float32), np.full(len(new_v), 2 * self._radius, dtype=np.float32))
        if self._verbose:
            print("Inserted %d new deformation nodes. Current number of deformation nodes: %d" % (len(new_v), self._wf.n_nodes))
        self._set_lookup(self._wf.knn_points(vd, self._knn) if len(new_v) else vknn)
        self._curr_tsdf = None
        self._curr_depths = None
        self._corridx = None
        self._correspondences = []
        if self._write_warpfield:
            self.write_warp_field(os.environ.get("DFB_DATA_PATH", "."), 'test')

    def setupCorrespondences(self, curr_tsdf, method='cnn', prune_result=True, tolerance=0.2, *, live_vertices=None, depths=None,
                             extrinsics=None, max_distance=None, min_normal_dot=0.5):
        """method='projective': projective data association against depth frames, DynamicFusion's own correspondence step,
        on the device (include/dfb.h dfb_corr_projective).  Every canonical vertex is warped to the live frame (`_lw` included,
        with its `_neighbor_look_up` nodes), projected into the views of `depths` ((rows,cols) or (V,rows,cols), host or CUDA,
        negative depth, 0 = no data, `extrinsics` and the object's K as in `fuseFrame`) and paired with the back-projected pixel
        it lands on, when that pixel and its four neighbours hold depths within `max_distance` of each other, the pair is closer
        than `max_distance` and the normals agree (cos >= `min_normal_dot`); the view with the smallest point-to-plane cost wins.
        `max_distance=None` is the truncation distance, the band in which fuseFrame trusts a measurement.  The canonical normals
        must point out of the surface, as marching cubes of the TSDF gives them: a vertex counts as visible when its warped
        normal faces the camera.  `curr_tsdf` and `tolerance` (the closest-point branch's cost bound) are not used.  Vertices
        without a correspondence are removed with `prune_result=True` (nodes re-linked, as below); with `prune_result=False`
        every vertex is kept, `_corridx` lists the associated ones and `_correspondences` holds their live points, and the data
        term of `solve` / `computef` covers those vertices only.  The frame is kept until `update_graph`, so that
        `solve(method='projective')` can re-associate.

        Any other method: core/fusion.py:243-313, closest-points branch (the CNN branch is out of scope, so `method` only keeps the
        signature; the reference itself takes this branch whenever no TF session exists, :252).  Every canonical vertex
        is warped to the live frame, its k nearest live vertices are searched, and the one with the smallest
        point-to-plane cost |n'.(v' - p)| (< 1, else the nearest) becomes its correspondence.  `live_vertices`
        replaces `marching_cubes(curr_tsdf, step_size=1)`.
        Pruning: vertices whose best cost exceeds `tolerance` are removed from `_vertices/_normals/_correspondences/
        _neighbor_look_up` and the nodes re-linked (:294-313).  The reference's clpts loop records the wrong index here
        (its inner `for idx in iidx` shadows the vertex index, :269-276, so it deletes the vertex whose number is the
        k-th nearest LIVE vertex's); the intended vertex is pruned instead (stated deviation, like SURVEY Q7)."""
        if method == 'projective' or depths is not None:
            if method != 'projective':
                raise ValueError("depths= is the input of method='projective'")
            if depths is None:
                raise ValueError("method='projective' needs depths=")
            return self._associate_projective(depths, extrinsics, max_distance, min_normal_dot, prune_result)
        self._corridx = None
        self._curr_tsdf = curr_tsdf
        if self._vertices is None or self._normals is None:
            raise ValueError('canonical vertices/normals have not been set')
        lv = self._live_vertices(curr_tsdf, live_vertices)
        loc = self._dev(self._neighbor_look_up, torch.int32).reshape(len(self._vertices), -1)
        wv, wn = engine.warp_points(self._wf, self._lw, self._dev(self._vertices), self._dev(self._normals), idx=loc, k=loc.shape[1])
        best, cost = self._closest_points(lv, wv, wn)
        self._correspondences = lv[best.long()].cpu().numpy()
        self._corr_cost = cost.cpu().numpy()
        if prune_result:
            pruned = np.nonzero(self._corr_cost > tolerance)[0]
            if self._verbose:
                print('ratio of correspondence outlier rejection', float(len(pruned)) / float(len(self._vertices)))
            self._vertices = np.delete(self._vertices, pruned, axis=0)
            self._correspondences = np.delete(self._correspondences, pruned, axis=0)
            self._neighbor_look_up = np.delete(np.asarray(self._neighbor_look_up), pruned, axis=0)
            self._normals = np.delete(self._normals, pruned, axis=0)
            self._faces = None
            self._relink_nodes()

    def _associate_projective(self, depths, extrinsics, max_distance, min_normal_dot, prune_result):
        if self._vertices is None or self._normals is None:
            raise ValueError('canonical vertices/normals have not been set')
        if self._K is None:
            raise ValueError('camera intrinsics K have not been set')
        d = engine._to_dev(depths, torch.float32, self._device)
        if d.dim() == 2:
            d = d[None]
        if d.dim() != 3:
            raise ValueError('depth maps must be (rows, cols) or (views, rows, cols)')
        if extrinsics is not None and len(extrinsics) != d.shape[0]:
            raise ValueError('length of camera matrix array must equal that of depth maps')
        md = self._tdist if max_distance is None else float(max_distance)
        views = engine.make_views(d, self._K, self._Kinv, extrinsics)
        loc = self._dev(self._neighbor_look_up, torch.int32).reshape(len(self._vertices), -1)
        wv, wn = engine.warp_points(self._wf, self._lw, self._dev(self._vertices), self._dev(self._normals), idx=loc, k=loc.shape[1])
        view, cost, corr = engine.corr_projective(wv, wn, views, md, min_normal_dot)
        hit = (view >= 0).cpu().numpy()
        if not hit.any():
            raise ValueError('no canonical vertex is associated with the depth frame')
        self._curr_depths, self._curr_extrinsics = d, extrinsics
        self._assoc_args = dict(max_distance=md, min_normal_dot=min_normal_dot, prune_result=prune_result)
        self._corr_view = view.cpu().numpy()
        self._corr_cost = cost.cpu().numpy()
        self._correspondences = corr[torch.from_numpy(hit).to(self._device)].cpu().numpy()
        if not prune_result:
            self._corridx = np.nonzero(hit)[0]
            return
        self._corridx = None
        pruned = np.nonzero(~hit)[0]
        if self._verbose:
            print('ratio of vertices without a projective correspondence', float(len(pruned)) / float(len(self._vertices)))
        if len(pruned):
            self._vertices = np.delete(self._vertices, pruned, axis=0)
            self._neighbor_look_up = np.delete(np.asarray(self._neighbor_look_up), pruned, axis=0)
            self._normals = np.delete(self._normals, pruned, axis=0)
            self._faces = None
            self._relink_nodes()

    def _reassociate(self):
        """setupCorrespondences(method='projective') again, against the frame and gates of the last call."""
        if self._curr_depths is None:
            raise ValueError("no depth frame on record: call setupCorrespondences(method='projective', depths=...) first")
        self.setupCorrespondences(None, method='projective', depths=self._curr_depths, extrinsics=self._curr_extrinsics, **self._assoc_args)

    # ---- a1 ---------------------------------------------------------------------------------------
    def updateTSDF(self, curr_tsdf=None, wmax=100.0):
        """core/fusion.py:153-198 (volume-sampling warped update; Q1 trilinear, Q4 weights)."""
        if curr_tsdf is not None:
            self._curr_tsdf = curr_tsdf
        if self._curr_tsdf is None:
            raise ValueError('tsdf of live frame has not been loaded')
        if not isinstance(self._curr_tsdf, (np.ndarray, torch.Tensor)):
            raise ValueError('Only accept 3D np array as tsdf')
        elif self._curr_tsdf.ndim != 3:
            raise ValueError('Only accept 3D np array as tsdf')
        curr = engine._to_dev(self._curr_tsdf, torch.float32, self._device)
        engine.update_volume(self._vol, self._wf, self._lw, curr, self._tdist, wmax, mode=self._mode)

    # ---- a3 ---------------------------------------------------------------------------------------
    def fuseFrame(self, depths, K=None, extrinsics=None, wmax=100.0, mode=None, want_masks=False):
        """The north-star path (README.md:9-14 TODO of the reference): warp every voxel centre canonical->live
        (`warp`, m_lw=self._lw), project through K, fold the depth measurement(s) into (v,w) with the rule of
        FusionDM.fuseDepths.  depths: (rows,cols) or (V,rows,cols), host numpy or CUDA tensor, negative depth."""
        if K is not None:
            self._K = np.asarray(K, dtype=np.float64)
            self._Kinv = np.linalg.inv(self._K)
        if self._K is None:
            raise ValueError('camera intrinsics K have not been set')
        d = engine._to_dev(depths, torch.float32, self._device)
        if d.dim() == 2:
            d = d[None]
        if d.dim() != 3:
            raise ValueError('depth maps must be (rows, cols) or (views, rows, cols)')
        if extrinsics is not None and len(extrinsics) != d.shape[0]:
            raise ValueError('length of camera matrix array must equal that of depth maps')
        return engine.update_projective(self._vol, self._wf, self._lw, d, self._K, self._Kinv, extrinsics, self._tdist, wmax,
                                        mode=self._mode if mode is None else mode, want_masks=want_masks)

    # ---- solve (core/fusion.py:327-491) -------------------------------------------------------------
    def _problem(self):
        if self._vertices is None or self._normals is None:
            raise ValueError('canonical vertices/normals have not been set')
        corr = np.asarray(self._correspondences, dtype=np.float64)
        if self._corridx is not None:
            # data term over the associated vertices only; the regularisation term keeps its neighbours from the full table
            if len(corr) != len(self._corridx):
                raise ValueError("Please first call setupCorrespondences to compute point to point correspondences between canonical and live frame vertices!")
            nlu = self._dev(np.asarray(self._neighbor_look_up), torch.int32).reshape(len(self._vertices), -1)
            sub = torch.from_numpy(np.asarray(self._corridx, dtype=np.int64)).to(self._device)
            nvi = torch.from_numpy(np.asarray(self._node_vertex_idx, dtype=np.int64)).to(self._device)
            return _gn.Problem(self._wf, self._dev(self._vertices)[sub], self._dev(self._normals)[sub], corr, nlu[sub].contiguous(),
                               self._node_vertex_idx, node_nbr=nlu[nvi].contiguous())
        if len(corr) != len(self._vertices):
            raise ValueError("Please first call setupCorrespondences to compute point to point correspondences between canonical and live frame vertices!")
        nlu = self._neighbor_look_up
        nlu = self._dev(nlu, torch.int32) if isinstance(nlu, np.ndarray) else np.asarray(nlu)
        return _gn.Problem(self._wf, self._dev(self._vertices), self._dev(self._normals), corr, nlu, self._node_vertex_idx)

    def computef(self, x, tdw, trw, rw):
        """core/fusion.py:459-491: residual vector (V + 3*k*N,), float64."""
        return self._problem().residuals(np.asarray(x, dtype=np.float64), self._lw, rw).cpu().numpy()

    def computef_lw(self, x, tdw, trw):
        """core/fusion.py:444-456: data term as a function of the global rigid dq."""
        return self._problem().residuals_lw(np.asarray(x, dtype=np.float64)).cpu().numpy()

    def computeSparsity(self, n, m):
        """Jacobian sparsity.  NOT the reference's pattern (core/fusion.py:416-442 declares only 3N of the 3kN
        regularisation rows, SURVEY Q7): this is the correct one -- data row i -> the 8 columns of each of its k
        nodes; reg row (i,j,c) -> the 16 columns of nodes i and j."""
        return _gn.sparsity(np.asarray(self._neighbor_look_up), self._node_vertex_idx, len(self._vertices), self._wf.n_nodes, n, m)

    def solve(self, correspondences=None, method='cnn', precompute_lw=True, tukey_data_weight=0.2,
              huber_regularization_weight=0.001, regularization_weight=1, *, gn_iterations=15, gn_options=None):
        """core/fusion.py:327-412.  Same call surface and outer schedule (rigid lw fit, then up to 3 warp-field
        rounds with the rw /= 8 relaxation); the inner optimiser is a damped Gauss-Newton on the explicitly
        assembled normal equations instead of scipy's finite-difference TRF/LSMR (SURVEY 8a row a12)."""
        if correspondences is not None:
            self._correspondences = correspondences
            self._corridx = None
            if len(self._correspondences) != len(self._vertices):
                raise ValueError("Please first call setupCorrespondences to compute point to point correspondences between canonical and live frame vertices!")
        iteration = 3 if method in ('clpts', 'projective') else 1
        self._itercounter += 1
        opts = dict(gn_options or {})
        prob = self._problem()
        if precompute_lw:
            self._lw = prob.solve_lw(np.asarray(self._lw, dtype=np.float64), max_iter=opts.get("lw_iterations", 20), verbose=self._verbose)
            # core/fusion.py:363-364 re-runs setupCorrespondences after the rigid fit whenever method == 'clpts' -- even over
            # correspondences the caller passed in.  Same here whenever a live TSDF is on record; with explicit correspondences
            # and no live TSDF (where the reference would fail inside marching cubes) the passed ones are kept.
            if method == 'clpts' and (correspondences is None or self._curr_tsdf is not None):
                self.setupCorrespondences(self._curr_tsdf, method='clpts')
                prob = self._problem()
            elif method == 'projective' and (correspondences is None or self._curr_depths is not None):
                self._reassociate()                                       # same rule against the depth frame on record
                prob = self._problem()
        rw = regularization_weight
        for it in range(iteration):
            if it > 0 and correspondences is None:
                if method == 'projective':
                    self._reassociate()
                else:
                    self.setupCorrespondences(self._curr_tsdf, method='clpts')
                prob = self._problem()
            x0 = self._wf.node_dq.double().reshape(-1)
            res = prob.gauss_newton(x0, self._lw, rw, max_iter=gn_iterations, huber=opts.get("huber", True),
                                    f_scale=opts.get("f_scale", 1.0), verbose=self._verbose, **opts.get("gn", {}))
            # written back un-normalised (core/fusion.py:400-403); the device node table is float32 (the reference keeps the
            # float64 `opt_result.x`, which also switches its dtype flow from then on -- stated deviation, DESIGN section 7)
            self._wf.set_dq(res.x.reshape(-1, 8).float())
            self.last_solve = res
            # core/fusion.py:376,405: plain 0.5 |f|^2 before, the optimiser's robust cost after
            reduct_rate = (res.cost0_l2 - res.cost) / res.cost0_l2 if res.cost0_l2 > 0 else 0.0
            if 0.05 < reduct_rate < 0.9:
                rw /= 8
            else:
                break


class FusionDM(_FusionBase):
    """Multi-view rigid depth-map fusion (core/fusion_dm.py:53)."""

    def __init__(self, trunc_distance, K, tsdf_res=256, subsample_rate=5.0, knn=4, marching_cubes_step_size=3,
                 verbose=False, write_warpfield=True, device=None):
        self._init_state(trunc_distance, knn, marching_cubes_step_size, verbose, write_warpfield, device)
        self._tsdf_res = tsdf_res
        self._set_volume(None, None, shape=(tsdf_res,) * 3)           # tsdf = +tdist, w = 0 (core/fusion_dm.py:61-62)
        self._lw = np.array([1, 0, 0, 0, 0, 0, 0, 0], dtype=np.float32)
        self._K = np.asarray(K, dtype=np.float64)
        self._Kinv = np.linalg.inv(self._K)
        self._IND = np.eye(4)
        self._INDinv = np.linalg.inv(self._IND)
        self._subsample_rate = subsample_rate

    def fuseDepths(self, dm, lw, tsdf, tsdf_w, scale=1.0, center=np.zeros(3), wmax=100.0):
        """core/fusion_dm.py:180-217.  numpy in -> numpy out exactly like the reference (one upload + one
        read-back); CUDA tensors in -> updated in place on the device and returned, no host traffic."""
        on_device = isinstance(tsdf, torch.Tensor) and tsdf.is_cuda
        if tsdf.ndim != 3:
            raise ValueError('Only 3D numpy array is accepted as tsdf')
        if on_device:
            if tsdf.dtype != torch.float32 or tsdf_w.dtype != torch.float32:
                raise ValueError('device volumes must be float32')
            vol = engine.DeviceVolume(tuple(tsdf.shape), device=tsdf.device, tsdf=tsdf, weight=tsdf_w)
            vol.tsdf, vol.weight = tsdf, tsdf_w
        else:
            vol = engine.DeviceVolume(tuple(tsdf.shape), device=self._device, tsdf=tsdf, weight=tsdf_w)
        d = engine._to_dev(dm, torch.float32, self._device)
        if d.dim() != 2:
            raise ValueError('depth map must be 2-D')
        engine.fuse_depth_rigid(vol, self._tsdf_res, d, lw, self._K, self._Kinv, scale, center, self._tdist, wmax, mode=self._mode)
        self._last_vol = vol
        if on_device:
            return (tsdf, tsdf_w)
        out_t = vol.tsdf.cpu().numpy().astype(_as_np(tsdf).dtype, copy=False)
        out_w = vol.weight.cpu().numpy().astype(_as_np(tsdf_w).dtype, copy=False)
        if isinstance(tsdf, np.ndarray):
            tsdf[...] = out_t
            tsdf_w[...] = out_w
            return (tsdf, tsdf_w)
        return (out_t, out_w)

    def marching_cubes(self, tsdf=None, step_size=1):
        """core/fusion_dm.py:319-331: same as Fusion.marching_cubes but the step size defaults to 1 (the reference's FusionDM also
        leaves skimage's allow_degenerate at its default True here; the device extractor always drops degenerate triangles)."""
        return super().marching_cubes(tsdf, step_size)

    def compute_live_tsdf(self, depths, lws, UseAutoAlignment=False, useICP=False, outputMesh=False, *, mesh_path=None):
        """core/fusion_dm.py:95-178, plain multi-view branch: the volume stays on the device across views.  outputMesh=True
        saves the volume as `tsdf_temp.npy` and writes the zero level set to `test.obj` (core/fusion_dm.py:174-176) under
        `mesh_path` (default: $DFB_DATA_PATH or the working directory -- the reference's DATA_PATH is a checkout-relative constant)."""
        if len(depths) != len(lws):
            raise ValueError('length of camera matrix array Ks must equal that of depth maps')
        if UseAutoAlignment or useICP:
            raise NotImplementedError("auto-alignment / ICP are outside the hot path (SURVEY 2 row 2)")
        avg = np.array([-0.03, -0.43, -5.6], dtype='float32')       # core/fusion_dm.py:106-107
        std = 1.3
        scale = 8 * std / self._tsdf_res
        self._IND[0, 0] = self._IND[1, 1] = self._IND[2, 2] = scale
        self._IND[0:3, 3] = avg - scale * self._tsdf_res / 2
        self._INDinv = np.linalg.inv(self._IND)
        self._vol = None
        self._set_volume(None, None, shape=(self._tsdf_res,) * 3)
        for idx in range(len(depths)):
            self._depthidx = idx
            d = engine._to_dev(depths[idx], torch.float32, self._device)
            engine.fuse_depth_rigid(self._vol, self._tsdf_res, d, lws[idx], self._K, self._Kinv, 12 * std / self._tsdf_res, avg,
                                    self._tdist, 100.0, mode=self._mode)
        tsdf, tsdfw = self._tsdf, self._tsdfw
        if outputMesh:
            out_dir = mesh_path if mesh_path is not None else os.environ.get("DFB_DATA_PATH", ".")
            np.save(os.path.join(out_dir, 'tsdf_temp'), tsdf)
            self.write_canonical_mesh(out_dir, 'test.obj')
        return (tsdf, tsdfw)

    def updateTSDF(self, curr_tsdf, wmax=100.0):
        """core/fusion_dm.py:300-316: rigid volume->volume fusion with the global dq `_lw`."""
        if curr_tsdf is None:
            raise ValueError('tsdf of live frame has not been loaded')
        if curr_tsdf.ndim != 3:
            raise ValueError('Only accept 3D np array as tsdf')
        curr = engine._to_dev(curr_tsdf, torch.float32, self._device)
        engine.update_volume(self._vol, None, self._lw, curr, self._tdist, wmax, mode=self._mode, rigid=True)

    def setupCorrespondences(self, curr_tsdf, prune_result=True, tolerance=1.0, *, live_vertices=None):
        """core/fusion_dm.py:219-244: canonical vertices/normals moved by the global rigid dq `_lw`, k nearest live
        vertices, best point-to-plane candidate; vertices with best cost <= tolerance are kept in `_corridx` with their
        `_correspondences`.  `live_vertices` replaces `marching_cubes(curr_tsdf, step_size=1)`."""
        if self._vertices is None or self._normals is None:
            raise ValueError('canonical vertices/normals have not been set')
        lv = self._live_vertices(curr_tsdf, live_vertices)
        wv, wn = engine.warp_points(self._wf, self._lw, self._vertices, self._normals, k=0)
        best, cost = self._closest_points(lv, wv, wn)
        keep = torch.nonzero(cost <= tolerance).reshape(-1)
        self._corridx = [int(i) for i in keep.cpu().numpy()]
        self._correspondences = list(lv[best[keep].long()].cpu().numpy())

    def _rigid_problem(self):
        """Data term of core/fusion_dm.py:284-297 as a warp-field problem whose single node carries the identity
        transform (weight exp(-(d/2w)^2) = 1 for w = 1e30, so the blended dq is exactly [1,0,0,0,0,0,0,0])."""
        wf = engine.DeviceWarpField(1, self._device)
        wf.set_nodes(np.zeros((1, 3), np.float32), np.array([[1, 0, 0, 0, 0, 0, 0, 0]], np.float32), np.float32(1e30))
        idx = np.asarray(self._corridx, dtype=np.int64)
        return _gn.Problem(wf, self._vertices[idx], self._normals[idx], np.asarray(self._correspondences, dtype=np.float64).reshape(-1, 3),
                           np.zeros((len(idx), 1), np.int64), np.zeros(1, np.int64))

    def computef_lw(self, x):
        """core/fusion_dm.py:284-297: point-to-plane residuals of the kept correspondences under the rigid dq x."""
        return self._rigid_problem().residuals_lw(np.asarray(x, dtype=np.float64)).cpu().numpy()

    def solve(self, curr_tsdf, *, live_vertices=None, lw_iterations=100):
        """core/fusion_dm.py:262-281: three rounds of (correspondences, rigid least squares on `_lw`).  The reference's
        `least_squares(self.computef_lw, ...)` (finite-difference TRF) is replaced by a damped Gauss-Newton on the
        analytic 8x8 normal equations (csrc/gn.cu lw_normal_eq_kernel), as in Fusion.solve."""
        self._itercounter += 1
        for _ in range(3):
            self.setupCorrespondences(curr_tsdf, live_vertices=live_vertices)
            if not self._corridx:
                raise ValueError('no correspondence within tolerance')
            self._lw = self._rigid_problem().solve_lw(np.asarray(self._lw, dtype=np.float64), max_iter=lw_iterations, verbose=self._verbose)


class FusionDM_GPU(FusionDM):
    """Name kept for drop-in with test.py:158-159 (`FusionDM_GPU(0.2, K, tsdf_res=256, verbose=True)`)."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        if self._verbose:
            self.verbose_gpu()                                        # core/fusion_dm.py:573-574

    def verbose_gpu(self):
        """core/fusion_dm.py:576-598 lists the OpenCL platforms and devices; this lists the CUDA devices the library runs on."""
        print('\n' + '=' * 60 + '\nCUDA devices (libdfb_b200 version %d)' % int(_capi.lib().dfb_version()))
        for i in range(torch.cuda.device_count()):
            p = torch.cuda.get_device_properties(i)
            print('    Device %d - Name:  %s' % (i, p.name))
            print('    Device %d - Compute capability:  %d.%d' % (i, p.major, p.minor))
            print('    Device %d - Multiprocessors:  %d' % (i, p.multi_processor_count))
            print('    Device %d - Global Memory:  %.0f GB' % (i, p.total_memory / 1024.0 ** 3))
        print('\n')
