"""CPU oracle, part 6: z-buffer rasterisation of a triangle mesh -- TEST INFRASTRUCTURE ONLY (see oracle/dq.py header).

The depth / face-id / normal maps of the live model as the live cameras see it (the reference renders depth and vertex ids with
GL, core/gl/glrender.py).  This module is the definition that the device kernels (csrc/dfb_render.h, csrc/render.cu
dfb_render) reproduce bit for bit, so every float64 operation below is written in the kernel's order: rows of matrix-vector
products summed left to right (`tsdf._matvec_rows`), dot products left to right, no fused multiply-add.

Per view v and face t = (a, b, c):
  1. culled when an index lies outside [0, n);
  2. l_i = E_v [P_i, 1] (P_i without extrinsics); culled unless every l_i.z > 0 (no near-plane clipping);
  3. q_i = K l_i, x_i = q_i0 / q_i2, y_i = q_i1 / q_i2; pixel (r, c) is sampled at its centre x = c, y = r;
  4. E(a, b, p) = (xb - xa)(py - ya) - (yb - ya)(px - xa), each product rounded; A = E(v0, v1, v2), culled when A == 0 or
     not finite;
  5. box: columns ceil(min x_i) .. floor(max x_i), rows likewise, clamped in float64 to the image; empty when lo > hi;
  6. pixel p of the box is covered when e0 = E(v1, v2, p), e1 = E(v2, v0, p), e2 = E(v0, v1, p) are all >= 0 (A > 0) or all
     <= 0 (A < 0): edges are inclusive, and the depth test decides between faces that share one;
  7. inv = ((e0 w0 + e1 w1) + e2 w2) / A with w_i = 1 / l_i.z; skipped unless inv > 0; zf = float32(1 / inv);
  8. key = bits(zf) << 32 | t: the smallest key wins (the nearest float32 depth, ties to the lower face id).
Outputs per view, [rows][cols]: depth = -zf (0 = no face), face = t (-1), normal = the winning face's (Pb - Pa) x (Pc - Pa)
divided by its norm, float32, in the frame of pts and not turned toward the camera (0 = no face, or n.n == 0).
"""
import numpy as np

from .tsdf import _matvec_rows

EMPTY = np.uint64(0xFFFFFFFFFFFFFFFF)


def _edge(xa, ya, xb, yb, px, py):
    return (xb - xa) * (py - ya) - (yb - ya) * (px - xa)


def face_normals(pts, faces):
    """(f,3) float32 unit normals of the faces (0 where n.n == 0); indices must be valid."""
    P = np.asarray(pts, dtype=np.float64).reshape(-1, 3)
    f = np.asarray(faces, dtype=np.int64).reshape(-1, 3)
    a, b, c = P[f[:, 0]], P[f[:, 1]], P[f[:, 2]]
    u, v = b - a, c - a
    n = np.stack([u[:, 1] * v[:, 2] - u[:, 2] * v[:, 1],
                  u[:, 2] * v[:, 0] - u[:, 0] * v[:, 2],
                  u[:, 0] * v[:, 1] - u[:, 1] * v[:, 0]], axis=-1)
    nn = (n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]) + n[:, 2] * n[:, 2]
    with np.errstate(invalid='ignore', divide='ignore'):
        out = (n / np.sqrt(nn)[:, None]).astype(np.float32)
    out[nn == 0] = 0
    return out


def face_setup(pts, faces, K, E, rows, cols):
    """Steps 1-5 for one view.  Returns (keep (f,) bool, x (f,3), y (f,3), w (f,3), A (f,), c0, c1, r0, r1 (f,) int64)."""
    P = np.asarray(pts, dtype=np.float64).reshape(-1, 3)
    f = np.asarray(faces, dtype=np.int64).reshape(-1, 3)
    K = np.asarray(K, dtype=np.float64)
    n, nf = len(P), len(f)
    keep = ((f >= 0) & (f < n)).all(1)
    fi = np.where(keep[:, None], f, 0)
    x = np.zeros((nf, 3)); y = np.zeros((nf, 3)); w = np.zeros((nf, 3))
    if n == 0:
        keep[:] = False
        return keep, x, y, w, np.zeros(nf), *(np.zeros(nf, np.int64) for _ in range(4))
    ones = np.ones(nf)
    with np.errstate(invalid='ignore', divide='ignore', over='ignore'):
        for i in range(3):
            Pi = P[fi[:, i]]
            if E is not None:
                l = _matvec_rows(np.asarray(E, dtype=np.float64).reshape(3, 4), [Pi[:, 0], Pi[:, 1], Pi[:, 2], ones])
            else:
                l = Pi
            keep &= l[:, 2] > 0
            q = _matvec_rows(K, [l[:, 0], l[:, 1], l[:, 2]])
            x[:, i] = q[:, 0] / q[:, 2]
            y[:, i] = q[:, 1] / q[:, 2]
            w[:, i] = 1.0 / l[:, 2]
        A = _edge(x[:, 0], y[:, 0], x[:, 1], y[:, 1], x[:, 2], y[:, 2])
        keep &= (A != 0) & np.isfinite(A)
        cl = np.maximum(np.ceil(np.minimum(np.minimum(x[:, 0], x[:, 1]), x[:, 2])), 0.0)
        ch = np.minimum(np.floor(np.maximum(np.maximum(x[:, 0], x[:, 1]), x[:, 2])), float(cols - 1))
        rl = np.maximum(np.ceil(np.minimum(np.minimum(y[:, 0], y[:, 1]), y[:, 2])), 0.0)
        rh = np.minimum(np.floor(np.maximum(np.maximum(y[:, 0], y[:, 1]), y[:, 2])), float(rows - 1))
        keep &= (cl <= ch) & (rl <= rh)
    box = [np.where(keep, b, 0).astype(np.int64) for b in (cl, ch, rl, rh)]
    return keep, x, y, w, A, *box


def zbuffer(pts, faces, K, E, rows, cols, chunk=1 << 22):
    """Steps 1-8 for one view: the (rows*cols,) uint64 z-buffer (EMPTY where no face covers the pixel)."""
    keep, x, y, w, A, c0, c1, r0, r1 = face_setup(pts, faces, K, E, rows, cols)
    zb = np.full(rows * cols, EMPTY, dtype=np.uint64)
    ids = np.nonzero(keep)[0]
    if not len(ids):
        return zb
    bw = c1[ids] - c0[ids] + 1
    area = bw * (r1[ids] - r0[ids] + 1)
    ends = np.cumsum(area)
    start = 0
    while start < len(ids):                                       # faces in groups of about `chunk` box pixels
        stop = int(np.searchsorted(ends, (ends[start - 1] if start else 0) + chunk, side='right'))
        stop = max(stop, start + 1)
        sel = ids[start:stop]
        cnt = area[start:stop]
        t = np.repeat(sel, cnt)
        j = np.arange(int(cnt.sum())) - np.repeat(np.cumsum(cnt) - cnt, cnt)
        wdt = np.repeat(bw[start:stop], cnt)
        py = (r0[t] + j // wdt).astype(np.float64)
        px = (c0[t] + j % wdt).astype(np.float64)
        xt, yt, wt, At = x[t], y[t], w[t], A[t]
        with np.errstate(invalid='ignore', divide='ignore', over='ignore'):
            e0 = _edge(xt[:, 1], yt[:, 1], xt[:, 2], yt[:, 2], px, py)
            e1 = _edge(xt[:, 2], yt[:, 2], xt[:, 0], yt[:, 0], px, py)
            e2 = _edge(xt[:, 0], yt[:, 0], xt[:, 1], yt[:, 1], px, py)
            pos = (e0 >= 0) & (e1 >= 0) & (e2 >= 0)
            neg = (e0 <= 0) & (e1 <= 0) & (e2 <= 0)
            cov = np.where(At > 0, pos, neg)
            inv = ((e0 * wt[:, 0] + e1 * wt[:, 1]) + e2 * wt[:, 2]) / At
            cov &= inv > 0
            zf = (1.0 / np.where(cov, inv, 1.0)).astype(np.float32)
        key = (zf.view(np.uint32).astype(np.uint64) << np.uint64(32)) | t.astype(np.uint64)
        pix = py.astype(np.int64) * cols + px.astype(np.int64)
        np.minimum.at(zb, pix[cov], key[cov])
        start = stop
    return zb


def resolve(zb, pts, faces, rows, cols):
    """(depth (rows,cols) float32, face (rows,cols) int32, normal (rows,cols,3) float32) of one view's z-buffer."""
    hit = zb != EMPTY
    depth = np.zeros(rows * cols, np.float32)
    face = np.full(rows * cols, -1, np.int32)
    normal = np.zeros((rows * cols, 3), np.float32)
    zf = (zb[hit] >> np.uint64(32)).astype(np.uint32).view(np.float32)
    t = (zb[hit] & np.uint64(0xFFFFFFFF)).astype(np.int64)
    depth[hit] = -zf
    face[hit] = t
    if hit.any():
        f = np.asarray(faces, dtype=np.int64).reshape(-1, 3)
        normal[hit] = face_normals(pts, f[t])
    return depth.reshape(rows, cols), face.reshape(rows, cols), normal.reshape(rows, cols, 3)


def render(pts, faces, K, rows, cols, extrinsics=None, n_views=None):
    """pts (n,3) float64 in the live frame (as dfb_warp_points returns them), faces (f,3) int32; K (3,3); extrinsics None or
    (V,3,4).  Returns (depth (V,rows,cols) float32, face (V,rows,cols) int32, normal (V,rows,cols,3) float32)."""
    V = (1 if n_views is None else int(n_views)) if extrinsics is None else len(extrinsics)
    out = [resolve(zbuffer(pts, faces, K, None if extrinsics is None else extrinsics[v], rows, cols), pts, faces, rows, cols)
           for v in range(V)]
    return tuple(np.stack([o[i] for o in out]) for i in range(3))
