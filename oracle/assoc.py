"""CPU oracle, part 5: projective data association -- TEST INFRASTRUCTURE ONLY (see oracle/dq.py header).

DynamicFusion's correspondence step (SURVEY 8f rank 1): every warped canonical point is projected into the depth views and
paired with the back-projected pixel it lands on.  This module is the definition that the device kernel
(csrc/dfb_math.h assoc_projective_ref, csrc/graph.cu dfb_corr_projective) reproduces bit for bit, so every float64 operation
below is written in the kernel's order: rows of matrix-vector products summed left to right (`tsdf._matvec_rows`), dot products
left to right, no fused multiply-add.

Per point and view v (ascending):
  1. l = E_v [w,1], ln = R_v m (w, m without extrinsics);
  2. front-facing: ln.l < 0;
  3. projection exactly as the a2/a3 update (u = p0/p2, v = p1/p2, 0 <= u < cols-1, 0 <= v < rows-1, round half to even),
     and 1 <= ui <= cols-2, 1 <= vi <= rows-2 so that the four 4-neighbours exist;
  4. centre and neighbour depths z = -D > 0, |z_nb - z| <= max_distance;
  5. P(a,b) = Kinv [z a, z b, z] at the integer pixel; c = P(ui,vi);
     g = (P(ui+1,vi) - P(ui-1,vi)) x (P(ui,vi+1) - P(ui,vi-1)), negated when g.c > 0, rejected when g.c == 0;
  6. |l - c|^2 <= max_distance^2 and ln.g >= min_normal_dot |ln| |g|;
  7. cost |ln.(l - c)|; the smallest cost wins, strict < (ties keep the lower view).
Outputs: view (int32, -1 = none), cost (+inf = none), corr = R_v^T (c - t_v) (0 = none).
"""
import numpy as np

from .tsdf import _matvec_rows


def _dot(a, b):
    return a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1] + a[..., 2] * b[..., 2]


# centre, u-1, u+1, v-1, v+1
_OFFS = ((0, 0), (-1, 0), (1, 0), (0, -1), (0, 1))


def associate(warped_pts, warped_normals, dms, K, Kinv, max_distance, min_normal_dot, extrinsics=None):
    """warped_pts / warped_normals (M,3) float64; dms: (V,rows,cols) float32 depth maps (negative depth, 0 = no data).
    Returns (view (M,) int32, cost (M,) float64, corr (M,3) float64)."""
    w = np.asarray(warped_pts, dtype=np.float64).reshape(-1, 3)
    m = np.asarray(warped_normals, dtype=np.float64).reshape(-1, 3)
    K = np.asarray(K, dtype=np.float64)
    Kinv = np.asarray(Kinv, dtype=np.float64)
    md = float(max_distance)
    mnd = float(min_normal_dot)
    md2 = md * md
    n = len(w)
    best = np.full(n, -1, dtype=np.int32)
    best_cost = np.full(n, np.inf)
    corr = np.zeros((n, 3))
    ones = np.ones(n)
    for v, dm in enumerate(dms):
        dm = np.asarray(dm, dtype=np.float32)
        rows, cols = dm.shape
        E = None if extrinsics is None else np.asarray(extrinsics[v], dtype=np.float64).reshape(3, 4)
        if E is not None:
            l = _matvec_rows(E, [w[:, 0], w[:, 1], w[:, 2], ones])
            ln = _matvec_rows(E[:, :3], [m[:, 0], m[:, 1], m[:, 2]])
        else:
            l, ln = w, m
        with np.errstate(invalid='ignore', divide='ignore', over='ignore'):
            ok = _dot(ln, l) < 0
            p = _matvec_rows(K, [l[:, 0], l[:, 1], l[:, 2]])
            ok &= p[:, 2] != 0
            u = p[:, 0] / p[:, 2]
            vv = p[:, 1] / p[:, 2]
            ok &= (u >= 0) & (u < cols - 1) & (vv >= 0) & (vv < rows - 1)
            ui = np.where(ok, np.rint(np.where(ok, u, 0)), 1).astype(np.int64)
            vi = np.where(ok, np.rint(np.where(ok, vv, 0)), 1).astype(np.int64)
            ok &= (ui >= 1) & (ui <= cols - 2) & (vi >= 1) & (vi <= rows - 2)
            ui = np.where(ok, ui, 1)
            vi = np.where(ok, vi, 1)
            z = [-1.0 * dm[vi + dv, ui + du].astype(np.float64) for du, dv in _OFFS]
            ok &= z[0] > 0
            for j in range(1, 5):
                ok &= (z[j] > 0) & (np.abs(z[j] - z[0]) <= md)
            P = []
            for j, (du, dv) in enumerate(_OFFS):
                a = z[j] * (ui + du).astype(np.float64)
                b = z[j] * (vi + dv).astype(np.float64)
                P.append(_matvec_rows(Kinv, [a, b, z[j] * 1.0]))
            c = P[0]
            dU = P[2] - P[1]
            dV = P[4] - P[3]
            g = np.stack([dU[:, 1] * dV[:, 2] - dU[:, 2] * dV[:, 1],
                          dU[:, 2] * dV[:, 0] - dU[:, 0] * dV[:, 2],
                          dU[:, 0] * dV[:, 1] - dU[:, 1] * dV[:, 0]], axis=-1)
            gc = _dot(g, c)
            ok &= gc != 0
            g = np.where((gc > 0)[:, None], -g, g)
            d = l - c
            ok &= _dot(d, d) <= md2
            nl = np.sqrt(_dot(ln, ln))
            ng = np.sqrt(_dot(g, g))
            ok &= _dot(ln, g) >= (mnd * nl) * ng
            cost = np.abs(_dot(ln, d))
            upd = ok & (cost < best_cost)
            if E is not None:
                e = c - E[:, 3]
                cv = np.stack([(E[0, j] * e[:, 0] + E[1, j] * e[:, 1]) + E[2, j] * e[:, 2] for j in range(3)], axis=-1)
            else:
                cv = c
        best = np.where(upd, np.int32(v), best).astype(np.int32)
        best_cost = np.where(upd, cost, best_cost)
        corr = np.where(upd[:, None], cv, corr)
    return best, best_cost, corr
