"""CPU oracle: raycasting the fused FusionDM volume -- TEST INFRASTRUCTURE ONLY (see oracle/dq.py header).

Depth and normal maps of the whole volume (tsdf, weight) seen from any camera, with no surface extraction.  This module DEFINES
what `dfb_raycast` (csrc/raycast.cu, per-ray arithmetic in csrc/dfb_raycast.h and csrc/dfb_track.h) computes, in float64
numpy, element-wise, in the order the device evaluates it, so both agree bit for bit.  The surface is the tracker's
(oracle/track.py): the same back-projection, grid mapping, gate and standard trilinear interpolant.

Per view v (world -> camera pose lw = [R|t] = E_v, identity without extrinsics) and pixel (r, c), sampled at x = c, y = r:
  1. samples z_k = z_near + k * step for k = 0, 1, ... while z_k <= z_far; camera point x = Kinv [c z, r z, z], world point
     p = R^T (x - t), grid coordinate g = (p - center) / scale + tsdf_res / 2: steps 2-4 of oracle/track.py, in its order;
  2. a sample is VALID when its cell passes the tracker's cell-range test (0 <= floor(g) <= r - 2) and gate (8 corners with
     weight > 0 and |tsdf| * scale < tdist); its value D is the tracker's interpolant;
  3. the march ends at the first pair of consecutive valid samples (k, k+1) whose signs change: D_k > 0 >= D_k+1 is a hit,
     D_k < 0 <= D_k+1 a back face (no hit); pairs with an invalid sample are skipped;
  4. one linear refinement z* = z_k + step * (D_k / (D_k - D_k+1)); value and gradient at z* with the same gate, no hit when
     it fails, else depth = -float32(z*) (stored negative, 0 = no hit) and normal = float32(grad / |grad|) in the world frame
     (0 when |grad| = 0);
  5. box clip (part of the definition, it only saves work): with d = Kinv [c, r, 1], o = R^T (0 - t), the ray's grid
     coordinate is about og + z dg, og = (o - center) / scale + tsdf_res / 2, dg = (R^T d) / scale.  Against the box
     [-1/2, r_a - 1/2] on every axis (half a cell wider than the cell range, so rounding can never clip a valid sample):
     z_in = max over axes of the entry depths, z_out = min of the exit depths (an axis with dg = 0 is all or nothing);
     k runs from max(0, ceil((z_in - z_near) / step) - 1) to min(floor((z_out - z_near) / step) + 1,
     floor((z_far - z_near) / step) + 1), and from none when z_in > z_out.
"""
import numpy as np

from .tsdf import _matvec_rows


def _point_cell(Kinv, lw, center, scale, half, R, rr, cc, z):
    """Steps 2-4 of oracle/track.py for pixels (rr, cc) at depths z: (in range, cell index (n,3) int64, fraction (n,3))."""
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        x = _matvec_rows(Kinv, [cc * z, rr * z, z])
        e = x - lw[:, 3]
        p = (lw[0, :3] * e[:, 0:1] + lw[1, :3] * e[:, 1:2]) + lw[2, :3] * e[:, 2:3]
        g = (p - center) / scale + half
        fl = np.floor(g)
        ok = np.ones(len(z), bool)
        for a in range(3):
            ok &= (fl[:, a] >= 0) & (fl[:, a] <= R[a] - 2)
    i = np.where(ok[:, None], fl, 0).astype(np.int64)
    return ok, i, g - fl


def _cell_value(tsdf, weight, scale, tdist, ok, i, f):
    """Steps 5-6 of oracle/track.py: (gate passed, D, grad D per grid unit (n,3))."""
    ok = ok.copy()
    v = np.zeros((len(ok), 2, 2, 2))
    for dx in (0, 1):
        for dy in (0, 1):
            for dz in (0, 1):
                t = tsdf[i[:, 0] + dx, i[:, 1] + dy, i[:, 2] + dz].astype(np.float64)
                wt = weight[i[:, 0] + dx, i[:, 1] + dy, i[:, 2] + dz].astype(np.float64)
                with np.errstate(invalid="ignore", over="ignore"):
                    ok &= (wt > 0) & (np.abs(t) * scale < tdist)
                v[:, dx, dy, dz] = t
    with np.errstate(invalid="ignore", over="ignore"):
        ix, iy, iz = 1.0 - f[:, 0], 1.0 - f[:, 1], 1.0 - f[:, 2]
        ez = v[..., 0] * iz[:, None, None] + v[..., 1] * f[:, 2, None, None]
        gz = v[..., 1] - v[..., 0]
        ey = ez[..., 0] * iy[:, None] + ez[..., 1] * f[:, 1, None]
        gy = ez[..., 1] - ez[..., 0]
        gzy = gz[..., 0] * iy[:, None] + gz[..., 1] * f[:, 1, None]
        D = ey[:, 0] * ix + ey[:, 1] * f[:, 0]
        grad = np.stack([ey[:, 1] - ey[:, 0], gy[:, 0] * ix + gy[:, 1] * f[:, 0], gzy[:, 0] * ix + gzy[:, 1] * f[:, 0]], 1)
    return ok, D, grad


def sample(tsdf, weight, tsdf_res, scale, center, tdist, Kinv, lw34, rr, cc, z):
    """Steps 1-2 for pixels (rr, cc) at camera depths z (float64): (valid, D, grad)."""
    tsdf = np.asarray(tsdf, dtype=np.float32)
    weight = np.asarray(weight, dtype=np.float32)
    lw = np.asarray(lw34, dtype=np.float64).reshape(3, 4)
    Kinv = np.asarray(Kinv, dtype=np.float64).reshape(3, 3)
    center = np.asarray(center, dtype=np.float64).reshape(3)
    rr, cc, z = (np.asarray(a, dtype=np.float64).ravel() for a in (rr, cc, z))
    ok, i, f = _point_cell(Kinv, lw, center, float(scale), tsdf_res / 2.0, tsdf.shape, rr, cc, z)
    return _cell_value(tsdf, weight, float(scale), float(tdist), ok, i, f)


def clip(shape, tsdf_res, scale, center, Kinv, lw34, rr, cc, step, z_near, z_far):
    """Step 5 for pixels (rr, cc): (first k, last k) as int64, first > last when the ray has no sample to take."""
    lw = np.asarray(lw34, dtype=np.float64).reshape(3, 4)
    Kinv = np.asarray(Kinv, dtype=np.float64).reshape(3, 3)
    center = np.asarray(center, dtype=np.float64).reshape(3)
    rr, cc = np.asarray(rr, dtype=np.float64).ravel(), np.asarray(cc, dtype=np.float64).ravel()
    n = len(rr)
    half = tsdf_res / 2.0
    d = _matvec_rows(Kinv, [cc, rr, np.ones(n)])
    e = 0.0 - lw[:, 3]
    z_in, z_out = np.full(n, -np.inf), np.full(n, np.inf)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        for a in range(3):
            o = (lw[0, a] * e[0] + lw[1, a] * e[1]) + lw[2, a] * e[2]
            og = (o - center[a]) / scale + half
            dg = ((lw[0, a] * d[:, 0] + lw[1, a] * d[:, 1]) + lw[2, a] * d[:, 2]) / scale
            lo, hi = -0.5, shape[a] - 0.5
            z0, z1 = (lo - og) / dg, (hi - og) / dg
            inside = (og >= lo) & (og <= hi)
            zl = np.where(dg != 0, np.where(z0 < z1, z0, z1), np.where(inside, -np.inf, np.inf))
            zh = np.where(dg != 0, np.where(z0 < z1, z1, z0), np.where(inside, np.inf, -np.inf))
            z_in = np.where(zl > z_in, zl, z_in)
            z_out = np.where(zh < z_out, zh, z_out)
        kf = np.ceil((z_in - z_near) / step) - 1.0
        kf = np.where(kf > 0.0, kf, 0.0)
        kcap = np.floor((z_far - z_near) / step) + 1.0
        kl = np.floor((z_out - z_near) / step) + 1.0
        kl = np.where(kl < kcap, kl, kcap)
        empty = ~(z_in <= z_out) | (kl < kf)
    kf = np.where(empty, 1.0, kf).astype(np.int64)
    kl = np.where(empty, 0.0, kl).astype(np.int64)
    return kf, kl


def raycast_view(tsdf, weight, tsdf_res, scale, center, tdist, Kinv, lw34, rows, cols, step, z_near, z_far):
    """Steps 1-5 for one view: (depth (rows,cols) float32, normal (rows,cols,3) float32, z* (rows,cols) float64, NaN = no hit)."""
    tsdf = np.asarray(tsdf, dtype=np.float32)
    weight = np.asarray(weight, dtype=np.float32)
    step, z_near, z_far = float(step), float(z_near), float(z_far)
    rr, cc = np.meshgrid(np.arange(rows, dtype=np.float64), np.arange(cols, dtype=np.float64), indexing="ij")
    rr, cc = rr.ravel(), cc.ravel()
    kf, kl = clip(tsdf.shape, tsdf_res, scale, center, Kinv, lw34, rr, cc, step, z_near, z_far)
    n = rows * cols
    hit = np.zeros(n, bool)
    z_lo, d_lo, d_hi = np.zeros(n), np.zeros(n), np.zeros(n)
    act = np.nonzero(kf <= kl)[0]
    k, kl = kf[act].copy(), kl[act]
    prev_ok, prev_d, prev_z = np.zeros(len(act), bool), np.zeros(len(act)), np.zeros(len(act))
    while len(act):
        z = z_near + k.astype(np.float64) * step
        live = z <= z_far
        ok, D, _ = sample(tsdf, weight, tsdf_res, scale, center, tdist, Kinv, lw34, rr[act], cc[act], z)
        ok &= live
        pair = prev_ok & ok
        front = pair & (prev_d > 0) & (D <= 0)
        back = pair & (prev_d < 0) & (D >= 0)
        hit[act[front]] = True
        z_lo[act[front]] = prev_z[front]
        d_lo[act[front]], d_hi[act[front]] = prev_d[front], D[front]
        go = live & ~front & ~back & (k < kl)
        act, k, kl, prev_ok, prev_d, prev_z = act[go], k[go] + 1, kl[go], ok[go], D[go], z[go]
    depth = np.zeros(n, np.float32)
    normal = np.zeros((n, 3), np.float32)
    zstar = np.full(n, np.nan)
    h = np.nonzero(hit)[0]
    if len(h):
        with np.errstate(invalid="ignore", divide="ignore"):
            zs = z_lo[h] + step * (d_lo[h] / (d_lo[h] - d_hi[h]))
        ok, _, g = sample(tsdf, weight, tsdf_res, scale, center, tdist, Kinv, lw34, rr[h], cc[h], zs)
        h, zs, g = h[ok], zs[ok], g[ok]
        depth[h] = -(zs.astype(np.float32))
        zstar[h] = zs
        nn = (g[:, 0] * g[:, 0] + g[:, 1] * g[:, 1]) + g[:, 2] * g[:, 2]
        with np.errstate(invalid="ignore", divide="ignore"):
            nrm = (g / np.sqrt(nn)[:, None]).astype(np.float32)
        nrm[nn == 0] = 0
        normal[h] = nrm
    return depth.reshape(rows, cols), normal.reshape(rows, cols, 3), zstar.reshape(rows, cols)


def raycast(tsdf, weight, tsdf_res, scale, center, tdist, K, rows, cols, extrinsics=None, step=None, z_near=0.0, z_far=None):
    """Depth (V,rows,cols) float32 and normal (V,rows,cols,3) float32 of the whole volume from the views `extrinsics` ((V,3,4)
    world -> camera, one identity view when None), intrinsics K (Kinv = inv(K), as engine.camera_views computes it).  step
    defaults to scale; z_far (required here) ends every ray."""
    Kinv = np.linalg.inv(np.asarray(K, dtype=np.float64))
    E = [np.concatenate([np.eye(3), np.zeros((3, 1))], 1)] if extrinsics is None else list(extrinsics)
    step = float(scale) if step is None else float(step)
    if z_far is None:
        raise ValueError("the oracle needs an explicit z_far")
    out = [raycast_view(tsdf, weight, tsdf_res, scale, center, tdist, Kinv, e, rows, cols, step, z_near, z_far) for e in E]
    return np.stack([o[0] for o in out]), np.stack([o[1] for o in out])
