"""CPU oracle: rigid point-to-TSDF tracking -- TEST INFRASTRUCTURE ONLY (see oracle/dq.py header).

Nothing in the reference tracks a FusionDM camera from depth alone: `compute_live_tsdf(useICP=True)` needs the reference's
ICP helpers and every pose comes from `proj*.txt`.  This module DEFINES what `dfb_track_normal_eq` (csrc/track.cu, per-pixel
arithmetic in csrc/dfb_track.h) computes, in float64 numpy, element-wise, in the order the device evaluates it -- so the gate,
the residual and the Jacobian of every pixel agree bit for bit and only the sums over pixels differ in their order.

For every pixel (r, c) with r % stride == 0 and c % stride == 0:
  1. z = -depth[r][c] (the project's convention: depth stored negative, 0 = no data); the pixel is skipped unless z > 0;
  2. camera point x = Kinv [c z, r z, z] (each row summed left to right, as `tsdf._matvec_rows`), world point p = R^T (x - t)
     for the pose lw = [R|t] (world -> camera, the `lw` of fuseDepths);
  3. grid coordinate g = (p - center) / scale + tsdf_res / 2, the inverse of fuseDepths' pos = scale (idx - tsdf_res/2) + center;
  4. cell i = floor(g) with 0 <= i_a <= r_a - 2 on every axis, fraction f = g - i;
  5. gate: every one of the 8 corners has weight > 0 and |tsdf| * scale < tdist (strict): unobserved voxels (+tdist, weight 0)
     and clamped ones carry no gradient;
  6. D = the STANDARD trilinear interpolant of the cell, evaluated along z, then y, then x.  This is a new definition: it is not
     `interpolate_tsdf` (core/util.py:102-137), whose y/z weights are swapped (Q1).  grad D is the analytic gradient of the same
     interpolant inside the cell, per grid unit;
  7. residual rho = scale * D (world units).  Its derivative under the twist xi = (tau, omega) acting on world points as
     p + tau + omega x p is J = [grad D, p x grad D] (grad_p g = I / scale cancels the scale of rho); Huber weight
     w = min(1, delta / |rho|).

Sums (29 float64): the upper triangle of H = sum w J^T J (21, row-major), g = sum w J rho (6), the Huber cost
sum(0.5 rho^2 if |rho| <= delta else delta (|rho| - delta / 2)) and the number of contributing pixels.
"""
import numpy as np

from .tsdf import _matvec_rows

N_SUMS = 29


def sampled_shape(rows, cols, stride):
    return (rows + stride - 1) // stride, (cols + stride - 1) // stride


def pixels(tsdf, weight, tsdf_res, scale, center, depth, Kinv, lw34, stride, tdist):
    """Steps 1-7 for every sampled pixel, flattened in (row, column) order of the sampled grid.  Returns a dict: ok (contributes),
    p (world points), g (grid coordinates), D, grad, rho, J (n, 6); values where ok is False are meaningless."""
    tsdf = np.asarray(tsdf, dtype=np.float32)
    weight = np.asarray(weight, dtype=np.float32)
    depth = np.asarray(depth, dtype=np.float32)
    rows, cols = depth.shape
    R = tsdf.shape
    lw34 = np.asarray(lw34, dtype=np.float64).reshape(3, 4)
    Kinv = np.asarray(Kinv, dtype=np.float64).reshape(3, 3)
    center = np.asarray(center, dtype=np.float64).reshape(3)
    rr, cc = np.meshgrid(np.arange(0, rows, stride), np.arange(0, cols, stride), indexing="ij")
    rr, cc = rr.ravel(), cc.ravel()
    z = -1.0 * depth[rr, cc].astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        ok = z > 0
        x = _matvec_rows(Kinv, [cc.astype(np.float64) * z, rr.astype(np.float64) * z, z])
        e = x - lw34[:, 3]
        p = (lw34[0, :3] * e[:, 0:1] + lw34[1, :3] * e[:, 1:2]) + lw34[2, :3] * e[:, 2:3]
        g = (p - center) / scale + tsdf_res / 2.0
        fl = np.floor(g)
        for a in range(3):
            ok &= (fl[:, a] >= 0) & (fl[:, a] <= R[a] - 2)
    i = np.where(ok[:, None], fl, 0).astype(np.int64)
    f = g - fl
    v = np.zeros((len(z), 2, 2, 2))
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
        ez = v[..., 0] * iz[:, None, None] + v[..., 1] * f[:, 2, None, None]          # (n, dx, dy)
        gz = v[..., 1] - v[..., 0]
        ey = ez[..., 0] * iy[:, None] + ez[..., 1] * f[:, 1, None]                     # (n, dx)
        gy = ez[..., 1] - ez[..., 0]
        gzy = gz[..., 0] * iy[:, None] + gz[..., 1] * f[:, 1, None]
        D = ey[:, 0] * ix + ey[:, 1] * f[:, 0]
        grad = np.stack([ey[:, 1] - ey[:, 0], gy[:, 0] * ix + gy[:, 1] * f[:, 0], gzy[:, 0] * ix + gzy[:, 1] * f[:, 0]], 1)
        rho = scale * D
        J = np.concatenate([grad, np.stack([p[:, 1] * grad[:, 2] - p[:, 2] * grad[:, 1],
                                            p[:, 2] * grad[:, 0] - p[:, 0] * grad[:, 2],
                                            p[:, 0] * grad[:, 1] - p[:, 1] * grad[:, 0]], 1)], 1)
    return dict(ok=ok, p=p, g=g, D=D, grad=grad, rho=rho, J=J)


def terms(rho, J, delta):
    """The 29 per-pixel terms (n, 29) of `pixels`' contributing pixels, in the order dfb_track.h:track_terms evaluates them."""
    ar = np.abs(rho)
    inside = ar <= delta
    with np.errstate(divide="ignore"):
        w = np.where(inside, 1.0, delta / ar)
    wJ = w[:, None] * J
    out = [wJ[:, a] * J[:, b] for a in range(6) for b in range(a, 6)]
    out += [wJ[:, a] * rho for a in range(6)]
    out.append(np.where(inside, 0.5 * (rho * rho), delta * (ar - 0.5 * delta)))
    out.append(np.ones_like(rho))
    return np.stack(out, 1)


def normal_eq(tsdf, weight, tsdf_res, scale, center, depth, Kinv, lw34, stride, tdist, delta, want_residual=False):
    """The 29 sums (float64) of the frame `depth` at pose lw34 against the whole volume (tsdf, weight), and, with
    want_residual, the residual map (ceil(rows/stride), ceil(cols/stride)) float64: rho, NaN where the pixel did not contribute."""
    px = pixels(tsdf, weight, tsdf_res, scale, center, depth, Kinv, lw34, stride, tdist)
    ok = px["ok"]
    sums = terms(px["rho"][ok], px["J"][ok], delta).sum(axis=0) if ok.any() else np.zeros(N_SUMS)
    if not want_residual:
        return sums
    res = np.where(ok, px["rho"], np.nan).reshape(sampled_shape(*np.shape(depth), stride))
    return sums, res


def unpack(sums):
    """(H (6,6) symmetric, g (6,), cost, count) from the 29 sums."""
    sums = np.asarray(sums, dtype=np.float64)
    H = np.zeros((6, 6))
    H[np.triu_indices(6)] = sums[:21]
    H = H + np.triu(H, 1).T
    return H, sums[21:27].copy(), float(sums[27]), int(round(sums[28]))
