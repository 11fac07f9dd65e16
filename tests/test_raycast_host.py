"""Raycasting the fused volume on the CPU: the host build of the per-ray function (csrc/dfb_raycast.h via
tests/hostshim/raycast_shim.cpp) against the oracle (oracle/raycast.py) bit for bit on a fused body volume and on knife edges,
known answers on a plane and a sphere, the box clip's margin, consistency with the tracker (oracle/track.py, engine.track_rigid),
agreement with the mesh path (oracle/mc.py + oracle/render.py), and the C-ABI argument validation of dfb_raycast.
tests/test_gpu_raycast.py runs the device kernel."""
import ctypes

import numpy as np
import pytest

import hostshim_api as hs
from dynamicfusion_body_b200 import engine, synth
from oracle import raycast as orc
from oracle import track as otr
from track_scenes import Ring, perturb, pose_error

# dyadic intrinsics: pixel (r, c) at depth z back-projects exactly to ((c - CX) z / F, (r - CY) z / F, z)
F, CX, CY = 16.0, 8.0, 6.0
K = np.array([[F, 0, CX], [0, F, CY], [0, 0, 1.0]])
ROWS, COLS = 13, 17
IDENT = np.concatenate([np.eye(3), np.zeros((3, 1))], 1)


def _both(T, W, res, scale, center, tdist, Kc, rows, cols, E, step=None, z_near=0.0, z_far=None):
    """host build and oracle on the same input, bit for bit; returns the oracle's (depth, normal, z*) of every view."""
    E = np.asarray(E, dtype=np.float64).reshape(-1, 3, 4)
    step = float(scale) if step is None else float(step)
    if z_far is None:
        z_far = max(engine.raycast_far(np.shape(T), res, engine.camera_views(Kc, rows, cols, E), scale, center), z_near + step)
    dh, nh = hs.raycast(T, W, res, scale, center, tdist, Kc, rows, cols, E, step, z_near, z_far)
    out = [orc.raycast_view(T, W, res, scale, center, tdist, np.linalg.inv(Kc), e, rows, cols, step, z_near, z_far) for e in E]
    do, no, zo = (np.stack([o[i] for o in out]) for i in range(3))
    assert np.array_equal(dh.view(np.uint32), do.view(np.uint32))
    assert np.array_equal(nh.view(np.uint32), no.view(np.uint32))
    assert np.array_equal(do, np.where(np.isnan(zo), 0.0, -zo.astype(np.float32)).astype(np.float32))
    return do, no, zo


def _linear_volume(R, a, b):
    i = np.indices((R, R, R)).astype(np.float64)
    return (a[0] * i[0] + a[1] * i[1] + a[2] * i[2] + b).astype(np.float32), np.ones((R, R, R), np.float32)


def _rays(lw, Kc, rows, cols):
    """camera centre C and world directions dw = R^T Kinv [c, r, 1] (camera z = 1) of every pixel."""
    lw = np.asarray(lw, dtype=np.float64)
    r, c = np.mgrid[0:rows, 0:cols]
    d = np.stack([c, r, np.ones_like(c)], -1).astype(np.float64) @ np.linalg.inv(Kc).T
    return -lw[:, :3].T @ lw[:, 3], d @ lw[:, :3]


# ---------------------------------------------------------------------------------------------------------------------------
# host build == oracle on the fused body volume


@pytest.fixture(scope="module")
def ring64():
    rg = Ring(64)
    T, W = rg.fuse_oracle([rg.pose(-20.0), rg.pose(20.0)])
    return rg, T, W


def _half_K(rg):
    Kh = rg.K.copy()
    Kh[:2] *= 0.5
    return Kh


@pytest.mark.parametrize("step", [0.5, 1.0, 2.5])
@pytest.mark.parametrize("n_views", [1, 3])
def test_host_build_equals_oracle_on_a_fused_volume(ring64, step, n_views):
    rg, T, W = ring64
    E = [rg.pose(0.0), perturb(rg.pose(15.0), 2.0, 1.0, 4), rg.pose(-30.0, 1.2)][:n_views]
    d, n, _ = _both(T, W, rg.res, rg.scale, rg.center, rg.tdist, _half_K(rg), 240, 320, E, step)
    hit = d != 0
    assert hit.mean(axis=(1, 2)).min() > 0.05
    assert np.allclose(np.linalg.norm(n[hit], axis=-1), 1.0, atol=1e-6)


def test_z_far_that_cuts_the_body(ring64):
    rg, T, W = ring64
    lw = rg.pose(0.0)
    d_all, _, _ = _both(T, W, rg.res, rg.scale, rg.center, rg.tdist, _half_K(rg), 240, 320, [lw], 1.0)
    cut = float(np.median(-d_all[d_all != 0]))
    d, _, z = _both(T, W, rg.res, rg.scale, rg.center, rg.tdist, _half_K(rg), 240, 320, [lw], 1.0, 0.0, cut)
    hit = d != 0
    assert 0 < hit.sum() < (d_all != 0).sum()
    assert np.all(z[hit] <= cut + 1e-9)                                          # z* <= z_k+1 <= z_far
    assert np.array_equal(d[hit], d_all[hit])                                    # a hit before the cut is the same hit


# ---------------------------------------------------------------------------------------------------------------------------
# known answers


@pytest.mark.parametrize("scale,center,deg", [(1.0, (0.0, 0.0, 0.0), 0.0), (0.25, (0.5, -1.0, 2.0), 10.0)])
def test_plane_gives_the_ray_plane_depth_and_normal(scale, center, deg):
    """D = a.g + b is reproduced exactly by the trilinear interpolant, so the one linear refinement lands on the plane."""
    R, a, b = 32, np.array([0.125, -0.0625, -0.5]), 8.0                       # dyadic: exact in float32 storage
    T, W = _linear_volume(R, a, b)
    center = np.array(center)
    lw = perturb(IDENT, deg, 0.05, 1) if deg else IDENT
    d, n, z = _both(T, W, R, scale, center, 1e3, K, ROWS, COLS, [lw], 0.1 * scale)
    C, dw = _rays(lw, K, ROWS, COLS)
    alpha = a @ ((C - center) / scale + R / 2.0) + b                          # D(z) = alpha + beta z along each ray
    beta = dw @ a / scale
    truth = -alpha / beta
    hit = d[0] != 0
    assert hit.sum() >= 0.9 * ROWS * COLS
    assert np.all(np.abs(z[0][hit] - truth[hit]) <= 1e-12 * truth[hit])
    assert np.allclose(n[0][hit], (a / np.linalg.norm(a)).astype(np.float32), rtol=0, atol=1e-7)


def _sphere(R, s, rho, tdist):
    i = np.indices((R, R, R)).astype(np.float64)
    sdf = np.sqrt(((i - np.asarray(s, dtype=np.float64).reshape(3, 1, 1, 1)) ** 2).sum(0)) - rho
    return np.clip(sdf, -tdist, tdist).astype(np.float32), np.ones((R, R, R), np.float32)


# measured: max depth error 0.0395 voxel over pixels whose normal faces the camera by more than 60 degrees (bound: 3 / (8 rho cos)
# <= 0.0625 there), max normal error 3.16 degrees (the trilinear gradient is continuous only inside a cell)
SPHERE_DEPTH_BAR, SPHERE_NORMAL_DEG = 0.06, 5.0


def test_sphere_depth_within_the_trilinear_error_bound():
    """A sphere SDF of radius rho (voxels): trilinear interpolation of a function with Hessian norm <= 1/rho errs by at most
    3/(8 rho) per unit grid spacing, so a hit seen at incidence angle theta is within 3/(8 rho cos theta) of the true sphere."""
    R, rho, tdist = 48, 12.0, 4.0
    s = np.array([23.5, 24.25, 24.0])
    T, W = _sphere(R, s, rho, tdist)
    Kc = np.array([[60.0, 0, 31.5], [0, 60.0, 23.5], [0, 0, 1.0]])
    lw = synth.look_at_extrinsic((24.0 - R / 2, 10.0 - R / 2, -40.0), s - R / 2)      # scale 1, center 0: world = grid - R/2
    d, n, z = _both(T, W, R, 1.0, np.zeros(3), tdist, Kc, 48, 64, [lw], 0.5)
    C, dw = _rays(lw, Kc, 48, 64)
    oc = C - (s - R / 2)
    bq = (dw * oc).sum(-1)
    aq = (dw * dw).sum(-1)
    disc = bq * bq - aq * ((oc * oc).sum() - rho * rho)
    truth = (-bq - np.sqrt(np.maximum(disc, 0))) / aq
    on = disc > 0
    hit = d[0] != 0
    p = C + z[0][..., None] * dw
    nt = (p - (s - R / 2)) / np.linalg.norm(p - (s - R / 2), axis=-1, keepdims=True)
    cos = -(nt * dw).sum(-1) / np.linalg.norm(dw, axis=-1)
    face = hit & on & (cos > 0.5)
    assert face.sum() > 300 and np.all(hit[on & (disc > 0.2 * aq * rho * rho)])     # every ray well inside the disc hits
    err = np.abs(z[0] - truth) * np.linalg.norm(dw, axis=-1)                           # along the ray, world = voxel units
    ang = np.degrees(np.arccos(np.clip((n[0].astype(np.float64) * nt).sum(-1), -1, 1)))
    print("sphere: max depth error %.4f voxel, max normal error %.3f deg" % (err[face].max(), ang[face].max()))
    assert np.all(err[face] <= 3.0 / (8.0 * rho) / cos[face])
    assert err[face].max() < SPHERE_DEPTH_BAR and ang[face].max() < SPHERE_NORMAL_DEG


# ---------------------------------------------------------------------------------------------------------------------------
# knife edges (identity pose, scale 1, center 0, R = 16: the centre pixel (6, 8) looks along +z at grid (8, 8, z + 8))


def _z_volume(D_of_gz, R=16):
    gz = np.arange(R, dtype=np.float64)
    T = np.broadcast_to(D_of_gz(gz), (R, R, R)).astype(np.float32).copy()
    return T, np.ones((R, R, R), np.float32)


def test_a_sample_exactly_on_the_surface_is_a_hit():
    T, W = _z_volume(lambda g: 0.5 * (12.0 - g))                              # D = 0 at g_z = 12: sample k = 4 (z = 4)
    d, n, z = _both(T, W, 16, 1.0, np.zeros(3), 100.0, K, ROWS, COLS, [IDENT], 1.0)
    assert z[0, 6, 8] == 4.0 and d[0, 6, 8] == -4.0                          # z* = z_3 + 1 * (0.5 / (0.5 - 0))
    assert np.array_equal(n[0, 6, 8], [0.0, 0.0, -1.0])


def test_refined_point_in_a_gated_cell_is_no_hit():
    """Samples at g_z = 9.5 and 12.5 (step 3) straddle the zero at 10.5, whose cell [10, 11] shares no corner plane with theirs
    along z: a zero weight on the plane g_z = 11 gates the refined point alone."""
    T, W = _z_volume(lambda g: 0.5 * (10.5 - g))
    d, _, z = _both(T, W, 16, 1.0, np.zeros(3), 100.0, K, ROWS, COLS, [IDENT], 3.0, 1.5)
    assert z[0, 6, 8] == 2.5 and d[0, 6, 8] == -2.5
    W2 = W.copy()
    W2[:, :, 11] = 0.0
    d, _, z = _both(T, W2, 16, 1.0, np.zeros(3), 100.0, K, ROWS, COLS, [IDENT], 3.0, 1.5)
    assert d[0, 6, 8] == 0 and np.isnan(z[0, 6, 8])


def test_camera_inside_the_body_sees_back_faces_only():
    R, rho = 32, 10.0
    T, W = _sphere(R, (16.0, 16.0, 16.0), rho, 3.0)
    d, n, _ = _both(T, W, R, 1.0, np.zeros(3), 3.0, K, ROWS, COLS, [IDENT], 0.5)   # camera at the sphere's centre
    assert not d.any() and not n.any()


def test_z_near_beyond_the_surface():
    R, rho = 32, 6.0
    T, W = _sphere(R, (16.0, 16.0, 24.0), rho, 3.0)                          # front at z = 2 on the axis, back at z = 14
    d, _, _ = _both(T, W, R, 1.0, np.zeros(3), 3.0, K, ROWS, COLS, [IDENT], 0.5)
    assert d[0, 6, 8] != 0 and -d[0, 6, 8] == pytest.approx(2.0, abs=0.05)
    for z_near in (5.0, 20.0):                                                # inside the body: back face; past it: nothing
        d, _, _ = _both(T, W, R, 1.0, np.zeros(3), 3.0, K, ROWS, COLS, [IDENT], 0.5, z_near)
        assert not d.any()


def test_camera_looking_away(ring64):
    rg, T, W = ring64
    lw0 = rg.pose(0.0)
    eye = -lw0[:, :3].T @ lw0[:, 3]
    away = synth.look_at_extrinsic(eye, 2 * eye - rg.target)
    d, n, _ = _both(T, W, rg.res, rg.scale, rg.center, rg.tdist, _half_K(rg), 60, 80, [away], 1.0, 0.0, 400.0)
    assert not d.any() and not n.any()
    kf, kl = orc.clip(T.shape, rg.res, rg.scale, rg.center, np.linalg.inv(_half_K(rg)), away, *np.mgrid[0:60, 0:80], 1.0, 0.0, 400.0)
    assert np.all(kf > kl)                                                    # the clip leaves no sample to take


def test_rays_that_miss_the_box_and_a_box_entry_on_a_sample():
    # camera in front of the box (grid z = -2) looking along +z: the centre ray enters the cell range at g_z = 0 exactly on
    # sample k = 2 with D = 0.5 there and 0 at the next sample; the clip must keep k = 2 for the hit at g_z = 1
    T, W = _z_volume(lambda g: 0.5 * (1.0 - g))
    lw = IDENT.copy()
    lw[2, 3] = 10.0                                                           # camera at world z = -10: grid z = -2
    d, _, z = _both(T, W, 16, 1.0, np.zeros(3), 100.0, K, ROWS, COLS, [lw], 1.0)
    kf, kl = orc.clip(T.shape, 16, 1.0, np.zeros(3), np.linalg.inv(K), lw, [6.0], [8.0], 1.0, 0.0, 40.0)
    assert kf[0] <= 2 <= kl[0]
    assert z[0, 6, 8] == 3.0 and d[0, 6, 8] == -3.0
    # a wide camera beside the box: its outer rays never meet it, the clip takes no sample for them
    Kw = np.array([[2.0, 0, CX], [0, 2.0, CY], [0, 0, 1.0]])
    side = IDENT.copy()
    side[0, 3] = -20.0                                                        # camera at world x = +20, outside the box
    d, _, _ = _both(T, W, 16, 1.0, np.zeros(3), 100.0, Kw, ROWS, COLS, [side], 1.0, 0.0, 40.0)
    kf, kl = orc.clip(T.shape, 16, 1.0, np.zeros(3), np.linalg.inv(Kw), side, *np.mgrid[0:ROWS, 0:COLS], 1.0, 0.0, 40.0)
    assert not d.any() and (kf > kl).any() and (kf <= kl).any()


@pytest.mark.parametrize("seed", [0, 1])
def test_box_clip_keeps_every_sample_in_the_cell_range(seed):
    """The clip is a pure saving: every sample whose cell passes the range test lies inside [first k, last k], for cameras in,
    beside and around the box, grazing rays included."""
    rng = np.random.default_rng(seed)
    R, scale, center = 12, 0.5, np.array([0.25, -0.5, 1.0])
    Kc = np.array([[6.0, 0, 8.0], [0, 6.0, 6.0], [0, 0, 1.0]])
    rr, cc = (a.ravel().astype(np.float64) for a in np.mgrid[0:ROWS, 0:COLS])
    for _ in range(20):
        eye = center + rng.uniform(-6, 6, 3)
        lw = synth.look_at_extrinsic(eye, center + rng.uniform(-2, 2, 3))
        if rng.random() < 0.3:                                                # axis-aligned views: dg == 0 on two axes
            lw = IDENT.copy()
            lw[:, 3] = -eye
        step, z_near = rng.choice([0.1, 0.37, 1.0]), rng.choice([0.0, 0.5])
        kf, kl = orc.clip((R, R, R), R, scale, center, np.linalg.inv(Kc), lw, rr, cc, step, z_near, 30.0)
        for k in range(int(30.0 / step) + 2):
            z = np.full(len(rr), z_near + k * step)
            ok, _, _ = orc._point_cell(np.linalg.inv(Kc), lw, center, scale, R / 2.0, (R, R, R), rr, cc, z)
            ok &= z <= 30.0
            assert np.all((kf[ok] <= k) & (k <= kl[ok]))


def test_oracle_sample_is_the_tracker_pixel(ring64):
    """The oracle's samples are the tracker's pixels: at float32-representable depths, validity, D and grad equal
    oracle/track.py bit for bit."""
    rg, T, W = ring64
    lw = rg.pose(5.0)
    dm = rg.frame(lw)
    px = otr.pixels(T, W, rg.res, rg.scale, rg.center, dm, rg.Kinv, lw, 1, rg.tdist)
    rr, cc = (a.ravel() for a in np.mgrid[0:rg.rows, 0:rg.cols])
    ok, D, g = orc.sample(T, W, rg.res, rg.scale, rg.center, rg.tdist, rg.Kinv, lw, rr, cc, -dm.ravel().astype(np.float64))
    ok &= dm.ravel() < 0
    assert np.array_equal(ok, px["ok"]) and ok.sum() > 10_000
    assert np.array_equal(D[ok].view(np.uint64), px["D"][ok].view(np.uint64))
    assert np.array_equal(g[ok].view(np.uint64), px["grad"][ok].view(np.uint64))


# ---------------------------------------------------------------------------------------------------------------------------
# consistency with tracking and with the mesh path

# measured on the 64^3 ring (step 1 voxel): median |rho| 0.0053 voxel, max 0.57 voxel.  The one linear refinement lands on the
# chord of the interpolant between two samples, not on its zero; the largest residuals are rays that cross the band obliquely
RESIDUAL_MEDIAN_BAR, RESIDUAL_MAX_BAR = 0.02, 1.0


def _frame(rg, T, W, lw, step=1.0):
    E = [lw]
    z_far = engine.raycast_far(T.shape, rg.res, engine.camera_views(rg.K, rg.rows, rg.cols, E), rg.scale, rg.center)
    return orc.raycast(T, W, rg.res, rg.scale, rg.center, rg.tdist, rg.K, rg.rows, rg.cols, E, step, 0.0, z_far)[0][0]


def test_track_residual_of_a_raycast_frame_is_near_zero(ring64):
    rg, T, W = ring64
    lw = rg.pose(5.0)
    dm = _frame(rg, T, W, lw)
    _, res = otr.normal_eq(T, W, rg.res, rg.scale, rg.center, dm, rg.Kinv, lw, 1, rg.tdist, 0.5 * rg.tdist, want_residual=True)
    ok = ~np.isnan(res)
    a = np.abs(res[ok]) / rg.scale
    print("raycast frame residual: %d of %d hits contribute, median %.2e, max %.2e voxel" % (ok.sum(), (dm != 0).sum(), np.median(a), a.max()))
    assert ok.sum() >= 0.95 * (dm != 0).sum()
    assert np.median(a) < RESIDUAL_MEDIAN_BAR and a.max() < RESIDUAL_MAX_BAR


# measured with the oracle: 0.0068 deg and 0.0073 voxel for each of seeds 1 / 2 / 3 (the loop ends at the same pose), against
# 0.045-0.070 deg and 0.075-0.112 voxel for the splatted frames of tests/test_track_host.py
ROT_BAR_DEG, TRANS_BAR_VOX = 0.02, 0.03


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_oracle_track_rigid_recovers_the_pose_of_a_raycast_frame(ring64, seed):
    rg, T, W = ring64
    truth = rg.pose(0.0)
    dm = _frame(rg, T, W, truth)
    lw0 = perturb(truth, 2.0, 1.0, seed)
    res = engine.track_rigid(lambda lw, s: otr.normal_eq(T, W, rg.res, rg.scale, rg.center, dm, rg.Kinv, lw, s, rg.tdist, 0.5 * rg.tdist), lw0)
    rot, tr = pose_error(res.lw, truth)
    print("seed %d: %.4f deg, %.4f voxel, iterations %s, converged %s" % (seed, rot, tr / rg.scale, res.iterations, res.converged))
    assert rot < ROT_BAR_DEG and tr / rg.scale < TRANS_BAR_VOX


# measured: hit/no-hit agreement 0.984, median |dz| 0.0097 voxel over the 79201 pixels both hit
MESH_AGREE_BAR, MESH_MEDIAN_DZ_BAR = 0.97, 0.03


def test_agreement_with_the_extracted_and_rasterised_mesh(ring64):
    """The mesh path (marching cubes of the tsdf at level 0, oracle/mc.py, rasterised by oracle/render.py) and the raycast see
    different surfaces by definition (linear edge interpolation of every cell against the gated trilinear interpolant), so this
    bounds their difference rather than pinning it."""
    from oracle import mc as omc
    from oracle import render as ore
    rg, T, W = ring64
    lw = rg.pose(0.0)
    verts, faces, _, _ = omc.marching_cubes(T, 1, level=0.0)
    pts = rg.scale * (verts.astype(np.float64) - rg.res / 2.0) + rg.center
    dr, _, _ = ore.render(pts, faces, rg.K, rg.rows, rg.cols, np.stack([lw]))
    dc = _frame(rg, T, W, lw)
    both = (dr[0] != 0) & (dc != 0)
    agree = ((dr[0] != 0) == (dc != 0)).mean()
    dz = np.abs(dr[0][both].astype(np.float64) - dc[both]) / rg.scale
    print("mesh vs raycast: agreement %.4f, median |dz| %.4f voxel, %d pixels both hit" % (agree, np.median(dz), both.sum()))
    assert agree > MESH_AGREE_BAR and np.median(dz) < MESH_MEDIAN_DZ_BAR


# ---------------------------------------------------------------------------------------------------------------------------


def test_argument_validation_without_gpu():
    from dynamicfusion_body_b200 import _capi
    lib = _capi.lib()
    p = ctypes.c_void_p(8)
    d3 = (ctypes.c_double * 3)()
    f64 = _capi.c_f64p

    def vol(x0=0, x1=16, r=16, t=8, w=8):
        v = _capi.Volume()
        v.tsdf, v.weight, v.rx, v.ry, v.rz, v.x0, v.x1 = t, w, r, r, r, x0, x1
        return v

    def views(n=1, rows=8, cols=8):
        v = engine.camera_views(K, 8, 8, n_views=1)
        v.n_views, v.rows, v.cols = n, rows, cols
        return v

    def call(v=None, res=16, scale=1.0, center=d3, vw=None, tdist=1.0, step=1.0, z_near=0.0, z_far=10.0, depth=p, normal=p):
        v = vol() if v is None else v
        vw = views() if vw is None else vw
        return lib.dfb_raycast(ctypes.byref(v) if v is not False else None, res, scale,
                               ctypes.cast(center, f64) if center is not None else None, ctypes.byref(vw) if vw is not False else None,
                               tdist, step, z_near, z_far, depth, normal, None)
    inf, nan = float("inf"), float("nan")
    cases = [(dict(v=False), b"null pointer"), (dict(center=None), b"null pointer"), (dict(vw=False), b"null pointer"),
             (dict(depth=None), b"null pointer"), (dict(normal=None), b"null pointer"), (dict(v=vol(t=0)), b"null pointer"),
             (dict(v=vol(w=0)), b"null pointer"), (dict(v=vol(r=1, x1=1)), b"smaller than one cell"),
             (dict(v=vol(0, 8)), b"slab"), (dict(v=vol(8, 16)), b"slab"), (dict(res=0), b"tsdf_res"),
             (dict(vw=views(n=0)), b"n_views"), (dict(vw=views(n=9)), b"n_views"), (dict(vw=views(rows=0)), b"empty"),
             (dict(vw=views(cols=0)), b"empty"), (dict(scale=0.0), b"scale"), (dict(scale=-1.0), b"scale"),
             (dict(tdist=0.0), b"truncation"), (dict(tdist=-1.0), b"truncation"), (dict(step=0.0), b"step"),
             (dict(step=-1.0), b"step"), (dict(z_near=-1.0), b"z_near"), (dict(z_near=10.0), b"z_near"),
             (dict(z_near=11.0), b"z_near"), (dict(z_far=inf), b"z_near"), (dict(z_far=nan), b"z_near"),
             (dict(z_near=nan), b"z_near"), (dict(step=1e-9), b"2^30")]
    for kw, msg in cases:
        assert call(**kw) == -1, kw
        assert msg in lib.dfb_last_error(), (kw, lib.dfb_last_error())
