"""Rigid point-to-TSDF tracking on the CPU: the oracle (oracle/track.py) on known answers, the host build of the per-pixel functions
(csrc/dfb_track.h via tests/hostshim/track_shim.cpp) against the oracle bit for bit on a fused body volume and on knife edges,
the Levenberg-Marquardt loop (engine.track_rigid) driven by the oracle, and the C-ABI argument validation of
dfb_track_normal_eq.  tests/test_gpu_track.py runs the device kernels."""
import ctypes

import numpy as np
import pytest

import hostshim_api as hs
from dynamicfusion_body_b200 import engine, synth
from oracle import track as otr
from track_scenes import Ring, perturb, pose_error

# dyadic intrinsics: pixel (r, c) at depth z back-projects exactly to ((c - CX) z / F, (r - CY) z / F, z)
F, CX, CY = 2.0, 8.0, 6.0
K = np.array([[F, 0, CX], [0, F, CY], [0, 0, 1.0]])
KINV = np.linalg.inv(K)
ROWS, COLS = 13, 17
IDENT = np.concatenate([np.eye(3), np.zeros((3, 1))], 1)


def _both(T, W, res, scale, center, dm, Kinv, lw, stride, tdist, delta):
    """host build and oracle on the same input: residual maps and Jacobians bit for bit, sums to rounding; returns the oracle's
    per-pixel dict and sums."""
    sh, rh, jh = hs.normal_eq(T, W, res, scale, center, dm, Kinv, lw, stride, tdist, delta)
    so, ro = otr.normal_eq(T, W, res, scale, center, dm, Kinv, lw, stride, tdist, delta, want_residual=True)
    px = otr.pixels(T, W, res, scale, center, dm, Kinv, lw, stride, tdist)
    assert np.array_equal(rh.view(np.uint64), ro.view(np.uint64))
    assert np.array_equal(jh.reshape(-1, 6).view(np.uint64), np.where(px["ok"][:, None], px["J"], 0.0).view(np.uint64))
    _assert_sums_close(sh, so)
    return px, so


def _assert_sums_close(a, b, rel=1e-12):
    """The 29 sums to `rel` of the Cauchy-Schwarz bound of each entry: |sum w J_i J_j| <= sqrt(H_ii H_jj) and
    |sum w J_i rho| <= sqrt(H_ii * 2 cost) (w rho^2 <= 2 Huber cost per pixel); cost relative, count exact."""
    Ha, ga, ca, na = otr.unpack(a)
    Hb, gb, cb, nb = otr.unpack(b)
    d = np.sqrt(np.abs(np.diag(Hb)))
    assert np.all(np.abs(Ha - Hb) <= rel * np.outer(d, d) + 1e-300)
    assert np.all(np.abs(ga - gb) <= rel * d * np.sqrt(2 * cb) + 1e-300)
    assert abs(ca - cb) <= rel * cb and na == nb


def _linear_volume(R, a, b):
    i = np.indices((R, R, R)).astype(np.float64)
    return (a[0] * i[0] + a[1] * i[1] + a[2] * i[2] + b).astype(np.float32), np.ones((R, R, R), np.float32)


@pytest.mark.parametrize("scale,center", [(1.0, (0.0, 0.0, 0.0)), (0.25, (0.5, -1.0, 2.0))])
def test_linear_volume_gives_exact_value_and_gradient(scale, center):
    R, a, b = 16, np.array([0.5, -0.25, 0.125]), 0.75            # dyadic: exact in float32 storage
    T, W = _linear_volume(R, a, b)
    rng = np.random.default_rng(5)
    dm = -rng.uniform(0.3, 3.0, size=(ROWS, COLS)).astype(np.float32)
    lw = perturb(IDENT, 10.0, 0.2, 1)
    px, sums = _both(T, W, R, scale, np.array(center), dm, KINV, lw, 1, 1e3, 0.5)
    ok = px["ok"]
    assert ok.sum() >= 20
    g = px["g"][ok]
    assert np.allclose(px["D"][ok], g @ a + b, rtol=0, atol=1e-12)
    assert np.allclose(px["grad"][ok], a, rtol=0, atol=1e-12)
    assert np.allclose(px["J"][ok][:, 3:], np.cross(px["p"][ok], a), rtol=0, atol=1e-12)
    assert np.array_equal(px["rho"][ok], scale * px["D"][ok])
    assert otr.unpack(sums)[3] == ok.sum()


def _corner_depth(lw, rows, cols, Kc, limit):
    """Ray-cast depth of the three walls x = 0, y = 0, z = 0 seen from inside the positive octant (0 beyond `limit`)."""
    lw = np.asarray(lw, dtype=np.float64)
    C = -lw[:, :3].T @ lw[:, 3]
    r, c = np.mgrid[0:rows, 0:cols]
    d = np.stack([c, r, np.ones_like(c)], -1).astype(np.float64) @ np.linalg.inv(Kc).T        # camera rays with z = 1
    dw = d @ lw[:, :3]                                                                          # R^T d
    with np.errstate(divide="ignore"):
        t = np.where(dw < 0, -C / dw, np.inf).min(-1)
    hit = C + t[..., None] * dw
    ok = np.isfinite(t) & (hit <= limit).all(-1)
    return np.where(ok, -t, 0.0).astype(np.float32)


def test_box_corner_recovers_a_known_offset():
    """Three orthogonal walls constrain all six degrees of freedom: the tracker finds the pose a frame was cast from."""
    R, tdist, scale, center = 48, 3.0, 1.0, np.full(3, 16.0)             # grid g = world + 8
    i = np.indices((R, R, R)).astype(np.float64) - 8.0
    T = np.clip(np.minimum(np.minimum(i[0], i[1]), i[2]), -tdist, tdist).astype(np.float32)
    W = np.ones((R, R, R), np.float32)
    Kc = np.array([[100.0, 0, 79.5], [0, 100.0, 59.5], [0, 0, 1.0]])
    lw0 = synth.look_at_extrinsic((26.0, 22.0, 30.0), (0.0, 0.0, 0.0))
    truth = perturb(lw0, 1.0, 0.5, 3)
    dm = _corner_depth(truth, 120, 160, Kc, 34.0)
    assert (dm != 0).mean() > 0.9
    res = engine.track_rigid(lambda lw, s: otr.normal_eq(T, W, R, scale, center, dm, np.linalg.inv(Kc), lw, s, tdist, 0.5 * tdist), lw0)
    rot, tr = pose_error(res.lw, truth)
    print("box corner: %.2e deg, %.2e world units, iterations %s" % (rot, tr, res.iterations))
    assert rot < 1e-3 and tr < 1e-3
    assert np.allclose(res.lw[:, :3] @ res.lw[:, :3].T, np.eye(3), atol=1e-12)


@pytest.fixture(scope="module")
def ring64():
    rg = Ring(64)
    T, W = rg.fuse_oracle([rg.pose(-20.0), rg.pose(20.0)])
    return rg, T, W


@pytest.mark.parametrize("stride", [1, 2, 4])
def test_host_build_equals_oracle_on_a_fused_volume(ring64, stride):
    rg, T, W = ring64
    for lw in (rg.pose(0.0), perturb(rg.pose(10.0), 2.0, 1.0, 7)):
        px, sums = _both(T, W, rg.res, rg.scale, rg.center, rg.frame(lw), rg.Kinv, lw, stride, rg.tdist, 0.5 * rg.tdist)
        assert px["ok"].sum() > 0.2 * (rg.rows // stride) * (rg.cols // stride) * 0.25


def test_knife_edges():
    R, tdist = 8, 0.5
    T, W = _linear_volume(R, np.array([0.01, 0.02, 0.03]), -0.2)           # |tsdf| <= 0.29 < tdist
    dm = np.zeros((ROWS, COLS), np.float32)
    # identity pose, scale 1, center 0: g = ((c - 8) z / 2, (r - 6) z / 2, z) + 4, exact
    cases = {(6, 8): (-2.0, True),      # g = (4, 4, 6): integers, i_z = R - 2 with f = 0
             (6, 9): (-3.0, False),     # g_z = 7 = R - 1
             (6, 7): (-2.5, True),      # g_z = 6.5 inside the last cell
             (7, 11): (-2.0, False),    # g_x = 7 = R - 1
             (7, 10): (-2.0, True),     # g_x = 6 = R - 2
             (8, 8): (0.0, False),      # no data
             (9, 8): (1.0, False),      # positive stored depth
             (4, 5): (-1.0, True)}      # g = (2.5, 3, 5): the cell the tdist / weight edges below act on
    for (r, c), (z, _) in cases.items():
        dm[r, c] = z
    px, _ = _both(T, W, R, 1.0, np.zeros(3), dm, KINV, IDENT, 1, tdist, 0.1)
    ok = px["ok"].reshape(ROWS, COLS)
    assert {rc: bool(ok[rc]) for rc in cases} == {rc: v[1] for rc, v in cases.items()}
    g = px["g"].reshape(ROWS, COLS, 3)
    assert np.array_equal(g[6, 8], [4.0, 4.0, 6.0]) and px["D"].reshape(ROWS, COLS)[6, 8] == np.float64(T[4, 4, 6])
    # the cell of pixel (4, 5) is x 2..3, y 3..4, z 5..6: one corner at |tsdf| scale == tdist drops it, just below keeps it
    for val, keep in ((tdist, False), (-tdist, False), (np.nextafter(np.float32(tdist), np.float32(0)), True)):
        T2 = T.copy()
        T2[3, 4, 6] = val
        px, _ = _both(T2, W, R, 1.0, np.zeros(3), dm, KINV, IDENT, 1, tdist, 0.1)
        assert bool(px["ok"].reshape(ROWS, COLS)[4, 5]) == keep, val
    W2 = W.copy()
    W2[2, 3, 5] = 0.0
    px, _ = _both(T, W2, R, 1.0, np.zeros(3), dm, KINV, IDENT, 1, tdist, 0.1)
    assert not px["ok"].reshape(ROWS, COLS)[4, 5]


def test_pose_looking_away_contributes_nothing(ring64):
    rg, T, W = ring64
    dm = rg.frame(rg.pose(0.0))
    lw0 = rg.pose(0.0)
    eye = -lw0[:, :3].T @ lw0[:, 3]
    away = synth.look_at_extrinsic(eye, 2 * eye - rg.target)            # the same camera turned to face away from the body
    sums = otr.normal_eq(T, W, rg.res, rg.scale, rg.center, dm, rg.Kinv, away, 1, rg.tdist, 0.5 * rg.tdist)
    sh, _, _ = hs.normal_eq(T, W, rg.res, rg.scale, rg.center, dm, rg.Kinv, away, 1, rg.tdist, 0.5 * rg.tdist)
    assert sums[28] == 0 and np.all(sh == 0)
    with pytest.raises(ValueError, match="pixels"):
        engine.track_rigid(lambda lw, s: otr.normal_eq(T, W, rg.res, rg.scale, rg.center, dm, rg.Kinv, lw, s, rg.tdist, 0.5 * rg.tdist), away)


# measured with the oracle (DESIGN §7): 0.045 / 0.062 / 0.070 deg and 0.075 / 0.096 / 0.112 voxel for seeds 1 / 2 / 3
ROT_BAR_DEG, TRANS_BAR_VOX = 0.15, 0.25


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_oracle_track_rigid_recovers_a_perturbed_pose(ring64, seed):
    """A frame rendered 2 degrees (seeded axis) and 1 voxel (seeded direction) away from a pose is tracked from that pose."""
    rg, T, W = ring64
    lw0 = rg.pose(0.0)
    truth = perturb(lw0, 2.0, 1.0, seed)
    dm = rg.frame(truth)
    res = engine.track_rigid(lambda lw, s: otr.normal_eq(T, W, rg.res, rg.scale, rg.center, dm, rg.Kinv, lw, s, rg.tdist, 0.5 * rg.tdist), lw0)
    rot, tr = pose_error(res.lw, truth)
    print("seed %d: %.4f deg, %.4f voxel, iterations %s, converged %s" % (seed, rot, tr, res.iterations, res.converged))
    assert rot < ROT_BAR_DEG and tr < TRANS_BAR_VOX
    assert np.allclose(res.lw[:, :3] @ res.lw[:, :3].T, np.eye(3), atol=1e-12)
    assert len(res.iterations) == 3 and res.pixels > 50_000


def test_argument_validation_without_gpu():
    from dynamicfusion_body_b200 import _capi
    lib = _capi.lib()
    assert lib.dfb_track_workspace_doubles(480, 640, 1) == 29 * ((480 * 640 + 255) // 256)
    assert lib.dfb_track_workspace_doubles(480, 640, 4) == 29 * ((120 * 160 + 255) // 256)
    for bad in ((0, 8, 1), (8, 0, 1), (8, 8, 0)):
        assert lib.dfb_track_workspace_doubles(*bad) == -1
    p = ctypes.c_void_p(8)
    d9 = (ctypes.c_double * 9)()
    d12 = (ctypes.c_double * 12)()
    d3 = (ctypes.c_double * 3)()
    f64 = _capi.c_f64p

    def vol(x0=0, x1=16, r=16, t=8, w=8):
        v = _capi.Volume()
        v.tsdf, v.weight, v.rx, v.ry, v.rz, v.x0, v.x1 = t, w, r, r, r, x0, x1
        return v
    words = lib.dfb_track_workspace_doubles(8, 8, 1)

    def call(v=None, res=16, scale=1.0, center=d3, depth=p, rows=8, cols=8, k=d9, kinv=d9, lw=d12, stride=1, tdist=1.0, delta=0.5,
             ws=p, n_ws=words, out=p):
        v = vol() if v is None else v
        cast = lambda a: ctypes.cast(a, f64) if a is not None else None
        return lib.dfb_track_normal_eq(ctypes.byref(v) if v is not False else None, res, scale, cast(center), depth, rows, cols,
                                       cast(k), cast(kinv), cast(lw), stride, tdist, delta, ws, n_ws, out, None, None)
    cases = [(dict(v=False), b"null pointer"), (dict(center=None), b"null pointer"), (dict(depth=None), b"null pointer"),
             (dict(k=None), b"null pointer"), (dict(kinv=None), b"null pointer"), (dict(lw=None), b"null pointer"),
             (dict(ws=None), b"null pointer"), (dict(out=None), b"null pointer"), (dict(v=vol(t=0)), b"null pointer"),
             (dict(v=vol(w=0)), b"null pointer"), (dict(v=vol(r=1, x1=1)), b"smaller than one cell"),
             (dict(v=vol(0, 8)), b"slab"), (dict(v=vol(8, 16)), b"slab"), (dict(res=0), b"tsdf_res"), (dict(rows=0), b"empty"),
             (dict(cols=0), b"empty"), (dict(stride=0), b"stride"), (dict(scale=0.0), b"scale"), (dict(scale=-1.0), b"scale"),
             (dict(tdist=0.0), b"truncation"), (dict(tdist=-1.0), b"truncation"), (dict(delta=0.0), b"Huber"),
             (dict(n_ws=words - 1), b"workspace")]
    for kw, msg in cases:
        assert call(**kw) == -1, kw
        assert msg in lib.dfb_last_error(), (kw, lib.dfb_last_error())
