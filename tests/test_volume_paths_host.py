"""a1 (Fusion.updateTSDF, FusionDM.updateTSDF) and a2 (FusionDM.fuseDepths) through the host build of the kernels' per-voxel
logic (tests/hostshim) against oracle/tsdf.py, at the edges tests/test_gpu_volume_paths.py takes the device to: every k = 1...8,
x-slabs that start past 0 and have ragged sizes, a live volume whose shape differs from the grid, untruncated / bench-truncated /
clipped live volumes, fresh and mid-sequence state, truncation distances float32 cannot represent, saturating weights, and an odd
`tsdf_res` (half-voxel grid centre) for a2.  When a device case fails, these tell a failure of the shared per-voxel functions
apart from one of the device-only code (kernel templates, work list, overflow bitmap, slab indexing).

Bars (as the device tests): masks bit for bit; values within 1e-5 tdist; weights within 1e-6 relative; hybrid and all-exact agree
on masks and weights bit for bit (their values may differ in the last float32 bits: the fast tier evaluates the clamped a1 update in
float32, the exact tier in float64).  Voxels whose k nearest nodes tie are excluded from the oracle comparison (the order of tied
neighbours is implementation-defined) and must be rare."""
import numpy as np
import pytest

import hostshim_api as hs
import scenes
from dynamicfusion_body_b200 import synth
from oracle import tsdf as ot

TSDF_TOL = 1e-5
W_RTOL = 1e-6
R = 24
TD = 2.0                     # truncation distance of the truncated live forms, in voxels (the benchmark's 256^3 scene: 5)
LWS = {"none": None, "f32_q5": np.array([1, 0, 0, 0, 0, 0.01, 0.01, 0], np.float32), "f64": np.array([1, 0, 0, 0, 0, 0.1, 0, 0.05])}


@pytest.fixture(scope="module")
def scene():
    sc = synth.make_scene(res=R, k=8, n_nodes=60, seed=11, rows=48, cols=64)
    wv = synth.blend_warp(sc.vertices, sc.node_pos, sc.node_dq, np.full(sc.n_nodes, sc.node_w), sc.vert_knn, lw=None)
    sdf = synth.mesh_sdf_volume((R + 2, R, R + 1), wv, sc.normals)          # live grid shape != canonical grid shape
    return sc, sdf


def live_form(sdf, form, td=TD):
    """(live volume, tdist).  'untruncated': the reference's own call, tdist = volume.max() (test.py:110); 'bench': the live volume
    as FusionDM / fuseFrame leave it, the expression bench.py times (band, +tdist elsewhere); 'clipped': clipped to [-1.5 tdist, tdist]
    (corners exactly +tdist: the fast tier's `mn >= tdist` equality case; -tdist itself is the documented irreproducible knife edge)."""
    if form == "untruncated":
        return sdf, float(sdf.max())
    if form == "bench":
        return np.where(sdf < -td, np.float32(td), np.minimum(sdf, np.float32(td))).astype(np.float32), td
    return np.clip(sdf, -1.5 * td, td).astype(np.float32), td


def run_a1(sc, live, tdist, k, lw, t0, w0, res=(R, R, R), x0=0, x1=None, wmax=100.0):
    """Host hybrid and all-exact against the oracle on the slab [x0, x1); returns (oracle mask, voxels the fast tier deferred,
    hybrid values, hybrid weights)."""
    x1 = res[0] if x1 is None else x1
    vox, idx, tie = scenes.oracle_knn(res, sc.node_pos, k, x0, x1)
    assert tie.mean() < 0.01
    nw = np.full(sc.n_nodes, sc.node_w)
    if k == 0:
        ov, ow, om = ot.update_rigid_volume(t0.astype(np.float64), w0.astype(np.float64), live, vox, lw, tdist, wmax=wmax)
        wf = hs.HostWarpField(np.zeros((0, 3)), np.zeros((0, 8)), np.zeros(0), 0, lw=lw)
        tie[:] = False
    else:
        ov, ow, om = ot.update_volume(t0.astype(np.float64), w0.astype(np.float64), live, vox, idx, sc.node_pos, sc.node_dq, nw, lw,
                                      tdist, wmax=wmax)
        wf = hs.HostWarpField(sc.node_pos, sc.node_dq, np.float32(sc.node_w), k, knn=idx, lw=lw)
    out = []
    for mode in (0, 1):
        tv, tw = t0.copy(), w0.copy()
        mask, cls, nunc = hs.update_volume(tv, tw, res, wf, live, tdist, wmax=wmax, mode=mode, x0=x0, x1=x1)
        ok = ~tie
        assert np.array_equal(mask.astype(bool)[ok], om[ok])
        assert np.abs(tv - ov)[ok].max() <= TSDF_TOL * abs(tdist)
        assert (np.abs(tw - ow) / np.maximum(1, ow))[ok].max() <= W_RTOL
        out.append((tv, tw, mask, nunc))
    assert np.array_equal(out[0][2], out[1][2]) and np.array_equal(out[0][1], out[1][1])
    return om, out[0][3], out[0][0], out[0][1]


@pytest.mark.parametrize("form", ["untruncated", "bench", "clipped"])
@pytest.mark.parametrize("k", range(1, 9))
def test_a1_every_k(scene, k, form):
    sc, sdf = scene
    live, td = live_form(sdf, form)
    for fresh in (True, False):
        t0, w0 = scenes.initial_state(R ** 3, seed=k, fresh=fresh, tdist=td)
        for lw in LWS.values():
            om, nunc = run_a1(sc, live, td, k, lw, t0, w0)[:2]
            assert 0 < om.sum() < om.size
            if form != "untruncated":
                assert nunc < 0.8 * R ** 3          # the fast tier settled part of the volume (CLAMP / SKIP)


@pytest.mark.parametrize("k", [3, 4, 8])
def test_a1_slabs(scene, k):
    """x0 > 0, ragged slab sizes, a live grid of another shape: each slab against the oracle, and the slabs concatenate to the
    full-volume result bit for bit (the fp32 error scale `coord_mag` is taken from the full grid, so a voxel's tier does not
    depend on the slab it is updated in)."""
    sc, sdf = scene
    res = (R, R - 3, R + 5)
    for form in ("untruncated", "bench"):
        live, td = live_form(sdf, form)
        t0, w0 = scenes.initial_state(int(np.prod(res)), seed=5, tdist=td)
        t3, w3 = t0.reshape(res), w0.reshape(res)
        parts = []
        for x0, x1 in ((0, 5), (5, 19), (19, R)):
            parts.append(run_a1(sc, live, td, k, LWS["f64"], t3[x0:x1].ravel(), w3[x0:x1].ravel(), res=res, x0=x0, x1=x1)[2:])
        _, _, tf, wfull = run_a1(sc, live, td, k, LWS["f64"], t0, w0, res=res)
        assert np.array_equal(np.concatenate([p[0] for p in parts]), tf)
        assert np.array_equal(np.concatenate([p[1] for p in parts]), wfull)


def test_a1_rigid_on_a_slab(scene):
    """FusionDM.updateTSDF (k = 0, core/fusion_dm.py:300-316) on a slab that starts past 0, fresh and mid-sequence."""
    sc, sdf = scene
    live, td = live_form(sdf, "bench")
    for fresh in (True, False):
        t0, w0 = scenes.initial_state((R - 7) * R * R, seed=2, fresh=fresh, tdist=td)
        om = run_a1(sc, live, td, 0, LWS["f32_q5"], t0, np.floor(w0), x0=7, x1=R)[0]
        assert 0 < om.sum() < om.size


@pytest.mark.parametrize("td", [2.0 / 3.0, 0.7, 1.1])
def test_a1_unrepresentable_tdist_and_saturating_weights(scene, td):
    """tdist not representable in float32 (rounded up: 2/3, 1.1; rounded down: 0.7), so the live volume's +tdist is float32(tdist),
    not tdist, and the exact tier's `tl < tdist` sees a value an ulp away from the fast tier's threshold; wmax = 7.3 (not a float32
    either) saturates most of the mid-sequence weights."""
    sc, sdf = scene
    for form in ("bench", "clipped"):
        live, _ = live_form(sdf, form, td)
        for k in (1, 4, 8):
            t0, w0 = scenes.initial_state(R ** 3, seed=7, tdist=td)
            for wmax in (100.0, 7.3):
                om = run_a1(sc, live, td, k, LWS["none"], t0, w0, wmax=wmax)[0]
                assert 0 < om.sum() < om.size


def _rigid_setup(R_, tdist):
    sc = synth.make_scene(res=R_, k=4, n_nodes=100, seed=1, rows=48, cols=64)
    K = np.array([[200., 0, 80], [0, 200, 60], [0, 0, 1]])
    ang = 0.1
    Rm = np.array([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]])
    scale = 12 * 1.3 / R_
    center = np.array([-0.03, -0.43, -5.6])
    lw34 = np.concatenate([Rm, -Rm @ center[:, None] + np.array([[0.1], [0.05], [22.0]])], 1)
    vw = scale * (sc.vertices.astype(np.float64) - R_ / 2) + center
    dm = synth.render_depth(vw @ lw34[:, :3].T + lw34[:, 3], sc.faces, K, 120, 160)
    return dict(dm=dm, lw34=lw34, K=K, Kinv=np.linalg.inv(K), scale=scale, center=center, tdist=tdist)


@pytest.mark.parametrize("R_", [24, 25])
def test_a2_slabs_and_odd_res(R_):
    """FusionDM.fuseDepths on slabs [0,7) / [7,16) / [16,R) of an even and an odd tsdf_res (grid centre on a voxel or half-way
    between two): each slab against the oracle, with and without the brick classifier, hybrid and all-exact; the slabs
    concatenate to the full volume bit for bit, values included (both tiers evaluate a clamped update with one expression)."""
    s = _rigid_setup(R_, 0.2)
    res = (R_, R_, R_)
    t0, w0 = scenes.initial_state(R_ ** 3, tdist=s["tdist"])
    t3, w3 = t0.reshape(res), w0.reshape(res)
    full = None
    for slabs in (((0, R_),), ((0, 7), (7, 16), (16, R_))):
        outs = {}
        for mode, bricks in ((0, False), (0, True), (1, False)):
            parts = []
            for x0, x1 in slabs:
                vox = ot.voxel_grid(res, x0, x1)
                tv, tw = t3[x0:x1].ravel().copy(), w3[x0:x1].ravel().copy()
                ov, ow, om, ofr = ot.fuse_depth_rigid(tv.astype(np.float64), tw.astype(np.float64), vox, s["dm"], s["lw34"], s["K"],
                                                      s["Kinv"], s["tdist"], R_, scale=s["scale"], center=s["center"])
                hs.set_bricks(slab_shape=(x1 - x0, R_, R_), enable=bricks)
                try:
                    mask, frus, cls, nunc = hs.fuse_depth_rigid(tv, tw, res, R_, s["dm"], s["lw34"], s["K"], s["Kinv"], s["scale"], s["center"],
                                                                s["tdist"], mode=mode, x0=x0, x1=x1)
                finally:
                    hs.set_bricks(enable=False)
                assert np.array_equal(mask.astype(bool), om) and np.array_equal(frus.astype(bool), ofr)
                assert np.abs(tv - ov).max() <= TSDF_TOL * s["tdist"]
                assert np.array_equal(tw, ow.astype(np.float32))
                parts.append((tv, tw, mask, frus))
            outs[(mode, bricks)] = [np.concatenate([p[i] for p in parts]) for i in range(4)]
        ref = outs[(0, False)]
        for o in outs.values():
            for a, b in zip(o, ref):
                assert np.array_equal(a, b)
        if full is None:
            full = ref
            assert 0.01 < ref[2].mean() < 0.99
        else:
            for a, b in zip(ref, full):
                assert np.array_equal(a, b)
