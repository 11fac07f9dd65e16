"""Device parity of the two volume-driven TSDF entry points at the shapes the benchmark times (run with -m gpu on the B200 box).

a1, Fusion.updateTSDF -> dfb_tsdf_update_volume: vol_fast_kernel<4|8> classifies, vol_exact_kernel<KMAX, KT> takes the deferred voxels
from the work list, then from the overflow bitmap (or, without a bitmap, by re-classifying the volume).  KT = k for k = 4 and 8, KT = 0
(run-time k) otherwise -- every instantiation is reached below.  a2, FusionDM.fuseDepths -> dfb_fuse_depth_rigid: the rigid branch of
the projective pass, with and without brick culling.

Each case is held to the float64 oracle (oracle/tsdf.py) and to the device-only properties the oracle cannot see:
* masks, weights and slab decompositions and list capacities: bit for bit;
* a1 hybrid vs all-exact values: to rounding (the fast tier evaluates the clamped update in float32, the exact tier in float64; the
  largest ulp gap is printed); a2 hybrid vs all-exact values: bit for bit (one clamped-update expression for both tiers);
* the overflow bitmap is all zero after every call and every deferred voxel is processed exactly once.

Bars against the oracle (north_star): masks bit for bit; |dTSDF| <= 1e-5 tdist; weights within 1e-6 relative.  Voxels whose k nearest
nodes tie are excluded from the comparison with the oracle's own kNN."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TSDF_TOL = 1e-5
W_RTOL = 1e-6
HYB_TOL = 1e-6       # a1 hybrid vs all-exact values, fraction of tdist
TD = 2.0             # truncation distance of the truncated live forms at small sizes, in voxels
SMALL_LIST = 1024


def _ctx():
    import torch
    from dynamicfusion_body_b200 import engine, _capi
    assert torch.cuda.is_available()
    return torch, engine, _capi


def _np(t):
    return t.cpu().numpy().ravel()


def ulp_gap(a, b):
    """Largest distance in float32 units in the last place between two float32 arrays (signed zeros count as equal)."""
    def ordered(x):
        i = np.asarray(x, np.float32).view(np.int32).astype(np.int64)
        return np.where(i < 0, -(i & 0x7fffffff), i)
    return int(np.abs(ordered(a) - ordered(b)).max()) if np.size(a) else 0


def live_form(sdf, form, td=TD):
    """(live volume, tdist): 'untruncated' = the reference's call (test.py:110, tdist = volume.max()); 'bench' = bench.py's
    c2_a1_256_truncated input: the band around the surface and +tdist everywhere else (as FusionDM / fuseFrame leave a volume)."""
    if form == "untruncated":
        return sdf, float(sdf.max())
    return np.where(sdf < -td, np.float32(td), np.minimum(sdf, np.float32(td))).astype(np.float32), td


def a1_call(engine, _capi, vol, wf, lw, live, td, mode=0, capacity=None, bitmap=True, want_masks=True):
    """One dfb_tsdf_update_volume call through the C ABI with the workspace struct built here: `capacity` shortens the work list the
    call sees, `bitmap=False` passes overflow_bits = NULL (the exact pass then re-classifies the volume)."""
    import torch
    knn = wf.knn_table(vol.res, vol.x0, vol.x1)
    ws = vol.workspace.struct(False)
    if capacity is not None:
        ws.capacity = capacity
    if not bitmap:
        ws.overflow_bits = None
    mask = torch.zeros(vol.n_voxels, dtype=torch.uint8, device=vol.device) if want_masks else None
    v = vol.struct()
    s = wf.struct(lw, knn)
    _capi.check(_capi.lib().dfb_tsdf_update_volume(C.byref(v), C.byref(s), engine._ptr(live), live.shape[0], live.shape[1], live.shape[2],
                                                   float(td), 100.0, int(mode), C.byref(ws), engine._ptr(mask), engine._stream()))
    torch.cuda.synchronize()
    return mask


def check_oracle_a1(om_ov_ow, mask, tsdf, weight, ok, td):
    om, ov, ow = om_ov_ow
    assert np.array_equal(mask.astype(bool)[ok], om[ok])
    assert np.abs(tsdf - ov)[ok].max() <= TSDF_TOL * td
    assert (np.abs(weight - ow) / np.maximum(1, ow))[ok].max() <= W_RTOL


def check_hybrid_exact_a1(hyb, exa, td, what):
    """hyb / exa = (tsdf, weight, mask): masks and weights bit for bit, values to rounding."""
    assert np.array_equal(hyb[2], exa[2]) and np.array_equal(hyb[1], exa[1])
    gap = ulp_gap(hyb[0], exa[0])
    dv = np.abs(hyb[0].astype(np.float64) - exa[0]).max()
    print("%s: hybrid vs exact values: largest gap %d ulp, %.3g tdist" % (what, gap, dv / td))
    assert dv <= HYB_TOL * td


def _small_a1_scene(k, R, seed):
    from dynamicfusion_body_b200 import synth
    sc = synth.make_scene(res=R, k=k, n_nodes=120, seed=seed, rows=48, cols=64)
    wv = synth.blend_warp(sc.vertices, sc.node_pos, sc.node_dq, np.full(sc.n_nodes, sc.node_w), sc.vert_knn, lw=None)
    sdf = synth.mesh_sdf_volume((R + 2, R, R + 1), wv, sc.normals)
    return sc, sdf


# ------------------------------------------------------------------------------------------------------------------------------
# a1
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", range(1, 9))
def test_a1_every_k(k):
    """k = 1...8 reaches vol_fast_kernel<4> / <8> and vol_exact_kernel<4,0> (k 1-3), <4,4>, <8,0> (k 5-7), <8,8>; untruncated and
    bench-truncated live volumes, fresh and mid-sequence state; hybrid and all-exact against the oracle and against each other."""
    torch, engine, _capi = _ctx()
    import scenes
    from oracle import tsdf as ot
    R = 22 + 2 * k
    res = (R, R - 3, R + 5)
    n = int(np.prod(res))
    sc, sdf = _small_a1_scene(k, R, seed=k)
    vox, idx, tie = scenes.oracle_knn(res, sc.node_pos, k)
    assert tie.mean() < 0.01
    ok = ~tie
    nw = np.full(sc.n_nodes, sc.node_w)
    wf = engine.DeviceWarpField(k)
    wf.set_nodes(sc.node_pos, sc.node_dq, np.float32(sc.node_w))
    assert tuple(wf.knn_table(res, 0, R).shape) == (n, k)         # the table the kernels index with the template's k
    for form in ("untruncated", "bench"):
        live_np, td = live_form(sdf, form)
        live = torch.from_numpy(live_np).cuda()
        for fresh in (True, False):
            t0, w0 = scenes.initial_state(n, seed=k, fresh=fresh, tdist=td)
            ov, ow, om = ot.update_volume(t0.astype(np.float64), w0.astype(np.float64), live_np, vox, idx, sc.node_pos, sc.node_dq, nw,
                                          None, td)
            outs = []
            for mode in (0, 1):
                vol = engine.DeviceVolume(res, tsdf=t0, weight=w0)
                mask = a1_call(engine, _capi, vol, wf, None, live, td, mode=mode)
                st = vol.workspace.stats()
                outs.append((_np(vol.tsdf), _np(vol.weight), _np(mask)))
                check_oracle_a1((om, ov, ow), outs[-1][2], outs[-1][0], outs[-1][1], ok, td)
                assert st["exact_processed"] == (st["deferred"] if mode == 0 else int(om.size))
                assert not vol.workspace.overflow_bits.any()
                if mode == 0 and form == "bench":
                    assert st["deferred"] < 0.8 * n                      # the fast tier settled voxels (CLAMP / SKIP)
            check_hybrid_exact_a1(outs[0], outs[1], td, "k=%d %s fresh=%s" % (k, form, fresh))
            assert 0 < om.sum() < om.size


@pytest.mark.parametrize("k", [3, 4, 8])
def test_a1_slabs_equal_full_volume(k):
    """Three uneven slabs, x0 > 0, thicknesses not multiples of 32: concatenated they equal the full-volume call bit for bit,
    values included -- a voxel's tier does not depend on the slab (the fp32 error scale comes from the full grid)."""
    torch, engine, _capi = _ctx()
    import scenes
    from oracle import tsdf as ot
    R = 48
    res = (R, 40, 44)
    n = int(np.prod(res))
    sc, sdf = _small_a1_scene(k, R, seed=20 + k)
    wf = engine.DeviceWarpField(k)
    wf.set_nodes(sc.node_pos, sc.node_dq, np.float32(sc.node_w))
    vox, idx, tie = scenes.oracle_knn(res, sc.node_pos, k)
    lw = np.array([1, 0, 0, 0, 0, 0.1, 0, 0.05])
    for form in ("untruncated", "bench"):
        live_np, td = live_form(sdf, form)
        live = torch.from_numpy(live_np).cuda()
        t0, w0 = scenes.initial_state(n, seed=3, tdist=td)
        full = engine.DeviceVolume(res, tsdf=t0, weight=w0)
        fm = _np(a1_call(engine, _capi, full, wf, lw, live, td))
        ov, ow, om = ot.update_volume(t0.astype(np.float64), w0.astype(np.float64), live_np, vox, idx, sc.node_pos, sc.node_dq,
                                      np.full(sc.n_nodes, sc.node_w), lw, td)
        check_oracle_a1((om, ov, ow), fm, _np(full.tsdf), _np(full.weight), ~tie, td)
        t3, w3 = t0.reshape(res), w0.reshape(res)
        parts = []
        for x0, x1 in ((0, 11), (11, 45), (45, R)):
            s = engine.DeviceVolume(res, x0, x1, tsdf=t3[x0:x1], weight=w3[x0:x1])
            m = a1_call(engine, _capi, s, wf, lw, live, td)
            assert not s.workspace.overflow_bits.any()
            parts.append((_np(s.tsdf), _np(s.weight), _np(m)))
        for i, ref in enumerate((_np(full.tsdf), _np(full.weight), fm)):
            assert np.array_equal(np.concatenate([p[i] for p in parts]), ref)


@pytest.mark.parametrize("k", [3, 4, 8])
def test_a1_overflow_paths(k):
    """The same frame through the default list, a 1024-entry list (the overflow bitmap is swept after the list) and a 1024-entry list
    without a bitmap (the exact pass re-classifies the volume): masks, values and weights bit-equal across the three, every deferred
    voxel processed once, the bitmap all zero after every call."""
    torch, engine, _capi = _ctx()
    import scenes
    from oracle import tsdf as ot
    R = 40
    res = (R, R, R)
    sc, sdf = _small_a1_scene(k, R, seed=30 + k)
    wf = engine.DeviceWarpField(k)
    wf.set_nodes(sc.node_pos, sc.node_dq, np.float32(sc.node_w))
    vox, idx, tie = scenes.oracle_knn(res, sc.node_pos, k)
    for form in ("untruncated", "bench"):
        live_np, td = live_form(sdf, form)
        live = torch.from_numpy(live_np).cuda()
        t0, w0 = scenes.initial_state(R ** 3, seed=4, tdist=td)
        ov, ow, om = ot.update_volume(t0.astype(np.float64), w0.astype(np.float64), live_np, vox, idx, sc.node_pos, sc.node_dq,
                                      np.full(sc.n_nodes, sc.node_w), None, td)
        outs = []
        for capacity, bitmap in ((None, True), (SMALL_LIST, True), (SMALL_LIST, False)):
            vol = engine.DeviceVolume(res, tsdf=t0, weight=w0)
            m = a1_call(engine, _capi, vol, wf, None, live, td, capacity=capacity, bitmap=bitmap)
            st = vol.workspace.stats()
            print("k=%d %s capacity=%s bitmap=%s" % (k, form, capacity, bitmap), st)
            assert st["exact_processed"] == st["deferred"]
            if capacity is not None:
                assert st["deferred"] > capacity                          # the sweep / the re-scan did run
            assert not vol.workspace.overflow_bits.any()
            outs.append((_np(vol.tsdf), _np(vol.weight), _np(m)))
        check_oracle_a1((om, ov, ow), outs[0][2], outs[0][0], outs[0][1], ~tie, td)
        for o in outs[1:]:
            for a, b in zip(o, outs[0]):
                assert np.array_equal(a, b)


def test_a1_sequence_with_overflowing_list():
    """Five a1 frames on one volume with a 1024-entry list (every frame overflows into the bitmap), alternating two live volumes, then
    an a3 frame (update_projective) and one more a1 frame, against the oracle carried through the same frames in float32 storage.
    A bitmap bit that survived a call would update its voxel twice in the next frame: its weight would then be off by a whole wi."""
    torch, engine, _capi = _ctx()
    import scenes
    from dynamicfusion_body_b200 import synth
    from oracle import tsdf as ot
    R = 40
    res = (R, R, R)
    sc = synth.make_scene(res=R, k=4, n_nodes=150, seed=8, rows=96, cols=128)
    nw = np.full(sc.n_nodes, sc.node_w)
    wv = synth.blend_warp(sc.vertices, sc.node_pos, sc.node_dq, nw, sc.vert_knn, lw=None)
    lives = []
    for shift in (0.0, 1.3):
        sdf = synth.mesh_sdf_volume((R + 2, R, R + 1), wv + shift, sc.normals)
        lives.append(live_form(sdf, "bench")[0])
    td = TD
    vox, idx, tie = scenes.oracle_knn(res, sc.node_pos, 4)
    ok = ~tie
    wf = engine.DeviceWarpField(4)
    wf.set_nodes(sc.node_pos, sc.node_dq, np.float32(sc.node_w))
    t0, w0 = scenes.initial_state(R ** 3, fresh=True, tdist=td)
    vol = engine.DeviceVolume(res, tsdf=t0, weight=w0)
    vol.workspace.capacity = SMALL_LIST
    ov, ow = t0.astype(np.float64), w0.astype(np.float64)
    depths = torch.from_numpy(sc.depths).cuda()
    frames = ["a1"] * 5 + ["a3", "a1"]
    for f, kind in enumerate(frames):
        if kind == "a1":
            live_np = lives[f % 2]
            m = _np(engine.update_volume(vol, wf, None, torch.from_numpy(live_np).cuda(), td, want_masks=True)).astype(bool)
            ov, ow, om = ot.update_volume(ov, ow, live_np, vox, idx, sc.node_pos, sc.node_dq, nw, None, td)
            st = vol.workspace.stats()
            assert st["exact_processed"] == st["deferred"] > SMALL_LIST, st
        else:
            mm, _ = engine.update_projective(vol, wf, sc.lw, depths, sc.K, sc.Kinv, None, td, want_masks=True)
            m = (_np(mm) & 1).astype(bool)
            ov, ow, oms, _ = ot.update_projective(ov, ow, vox, idx, sc.node_pos, sc.node_dq, nw, sc.lw, sc.depths, sc.K, sc.Kinv, td)
            om = oms[0]
        torch.cuda.synchronize()
        assert not vol.workspace.overflow_bits.any()
        ov, ow = ov.astype(np.float32).astype(np.float64), ow.astype(np.float32).astype(np.float64)   # the volume stores float32
        assert np.array_equal(m[ok], om[ok]), "frame %d (%s)" % (f, kind)
        assert np.abs(_np(vol.tsdf) - ov)[ok].max() <= TSDF_TOL * td, "frame %d (%s)" % (f, kind)
        assert (np.abs(_np(vol.weight) - ow) / np.maximum(1, ow))[ok].max() <= W_RTOL, "frame %d (%s)" % (f, kind)
        assert 0 < om.sum() < om.size


@pytest.fixture(scope="module")
def bench_scene_256():
    """The scene and live volumes bench.py's c2_a1_256_* entries time (bench.py:646, 680-688)."""
    import time
    from dynamicfusion_body_b200 import synth
    t = time.time()
    sc = synth.make_scene(res=256, n_nodes=1000, seed=0, background=True)
    wv = synth.blend_warp(sc.vertices, sc.node_pos, sc.node_dq, np.full(sc.n_nodes, np.float32(sc.node_w)), sc.vert_knn, lw=None)
    sdf = synth.mesh_sdf_volume((256, 256, 256), wv, sc.normals)
    trunc = np.where(sdf < -sc.tdist, np.float32(sc.tdist), np.minimum(sdf, np.float32(sc.tdist))).astype(np.float32)
    print("256^3 scene + live SDF: %.1f s" % (time.time() - t))
    return sc, {"reference_usage": (sdf, float(sdf.max())), "truncated": (trunc, sc.tdist)}


@pytest.mark.parametrize("k", [4, 8])
def test_a1_256_as_benchmarked(bench_scene_256, k):
    """a1 at 256^3 as bench.py runs it (fresh volume fill = tdist, w = 0, no lw), untruncated (every voxel in the band, three
    quarters of them through the overflow bitmap) and truncated (89 % of the voxels exactly +tdist: the fast tier's `mn >= tdist`
    equality case); k = 8 reaches the device-only KT = 8 exact kernel.  hybrid == exact on masks and weights, two slabs == full,
    and the oracle on three 200 k-voxel samples: uniform, voxels the fast tier deferred, voxels it settled as CLAMP."""
    import time
    torch, engine, _capi = _ctx()
    from oracle import dq as odq
    from oracle import tsdf as ot
    sc, lives = bench_scene_256
    R = 256
    res = (R, R, R)
    n = R ** 3
    rng = np.random.default_rng(k)
    wf = engine.DeviceWarpField(k)
    wf.set_nodes(sc.node_pos, sc.node_dq, np.float32(sc.node_w))
    knn = wf.knn_table(res, 0, R).cpu().numpy().view(np.uint16).astype(np.int64)
    uni = np.sort(rng.choice(n, 200_000, replace=False))
    vox_u = np.stack(np.unravel_index(uni, res), 1).astype(np.float32)
    # the device's kNN table against the brute-force oracle on the uniform sample (ties excluded); the a1 comparisons below
    # then feed the oracle the device's own table, so no voxel needs to be excluded from them
    bidx, d2 = odq.knn_bruteforce(vox_u, sc.node_pos, k)
    tie = odq.knn_has_tie(d2)
    assert tie.mean() < 0.01 and np.array_equal(knn[uni][~tie], bidx[~tie])
    for name, (live_np, td) in lives.items():
        live = torch.from_numpy(live_np).cuda()
        t = time.time()
        vol = engine.DeviceVolume(res, fill=td)
        mask = _np(a1_call(engine, _capi, vol, wf, None, live, td))
        st = vol.workspace.stats()
        cap = vol.workspace.capacity
        deferred_list = vol.workspace.list[:min(st["deferred"], cap)].cpu().numpy().astype(np.int64)
        assert st["exact_processed"] == st["deferred"] and not vol.workspace.overflow_bits.any()
        hyb = (_np(vol.tsdf), _np(vol.weight), mask)
        del vol
        ex = engine.DeviceVolume(res, fill=td)
        em = _np(a1_call(engine, _capi, ex, wf, None, live, td, mode=1))
        check_hybrid_exact_a1(hyb, (_np(ex.tsdf), _np(ex.weight), em), td, "256^3 k=%d %s" % (k, name))
        del ex
        # what the fast tier settled as CLAMP: the fast pass alone writes mask 1 exactly there (deferred voxels keep 0)
        fo = engine.DeviceVolume(res, fill=td)
        clamp = np.flatnonzero(_np(a1_call(engine, _capi, fo, wf, None, live, td, mode=_capi.MODE_FAST_ONLY)))
        del fo
        print("256^3 k=%d %s: deferred %d (list %d), CLAMP %d, updated %d" % (k, name, st["deferred"], cap, len(clamp), int(mask.sum())))
        if name == "reference_usage":
            assert st["deferred"] > cap                                  # the bitmap sweep ran
        else:
            assert len(clamp) > n // 2                                   # the equality case settled most of the volume
        # two slabs == full volume
        for x0, x1 in ((0, 100), (100, R)):
            s = engine.DeviceVolume(res, x0, x1, fill=td)
            m = _np(a1_call(engine, _capi, s, wf, None, live, td))
            lo, hi = x0 * R * R, x1 * R * R
            assert np.array_equal(_np(s.tsdf), hyb[0][lo:hi]) and np.array_equal(_np(s.weight), hyb[1][lo:hi])
            assert np.array_equal(m, hyb[2][lo:hi])
            assert not s.workspace.overflow_bits.any()
            del s
        # the oracle on three samples
        samples = {"uniform": uni, "deferred": deferred_list, "clamp": clamp}
        for sname, sel in samples.items():
            if len(sel) > 200_000:
                sel = np.sort(rng.choice(sel, 200_000, replace=False))
            if sname != "clamp" or name == "truncated":
                assert len(sel) > 1000, sname
            if len(sel) == 0:
                continue
            vox = np.stack(np.unravel_index(sel, res), 1).astype(np.float32)
            ov, ow, om = ot.update_volume(np.full(len(sel), td, np.float64), np.zeros(len(sel)), live_np, vox, knn[sel], sc.node_pos,
                                          sc.node_dq, np.full(sc.n_nodes, np.float32(sc.node_w)), None, td)
            ok = np.ones(len(sel), bool)
            check_oracle_a1((om, ov, ow), hyb[2][sel], hyb[0][sel], hyb[1][sel], ok, td)
            if sname == "clamp":
                assert om.all()
        del live
        torch.cuda.empty_cache()
        print("256^3 k=%d %s: %.1f s" % (k, name, time.time() - t))


# ------------------------------------------------------------------------------------------------------------------------------
# a2
# ------------------------------------------------------------------------------------------------------------------------------
def _rigid_setup(R, tdist=0.2):
    """The a2 frame of test_fuse_depth_rigid_a2 at grid size R (tsdf_res = R)."""
    from dynamicfusion_body_b200 import synth
    sc = synth.make_scene(res=min(R, 96), k=4, n_nodes=100, seed=1, rows=48, cols=64)
    verts = sc.vertices.astype(np.float64) * ((R - 1) / (min(R, 96) - 1))
    K = np.array([[200., 0, 80], [0, 200, 60], [0, 0, 1]])
    ang = 0.1
    Rm = np.array([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]])
    scale = 12 * 1.3 / R
    center = np.array([-0.03, -0.43, -5.6])
    lw34 = np.concatenate([Rm, -Rm @ center[:, None] + np.array([[0.1], [0.05], [22.0]])], 1)
    vw = scale * (verts - R / 2) + center
    dm = synth.render_depth(vw @ lw34[:, :3].T + lw34[:, 3], sc.faces, K, 120, 160)
    return dict(dm=dm, lw34=lw34, K=K, Kinv=np.linalg.inv(K), scale=scale, center=center, tdist=tdist)


def a2_run(torch, engine, s, R, t0, w0, x0=0, x1=None, mode=0, use_bricks=True, capacity=None):
    res = (R, R, R)
    x1 = R if x1 is None else x1
    t3, w3 = t0.reshape(res), w0.reshape(res)
    vol = engine.DeviceVolume(res, x0, x1, tsdf=t3[x0:x1], weight=w3[x0:x1])
    if capacity:
        vol.workspace.capacity = capacity
    m, f = engine.fuse_depth_rigid(vol, R, torch.from_numpy(s["dm"]).cuda(), s["lw34"], s["K"], s["Kinv"], s["scale"], s["center"],
                                   s["tdist"], mode=mode, want_masks=True, use_bricks=use_bricks)
    torch.cuda.synchronize()
    st = vol.workspace.stats()
    assert st["exact_processed"] == (st["deferred"] if mode == 0 else vol.n_voxels)
    assert not vol.workspace.overflow_bits.any()
    return (_np(vol.tsdf), _np(vol.weight), _np(m), _np(f)), st


@pytest.mark.parametrize("R", [64, 81, 96])
def test_a2_paths(R):
    """FusionDM.fuseDepths at 64^3 / 81^3 (odd tsdf_res: the grid centre falls between voxels) / 96^3: bricks on == bricks off
    (proj_fast_kernel rigid) == all-exact == a 1024-entry list == uneven slabs, bit for bit (masks, frusta, values, weights),
    and the oracle for the full volume."""
    torch, engine, _ = _ctx()
    import scenes
    from oracle import tsdf as ot
    s = _rigid_setup(R)
    res = (R, R, R)
    t0, w0 = scenes.initial_state(R ** 3, tdist=s["tdist"])
    ov, ow, om, ofr = ot.fuse_depth_rigid(t0.astype(np.float64), w0.astype(np.float64), ot.voxel_grid(res), s["dm"], s["lw34"], s["K"],
                                          s["Kinv"], s["tdist"], R, scale=s["scale"], center=s["center"])
    assert 0.02 < om.mean() < 0.98
    ref, st = a2_run(torch, engine, s, R, t0, w0)
    print("a2 %d^3 bricks on:" % R, st)
    assert st["bricks_streamed"] + st["bricks_mixed"] > 0 and st["bricks_mixed"] < st["bricks"]
    assert np.array_equal(ref[2].astype(bool), om) and np.array_equal(ref[3].astype(bool), ofr)
    assert np.abs(ref[0] - ov).max() <= TSDF_TOL * s["tdist"]
    assert np.array_equal(ref[1], ow.astype(np.float32))
    off, st_off = a2_run(torch, engine, s, R, t0, w0, use_bricks=False)
    assert st_off["bricks_streamed"] == 0 and st_off["bricks_mixed"] == 0
    exa, _ = a2_run(torch, engine, s, R, t0, w0, mode=1)
    small, st_small = a2_run(torch, engine, s, R, t0, w0, capacity=SMALL_LIST)
    assert st_small["deferred"] > SMALL_LIST
    small_off, st_small_off = a2_run(torch, engine, s, R, t0, w0, use_bricks=False, capacity=SMALL_LIST)
    assert st_small_off["deferred"] > SMALL_LIST
    cut = (0, R // 3 + 1, R // 3 + 30, R)
    parts = [a2_run(torch, engine, s, R, t0, w0, x0=cut[i], x1=cut[i + 1])[0] for i in range(3)]
    slabs = tuple(np.concatenate([p[i] for p in parts]) for i in range(4))
    for what, o in (("bricks off", off), ("all-exact", exa), ("1024 list", small), ("1024 list, bricks off", small_off), ("slabs", slabs)):
        for a, b, field in zip(o, ref, ("tsdf", "weight", "mask", "frustum")):
            assert np.array_equal(a, b), "%s: %s" % (what, field)


def test_a2_256_slab_pair():
    """a2 at 256^3: two slabs == the full volume bit for bit, and the oracle on a 200 k-voxel sample."""
    torch, engine, _ = _ctx()
    from oracle import tsdf as ot
    R = 256
    res = (R, R, R)
    s = _rigid_setup(R)
    t0 = np.full(R ** 3, s["tdist"], np.float32)
    w0 = np.zeros(R ** 3, np.float32)
    full, st = a2_run(torch, engine, s, R, t0, w0)
    assert st["bricks_streamed"] + st["bricks_mixed"] > 0
    parts = [a2_run(torch, engine, s, R, t0, w0, x0=a, x1=b)[0] for a, b in ((0, 100), (100, R))]
    for i in range(4):
        assert np.array_equal(np.concatenate([p[i] for p in parts]), full[i])
    rng = np.random.default_rng(0)
    upd = np.flatnonzero(full[2])
    sel = np.unique(np.concatenate([rng.choice(R ** 3, 150_000, replace=False), rng.choice(upd, min(50_000, len(upd)), replace=False)]))
    vox = np.stack(np.unravel_index(sel, res), 1).astype(np.float32)
    ov, ow, om, ofr = ot.fuse_depth_rigid(t0[sel].astype(np.float64), w0[sel].astype(np.float64), vox, s["dm"], s["lw34"], s["K"], s["Kinv"],
                                          s["tdist"], R, scale=s["scale"], center=s["center"])
    assert om.sum() > 10_000
    assert np.array_equal(full[2][sel].astype(bool), om) and np.array_equal(full[3][sel].astype(bool), ofr)
    assert np.abs(full[0][sel] - ov).max() <= TSDF_TOL * s["tdist"]
    assert np.array_equal(full[1][sel], ow.astype(np.float32))
