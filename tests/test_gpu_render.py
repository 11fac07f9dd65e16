"""Z-buffer rasteriser on the device (run with -m gpu): dfb_render against oracle/render.py bit for bit on a production-size
mesh and on large faces, multi-view calls against single views, the geometry of the depth map, and Fusion.render_live after
fusing a scene."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _fusion(sc, **kw):
    """A Fusion object holding the scene's canonical model and nodes (normals turned outward, as marching cubes gives them),
    `_lw` = the scene's camera."""
    from dynamicfusion_body_b200.fusion import Fusion
    fus = Fusion(sc.tdist, knn=sc.k, use_cnn=False, write_warpfield=False, **kw)
    R = sc.res
    fus.InitializeCanonicalSpace(tsdf_shape=(R, R, R), K=sc.K, vertices=sc.vertices, normals=-sc.normals, faces=sc.faces,
                                 nodes=sc.nodes_as_reference_tuples(), radius=sc.radius)
    fus._lw = sc.lw
    return fus


def _assert_bits(dev, ora):
    d, f, n = (t.cpu().numpy() for t in dev)
    assert np.array_equal(d.view(np.uint32), ora[0].view(np.uint32))
    assert np.array_equal(f, ora[1])
    assert np.array_equal(n.view(np.uint32), ora[2].view(np.uint32))


@pytest.fixture(scope="module")
def fused_256():
    """Surface of a 256^3 volume fused from the 8 ring views of the body scene, warped to the live frame by the scene's field."""
    import torch
    from dynamicfusion_body_b200 import engine, synth
    sc = synth.make_scene(res=256, k=4, n_nodes=1000, seed=0, n_views=8)
    fus = _fusion(sc)
    fus.fuseFrame(sc.depths, extrinsics=sc.extrinsics)
    v, f, _, _ = engine.marching_cubes(fus._vol.tsdf, 1, keep_on_device=True)
    live = engine.warp_points(fus._wf, fus._lw, v, idx=fus._wf.knn_points(v, sc.k), k=sc.k)
    torch.cuda.synchronize()
    return sc, live, f


def _ring_views(sc, extrinsics):
    from dynamicfusion_body_b200 import engine
    return engine.camera_views(sc.K, sc.rows, sc.cols, extrinsics)


def test_production_mesh_8_views_equals_oracle(fused_256):
    from dynamicfusion_body_b200 import engine
    from oracle import render as orr
    sc, live, f = fused_256
    assert f.shape[0] >= 100_000
    dev = engine.render(live, f, _ring_views(sc, sc.extrinsics))
    ora = orr.render(live.cpu().numpy(), f.cpu().numpy(), sc.K, sc.rows, sc.cols, sc.extrinsics)
    _assert_bits(dev, ora)
    assert all((ora[1][v] >= 0).mean() > 0.05 for v in range(8))


def test_production_mesh_1_view_equals_oracle_and_geometry(fused_256):
    """One view without extrinsics (the points moved into the first camera's frame on the host); every covered pixel's depth
    is the intersection of its ray with its face's plane, to float32 rounding."""
    from dynamicfusion_body_b200 import engine
    from oracle import render as orr
    sc, live, f = fused_256
    E = sc.extrinsics[0]
    P = live.cpu().numpy() @ E[:, :3].T + E[:, 3]
    F = f.cpu().numpy()
    dev = engine.render(P, F, engine.camera_views(sc.K, sc.rows, sc.cols))
    ora = orr.render(P, F, sc.K, sc.rows, sc.cols)
    _assert_bits(dev, ora)
    d, face = ora[0][0], ora[1][0]
    r, c = np.nonzero(face >= 0)
    assert len(r) > 0.05 * sc.rows * sc.cols
    tri = F[face[r, c]].astype(np.int64)
    a, b, cc = P[tri[:, 0]], P[tri[:, 1]], P[tri[:, 2]]
    n = np.cross(b - a, cc - a)
    ray = np.stack([(c - sc.K[0, 2]) / sc.K[0, 0], (r - sc.K[1, 2]) / sc.K[1, 1], np.ones(len(r))], 1)
    z = (n * a).sum(1) / (n * ray).sum(1)
    zf = -d[r, c].astype(np.float64)
    assert np.all(np.abs(zf - z) <= 0.5 * np.spacing(np.float32(zf)) + 1e-9 * z)


def test_eight_views_in_one_call_equal_single_views(fused_256):
    from dynamicfusion_body_b200 import engine
    sc, live, f = fused_256
    all8 = [t.cpu().numpy() for t in engine.render(live, f, _ring_views(sc, sc.extrinsics))]
    for v in range(8):
        one = [t.cpu().numpy() for t in engine.render(live, f, _ring_views(sc, sc.extrinsics[v:v + 1]))]
        for a, b in zip(all8, one):
            assert np.array_equal(a[v:v + 1].view(np.uint32), b.view(np.uint32)), v


def _large_faces(K, rows, cols, rng):
    """Camera-frame triangles from a whole-image face down to sub-pixel ones, overlapping at random depths, plus exact ties."""
    Kinv = np.linalg.inv(K)

    def cam(x, y, z):
        return (Kinv @ np.array([x, y, 1.0])) * z

    tris = [[cam(-5 * cols, -5 * rows, 9.0), cam(10 * cols, -5 * rows, 9.0), cam(-5 * cols, 10 * rows, 9.0)]]   # covers the image
    tris.append([cam(-30, -40, 3.0), cam(cols + 50, 20, 5.0), cam(cols / 2, rows + 60, 4.0)])                  # past three borders
    for _ in range(400):
        ctr = rng.uniform([-50, -50], [cols + 50, rows + 50])
        size = np.exp(rng.uniform(np.log(0.5), np.log(400)))
        z = rng.uniform(2.0, 8.0, 3)
        tris.append([cam(*(ctr + size * rng.uniform(-1, 1, 2)), zi) for zi in z])
    tris.append(tris[-1])                                                                                    # an exact tie
    tris.append([cam(100, 100, 4.0), cam(300, 100, 4.0), cam(100, 300, 4.0)])                               # on pixel centres
    tris.append([cam(300, 100, 4.0), cam(300, 300, 4.0), cam(100, 300, 4.0)])
    pts = np.asarray(tris, np.float64).reshape(-1, 3)
    return pts, np.arange(len(pts), dtype=np.int32).reshape(-1, 3)


def test_large_faces_equal_oracle_and_take_the_large_face_path():
    import torch
    from dynamicfusion_body_b200 import engine, synth
    from oracle import render as orr
    rows, cols = 480, 640
    K = np.array([[525.0, 0, (cols - 1) / 2.0], [0, 525.0, (rows - 1) / 2.0], [0, 0, 1.0]])
    pts, faces = _large_faces(K, rows, cols, np.random.default_rng(3))
    for E in (None, np.stack([synth.look_at_extrinsic([0.3 * i, -0.2, -0.5 * i], [0.0, 0.0, 5.0]) for i in range(3)])):
        views = engine.camera_views(K, rows, cols, E)
        ws = engine.render_workspace(len(faces), views)
        dev = engine.render(pts, faces, views, workspace=ws)
        n_large = int(ws[0])
        ora = orr.render(pts, faces, K, rows, cols, E)
        _assert_bits(dev, ora)
        assert n_large > 50
        if E is None:
            assert (ora[1] >= 0).all()                               # the whole-image face leaves no pixel empty
        torch.cuda.synchronize()


def test_render_live_after_fusing_a_scene():
    import torch
    from dynamicfusion_body_b200 import engine, synth
    sc = synth.make_scene(res=128, k=4, n_nodes=400, seed=0, rows=240, cols=320)
    fus = _fusion(sc)
    for _ in range(3):
        fus.fuseFrame(sc.depths)
    out = fus.render_live(rows=sc.rows, cols=sc.cols)
    assert out.depth.shape == (1, sc.rows, sc.cols) and out.normal.shape == (1, sc.rows, sc.cols, 3)
    assert out.depth.is_cuda and out.face.dtype == torch.int32
    d = out.depth.cpu().numpy()[0]
    sil = sc.depths[0] != 0
    ok = (d != 0) & (np.abs(d - sc.depths[0]) <= sc.tdist)
    frac = float(ok[sil].mean())
    print("render_live: %.4f of the input silhouette within tdist, %d faces" % (frac, len(out.faces)))
    assert frac >= 0.95
    # the id map indexes the canonical mesh: a covered pixel lies in the live projection of its face's canonical vertices
    V, F = out.vertices, out.faces
    assert int(F.min()) >= 0 and int(F.max()) < len(V)
    face = out.face.cpu().numpy()[0]
    assert face.max() < len(F)
    r, c = np.nonzero(face >= 0)
    sel = np.random.default_rng(0).choice(len(r), 2000, replace=False)
    r, c = r[sel], c[sel]
    tri = F[torch.from_numpy(face[r, c]).long().cuda()].reshape(-1).long()
    live = engine.warp_points(fus._wf, fus._lw, V[tri], idx=fus._wf.knn_points(V[tri], sc.k), k=sc.k).cpu().numpy()
    q = live @ sc.K.T
    x, y = (q[:, 0] / q[:, 2]).reshape(-1, 3), (q[:, 1] / q[:, 2]).reshape(-1, 3)
    assert np.all((x.min(1) <= c + 1e-9) & (c <= x.max(1) + 1e-9) & (y.min(1) <= r + 1e-9) & (r <= y.max(1) + 1e-9))
    # the depth map is a depth frame: fuseFrame and projective association take it as it is
    w0 = float(fus._vol.weight.double().sum())
    fus.fuseFrame(out.depth)
    assert float(fus._vol.weight.double().sum()) > w0
    fus.setupCorrespondences(None, method='projective', depths=out.depth, prune_result=False)
    assert len(fus._corridx) > 0.2 * len(fus._vertices)
    # extrinsics: the same camera as a 3x4 view gives the same maps
    E = np.concatenate([np.eye(3), np.zeros((3, 1))], 1)
    two = fus.render_live(extrinsics=np.stack([E, E]), rows=sc.rows, cols=sc.cols)
    again = fus.render_live(rows=sc.rows, cols=sc.cols)
    assert torch.equal(two.depth[0], again.depth[0]) and torch.equal(two.face[1], again.face[0])


def test_render_live_empty_volume_and_missing_intrinsics():
    from dynamicfusion_body_b200.fusion import Fusion
    K = np.array([[100.0, 0, 31.5], [0, 100.0, 23.5], [0, 0, 1.0]])
    fus = Fusion(1.0, knn=4, use_cnn=False, write_warpfield=False)
    fus.InitializeCanonicalSpace(tsdf_shape=(32, 32, 32))
    with pytest.raises(ValueError):
        fus.render_live(rows=48, cols=64)
    out = fus.render_live(K=K, rows=48, cols=64)
    assert out.depth.shape == (1, 48, 64) and not out.depth.any() and (out.face == -1).all() and not out.normal.any()
    assert len(out.vertices) == 0 and len(out.faces) == 0
