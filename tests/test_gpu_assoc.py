"""Projective data association on the device (run with -m gpu): dfb_corr_projective against oracle/assoc.py bit for bit,
its geometry on a scene with a known warp field, and Fusion.setupCorrespondences(method='projective') driving solve and
the depth-only frame loop  setupCorrespondences(depths) -> solve -> fuseFrame(depths) -> update_graph."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _fusion(sc, **kw):
    """A Fusion object holding the scene's canonical model: the body mesh with its normals turned outward (the fixture's point
    into the body; association takes them as marching cubes of the TSDF gives them), the scene's nodes, `_lw` = the camera."""
    from dynamicfusion_body_b200.fusion import Fusion
    fus = Fusion(sc.tdist, knn=sc.k, use_cnn=False, write_warpfield=False, **kw)
    R = sc.res
    fus.InitializeCanonicalSpace(tsdf_shape=(R, R, R), K=sc.K, vertices=sc.vertices, normals=-sc.normals, faces=sc.faces,
                                 nodes=sc.nodes_as_reference_tuples(), radius=sc.radius)
    fus._lw = sc.lw
    return fus


def _device_warp(sc):
    import torch
    from dynamicfusion_body_b200 import engine
    wf = engine.DeviceWarpField(sc.k)
    wf.set_nodes(sc.node_pos, sc.node_dq, np.float32(sc.node_w))
    return engine.warp_points(wf, sc.lw, sc.vertices, -sc.normals, idx=sc.vert_knn.astype(np.int32), k=sc.k)


@pytest.mark.parametrize("n_views", [1, 8])
def test_parity_with_oracle_256(n_views):
    import torch
    from dynamicfusion_body_b200 import engine, synth
    from oracle import assoc as oa
    sc = synth.make_scene(res=256, k=8, n_nodes=1000, seed=0, n_views=n_views, background=True)
    wv, wn = _device_warp(sc)
    views = engine.make_views(torch.from_numpy(sc.depths).cuda(), sc.K, sc.Kinv, sc.extrinsics)
    for md, mnd in ((sc.tdist, 0.5), (2.5 * sc.tdist, -0.25)):
        view, cost, corr = engine.corr_projective(wv, wn, views, md, mnd)
        ov, oc, op = oa.associate(wv.cpu().numpy(), wn.cpu().numpy(), sc.depths, sc.K, sc.Kinv, md, mnd, sc.extrinsics)
        assert np.array_equal(view.cpu().numpy(), ov)
        assert np.array_equal(cost.cpu().numpy().view(np.uint64), oc.view(np.uint64))
        assert np.array_equal(corr.cpu().numpy().view(np.uint64), op.view(np.uint64))
        assert (ov >= 0).mean() > 0.2
        if n_views > 1:
            assert len(np.unique(ov[ov >= 0])) == n_views


def test_geometry_with_the_true_warp():
    """Under the scene's own warp most visible vertices associate, and their live points lie within a pixel footprint of them
    along the normal (point-to-plane, what the solve uses).  The full distance |corr - w| is also bounded, by 1.5 footprints: the
    synthetic renderer (synth.render_depth) splats every surface sample over a 2x2 pixel block into a min-depth z-buffer, which
    moves a slanted surface's measured depth up to about a pixel toward the camera (host build at this size: median |corr - w|
    0.58 voxels of which 0.31 along the normal, footprint 0.44-0.56)."""
    import torch
    from dynamicfusion_body_b200 import engine, synth
    sc = synth.make_scene(res=256, k=4, n_nodes=1000, seed=0, focal=775.0)
    wv, wn = _device_warp(sc)
    views = engine.make_views(torch.from_numpy(sc.depths).cuda(), sc.K, sc.Kinv, None)
    view, cost, corr = engine.corr_projective(wv, wn, views, sc.tdist, 0.5)
    w, n = wv.cpu().numpy(), wn.cpu().numpy()
    hit = view.cpu().numpy() >= 0
    p = w @ sc.K.T
    u, v = p[:, 0] / p[:, 2], p[:, 1] / p[:, 2]
    visible = ((n * w).sum(1) < 0) & (u >= 1) & (u < sc.cols - 2) & (v >= 1) & (v < sc.rows - 2)   # front-facing, in the frustum
    frac = hit[visible].mean()
    footprint = float(np.median(w[hit, 2])) / sc.K[0, 0]
    dc = corr.cpu().numpy()[hit] - w[hit]
    err = float(np.median(np.linalg.norm(dc, axis=1)))
    err_n = float(np.median(np.abs((dc * n[hit]).sum(1)) / np.linalg.norm(n[hit], axis=1)))
    print("associated: %.3f of front-facing in-frustum vertices (%.3f of all); median |corr - w| = %.3f voxels, along the normal "
          "%.3f, pixel footprint %.3f" % (frac, hit.mean(), err, err_n, footprint))
    assert frac > 0.5 and err_n < footprint and err < 1.5 * footprint
    assert np.isinf(cost.cpu().numpy()[~hit]).all() and not corr.cpu().numpy()[~hit].any()


def test_solve_from_perturbed_transforms():
    import torch
    from dynamicfusion_body_b200 import synth
    sc = synth.make_scene(res=64, k=4, n_nodes=300, seed=0)
    fus = _fusion(sc)
    x0 = synth.make_gn_problem(sc, 10, seed=1, perturb=1e-2).x0
    fus.set_node_dqs(x0.reshape(-1, 8).astype(np.float32))
    fus.setupCorrespondences(None, method='projective', depths=sc.depths, prune_result=False)
    V, nlu = fus._vertices, fus._neighbor_look_up
    nw = np.full(sc.n_nodes, np.float32(sc.node_w))
    truth = synth.blend_warp(V, sc.node_pos, sc.node_dq, nw, nlu, lw=sc.lw)
    before = np.linalg.norm(fus.warp(V, locations=nlu, m_lw=fus._lw) - truth, axis=1).mean()
    fus.solve(method='projective', regularization_weight=0.5, gn_iterations=10)
    after = np.linalg.norm(fus.warp(V, locations=nlu, m_lw=fus._lw) - truth, axis=1).mean()
    print("projective solve: robust cost %.4e -> %.4e, mean distance to the true warp %.4f -> %.4f voxels"
          % (fus.last_solve.cost0, fus.last_solve.cost, before, after))
    assert fus._vertices is V
    assert fus.last_solve.cost < fus.last_solve.cost0
    assert after < before
    torch.cuda.synchronize()


def test_depth_only_driver_loop():
    import torch
    from dynamicfusion_body_b200 import synth
    frames = [synth.make_scene(res=80, k=4, n_nodes=300, seed=0, rows=240, cols=320, max_disp=a) for a in (0.3, 0.5, 0.7)]
    fus = _fusion(frames[0])
    w_prev = 0.0
    for sc in frames:
        d = torch.from_numpy(sc.depths).cuda()
        fus.setupCorrespondences(None, method='projective', depths=d)                  # no live TSDF, no live vertices
        assert len(fus._correspondences) == len(fus._vertices) > 100
        fus.solve(method='projective', regularization_weight=0.5, gn_iterations=6)
        assert fus.last_solve.cost <= fus.last_solve.cost0 and np.isfinite(fus.last_solve.cost)
        fus.fuseFrame(d)
        w = float(fus._vol.weight.double().sum())
        assert w > w_prev and torch.isfinite(fus._vol.tsdf).all()
        w_prev = w
        fus.update_graph()                                                             # canonical surface from the fused volume
        assert fus._curr_depths is None and fus._correspondences == []
        assert len(fus._vertices) > 100
    with pytest.raises(ValueError):
        fus.solve(method='projective')                                                 # the frame was released by update_graph


def test_subset_path_and_arguments():
    from dynamicfusion_body_b200 import synth
    sc = synth.make_scene(res=64, k=4, n_nodes=300, seed=2, rows=240, cols=320)
    fus = _fusion(sc)
    V = fus._vertices
    fus.setupCorrespondences(None, method='projective', depths=sc.depths, prune_result=False)
    assert fus._vertices is V and 0 < len(fus._corridx) < len(V)
    assert len(fus._correspondences) == len(fus._corridx)
    x = fus._wf.node_dq.double().reshape(-1).cpu().numpy()
    f = fus.computef(x, 0.2, 0.001, 0.5)
    assert f.shape == (len(fus._corridx) + 3 * sc.k * sc.n_nodes,)
    # the regularisation rows are those of the full problem
    fus2 = _fusion(sc)
    fus2.setupCorrespondences(None, method='projective', depths=sc.depths, prune_result=False)
    fus2._corridx = None
    fus2._correspondences = np.zeros((len(V), 3))
    assert np.array_equal(fus2.computef(x, 0.2, 0.001, 0.5)[len(V):], f[len(fus._corridx):])
    # prune_result=True keeps exactly the vertices the subset held
    fus.setupCorrespondences(None, method='projective', depths=sc.depths)
    assert len(fus._vertices) == len(fus._correspondences) == len(f) - 3 * sc.k * sc.n_nodes
    with pytest.raises(ValueError):
        fus.setupCorrespondences(None, method='projective')
    with pytest.raises(ValueError):
        fus.setupCorrespondences(None, method='clpts', depths=sc.depths)
