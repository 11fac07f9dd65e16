"""Oracle against the UNMODIFIED reference executed live from a checkout at oracle/_ref/ (see oracle/refload.py; skipped
where it is absent -- the committed golden vectors cover that case).  Randomised inputs beyond the golden set."""
import numpy as np
import pytest

from oracle import dq as odq
from oracle import gn as ogn
from oracle import refload
from oracle import tsdf as ot


def live(test):
    """the test executes the reference: skipped where no checkout is present"""
    return pytest.mark.reference(pytest.mark.skipif(not refload.available(), reason="reference checkout not present")(test))


def _dq(rng, n, dtype):
    q = rng.normal(size=(n, 8)) * 0.1
    q[:, 0] += 1
    return q.astype(dtype)


def test_norm3_float32_semantics():
    """la.norm of a float32 3-vector (cblas_sdot accumulation) -- see oracle/dq.py:norm3_like_la."""
    from numpy import linalg as la
    rng = np.random.default_rng(0)
    x = (rng.normal(size=(20000, 3)) * 50).astype(np.float32)
    ref = np.array([la.norm(r) for r in x])
    assert np.array_equal(ref, odq.norm3_like_la(x))


@live
@pytest.mark.parametrize("seed", [0, 1])
@pytest.mark.parametrize("lw_dtype", [np.float32, np.float64])
def test_updateTSDF_live(seed, lw_dtype):
    rng = np.random.default_rng(seed)
    R, N, k = 9, 25, 4 if seed == 0 else 3
    node_pos = (rng.random((N, 3)) * R).astype(np.float32)
    node_dq = _dq(rng, N, np.float32)
    lw = _dq(rng, 1, lw_dtype)[0]
    tsdf = rng.normal(size=(R, R, R)); w = np.where(rng.random((R, R, R)) < 0.5, 0.0, rng.random((R, R, R)) * 120)
    curr = rng.normal(size=(R, R + 1, R))
    f = refload.make_fusion([(i, node_pos[i], node_dq[i], 4.0) for i in range(N)], tsdf.copy(), w.copy(), 0.7, k, lw)
    with refload.quiet():
        f.updateTSDF(curr)
    vox = ot.voxel_grid((R, R, R))
    kd = np.array([f._kdtree.query(v, k=k + 1)[1][:-1] for v in vox])
    v, ww, m = ot.update_volume(tsdf.ravel(), w.ravel(), curr, vox, kd, node_pos, node_dq, np.full(N, 4.0), lw, 0.7)
    assert np.array_equal(v, f._tsdf.ravel()) and np.array_equal(ww, f._tsdfw.ravel())
    idx, d2 = odq.knn_bruteforce(vox, node_pos, k)
    tie = odq.knn_has_tie(d2)
    assert np.array_equal(idx[~tie], kd[~tie])


@live
def test_updateTSDF_errors_like_reference():
    f = refload.make_fusion([(0, np.zeros(3, np.float32), np.array([1, 0, 0, 0, 0, 0, 0, 0], np.float32), 1.0)] * 5,
                            np.zeros((2, 2, 2)), np.zeros((2, 2, 2)), 1.0, 4, np.array([1, 0, 0, 0, 0, 0, 0, 0], np.float32))
    with pytest.raises(ValueError):
        f.updateTSDF(None)
    with pytest.raises(ValueError):
        f.updateTSDF(np.zeros((3, 3)))


@live
def test_fuseDepths_live():
    util, Fusion, FusionDM = refload.load()
    rng = np.random.default_rng(3)
    R = 8
    K = np.array([[50., 0, 20], [0, 55., 15], [0, 0, 1]])
    fdm = FusionDM(0.5, K, tsdf_res=R)
    dm = -(rng.random((32, 40)) * 6 + 10).astype(np.float32); dm[rng.random((32, 40)) < 0.3] = 0
    lw34 = np.concatenate([np.eye(3), np.array([[0.2], [0.1], [12.]])], 1)
    t0 = rng.normal(size=(R, R, R)); w0 = np.floor(rng.random((R, R, R)) * 3)
    with refload.quiet():
        rt, rw = fdm.fuseDepths(dm, lw34, t0.copy(), w0.copy(), scale=0.9, center=np.array([0.1, -0.1, 0.0]))
    v, w, m, fr = ot.fuse_depth_rigid(t0.ravel(), w0.ravel(), ot.voxel_grid((R, R, R)), dm, lw34, K, np.linalg.inv(K), 0.5, R, scale=0.9,
                                      center=np.array([0.1, -0.1, 0.0]))
    assert np.array_equal(v, rt.ravel()) and np.array_equal(w, rw.ravel()) and m.sum() > 10


@live
def test_computef_live():
    rng = np.random.default_rng(5)
    N, V, k = 20, 50, 4
    node_pos = (rng.random((N, 3)) * 10).astype(np.float32)
    node_dq = _dq(rng, N, np.float32)
    verts = (rng.random((V, 3)) * 10).astype(np.float32); norms = rng.normal(size=(V, 3)).astype(np.float32)
    corr = verts + rng.normal(size=(V, 3)) * 0.1
    lw = _dq(rng, 1, np.float64)[0]
    nvi = rng.integers(0, V, N)
    nodes = [(int(nvi[i]), node_pos[i], node_dq[i], 5.0) for i in range(N)]
    f = refload.make_fusion(nodes, None, None, 1.0, k, lw)
    vknn = np.array([f._kdtree.query(v, k=k)[1] for v in verts])
    f._vertices, f._normals, f._neighbor_look_up, f._correspondences = verts, norms, list(vknn), corr
    x = node_dq.reshape(-1).astype(np.float64) + rng.normal(size=8 * N) * 1e-3
    ref = f.computef(x, 0.2, 0.001, 0.7)
    mine = ogn.computef(x, verts, norms, corr, vknn, node_pos, 5.0, nvi, lw, 0.7)
    assert np.abs(ref - mine).max() <= 1e-13
    # Q7: the reference's own sparsity pattern misses most regularisation rows; ours covers every non-zero
    sp_ref = f.computeSparsity(len(ref), len(x)).toarray() > 0
    sp = ogn.sparsity_pattern(vknn, nvi, N).toarray() > 0
    assert sp_ref[:V].sum() == sp[:V].sum()
    assert (sp_ref[V + 3 * N:].sum() == 0) and sp[V + 3 * N:].sum() > 0


# ---- SURVEY 8f ranks 1-2: correspondences and graph maintenance (oracle/graph.py) --------------------------------
def _corr_scene(rng, V=60, L=300, N=20, k=4):
    from oracle import graph as og  # noqa: F401
    node_pos = (rng.random((N, 3)) * 10).astype(np.float32)
    node_dq = _dq(rng, N, np.float32)
    verts = (rng.random((V, 3)) * 10).astype(np.float32)
    norms = rng.normal(size=(V, 3)).astype(np.float32)
    norms /= np.linalg.norm(norms, axis=1, keepdims=True)
    lverts = (rng.random((L, 3)) * 10).astype(np.float32)
    return node_pos, node_dq, verts, norms, lverts


@live
def test_setupCorrespondences_live():
    """Fusion.setupCorrespondences (clpts branch, core/fusion.py:258-276) with marching cubes replaced by the live vertices."""
    from oracle import graph as og
    rng = np.random.default_rng(11)
    N, k = 20, 4
    node_pos, node_dq, verts, norms, lverts = _corr_scene(rng, N=N, k=k)
    lw = _dq(rng, 1, np.float64)[0]
    nodes = [(0, node_pos[i], node_dq[i], 5.0) for i in range(N)]
    f = refload.make_fusion(nodes, None, None, 1.0, k, lw)
    vknn = np.array([f._kdtree.query(v, k=k)[1] for v in verts])
    f._vertices, f._normals, f._neighbor_look_up = verts, norms, list(vknn)
    f.marching_cubes = lambda *a, **kw: (lverts, None, None, None)
    with refload.quiet():
        f.setupCorrespondences(np.zeros((2, 2, 2)), method='clpts', prune_result=False)
    ref = np.array(f._correspondences)
    wv, wn = odq.warp(verts, node_pos[vknn], node_dq[vknn], np.full(vknn.shape, 5.0), lw=lw, normal=norms)
    nn, _ = og.knn_points(lverts, wv, k)
    best, cost = og.corr_select(wv, wn, lverts, nn)
    assert not og.knn_tie(lverts, wv, k).any()
    assert np.array_equal(ref, lverts[best])
    assert (cost < 1).any() and (cost == 1).any()


@live
def test_fusiondm_setupCorrespondences_live():
    """FusionDM.setupCorrespondences (core/fusion_dm.py:219-244): rigid warp by _lw, keeps best_cost <= tolerance."""
    from oracle import graph as og
    util, Fusion, FusionDM = refload.load()
    rng = np.random.default_rng(12)
    _, _, verts, norms, lverts = _corr_scene(rng)
    fdm = FusionDM(0.5, np.eye(3), tsdf_res=4)
    fdm._lw = _dq(rng, 1, np.float64)[0]
    fdm._vertices, fdm._normals = verts, norms
    fdm.marching_cubes = lambda *a, **kw: (lverts, None, None, None)
    with refload.quiet():
        fdm.setupCorrespondences(None, tolerance=0.3)
    wv = odq.dqb_warp(fdm._lw, verts)
    wn = odq.dqb_warp_normal(fdm._lw, norms)
    nn, _ = og.knn_points(lverts, wv, fdm._knn)
    best, cost = og.corr_select(wv, wn, lverts, nn)
    keep = np.nonzero(cost <= 0.3)[0]
    assert 0 < len(keep) < len(verts)
    assert np.array_equal(np.array(fdm._corridx), keep)
    assert np.array_equal(np.array(fdm._correspondences), lverts[best[keep]])


@live
def test_uniform_sample_live():
    from oracle import graph as og
    util, _, _ = refload.load()
    rng = np.random.default_rng(13)
    pts = (rng.random((500, 3)) * 10).astype(np.float32)
    for radius in (0.8, 1.7, 30.0):
        rv, ri = util.uniform_sample(pts, radius)
        ov, oi = og.uniform_sample(pts, radius)
        assert np.array_equal(ri, oi) and np.array_equal(rv, ov)


@live
def test_update_graph_live():
    """Fusion.update_graph (core/fusion.py:201-239) with marching cubes a no-op: vertex re-linking, unsupported points,
    new nodes initialised by dq_blend, refreshed vertex->node table."""
    from oracle import graph as og
    rng = np.random.default_rng(14)
    N, k, V = 12, 4, 150
    node_pos = (rng.random((N, 3)) * 4 + 3).astype(np.float32)
    node_dq = _dq(rng, N, np.float32)
    verts = (rng.random((V, 3)) * 10).astype(np.float32)
    radius = 1.1
    nodes = [(0, node_pos[i], node_dq[i], 2 * radius) for i in range(N)]
    f = refload.make_fusion(nodes, None, None, 1.0, k, _dq(rng, 1, np.float64)[0])
    f._vertices, f._radius = verts, radius
    f.marching_cubes = lambda *a, **kw: None
    with refload.quiet():
        f.update_graph()
    vknn, _ = og.knn_points(node_pos, verts, k)
    uns = og.unsupported(verts, vknn, node_pos, np.full(N, 2 * radius))
    assert 0 < uns.sum() < V
    new_v, new_i = og.uniform_sample(verts[uns], radius)
    assert len(f._nodes) == N + len(new_v)
    assert np.array_equal(np.array([n[1] for n in f._nodes[N:]]), new_v)
    assert [n[0] for n in f._nodes[N:]] == list(new_i)
    link, _ = og.knn_points(verts, node_pos, 1)
    assert [n[0] for n in f._nodes[:N]] == list(link[:, 0])
    # new node transforms: dq_blend at the new position over the OLD graph's k nearest nodes (core/fusion.py:219-223)
    nk, _ = og.knn_points(node_pos, new_v, k)
    b = odq.dq_blend(new_v, node_pos[nk], node_dq[nk], np.full(nk.shape, 2 * radius))
    assert np.abs(np.array([n[2] for n in f._nodes[N:]]) - b).max() <= 1e-15
    allpos = np.array([n[1] for n in f._nodes])
    look, _ = og.knn_points(allpos, verts, k)
    assert np.array_equal(np.array(f._neighbor_look_up), look)


@live
def test_fuseDepths_invalid_depth_values_live():
    """NaN, +-inf and positive depth pixels through the unmodified FusionDM.fuseDepths: all skipped (an infinite depth
    becomes NaN in K^-1 * (z*u, z*v, z) for a pinhole K) -- the oracle follows op for op."""
    util, Fusion, FusionDM = refload.load()
    rng = np.random.default_rng(4)
    R = 8
    K = np.array([[50., 0, 20], [0, 55., 15], [0, 0, 1]])
    fdm = FusionDM(0.5, K, tsdf_res=R)
    dm = -(rng.random((32, 40)) * 6 + 10).astype(np.float32)
    r = rng.random(dm.shape)
    dm[r < 0.15] = np.nan; dm[(r >= 0.15) & (r < 0.3)] = np.inf; dm[(r >= 0.3) & (r < 0.45)] = -np.inf; dm[(r >= 0.45) & (r < 0.6)] = 3.0
    lw34 = np.concatenate([np.eye(3), np.array([[0.2], [0.1], [12.]])], 1)
    t0 = rng.normal(size=(R, R, R)); w0 = np.floor(rng.random((R, R, R)) * 3)
    with refload.quiet(), np.errstate(invalid="ignore"):
        rt, rw = fdm.fuseDepths(dm, lw34, t0.copy(), w0.copy())
        v, w, m, fr = ot.fuse_depth_rigid(t0.ravel(), w0.ravel(), ot.voxel_grid((R, R, R)), dm, lw34, K, np.linalg.inv(K), 0.5, R)
    assert np.array_equal(v, rt.ravel()) and np.array_equal(w, rw.ravel())
    assert 0 < m.sum() < fr.sum() and np.isfinite(rt).all()


@live
def test_fuseDepths_camera_inside_volume_live():
    """Voxels behind the camera (negative projective divisor) and exactly on the camera plane (divisor 0 -> None) through
    the unmodified FusionDM.fuseDepths (core/util.py:312-320 has no sign test)."""
    util, Fusion, FusionDM = refload.load()
    rng = np.random.default_rng(6)
    R = 8
    K = np.array([[12., 0, 20], [0, 12., 16], [0, 0, 1]])
    fdm = FusionDM(0.5, K, tsdf_res=R)
    dm = -(rng.random((32, 40)) * 3 + 1).astype(np.float32)
    lw34 = np.concatenate([np.eye(3), np.zeros((3, 1))], 1)                     # camera at the volume centre (pos = idx - R/2)
    t0 = rng.normal(size=(R, R, R)); w0 = np.floor(rng.random((R, R, R)) * 3)
    with refload.quiet(), np.errstate(all="ignore"):
        rt, rw = fdm.fuseDepths(dm, lw34, t0.copy(), w0.copy())
        v, w, m, fr = ot.fuse_depth_rigid(t0.ravel(), w0.ravel(), ot.voxel_grid((R, R, R)), dm, lw34, K, np.linalg.inv(K), 0.5, R)
    assert np.array_equal(v, rt.ravel()) and np.array_equal(w, rw.ravel())
    m = m.reshape(R, R, R)
    assert m[:, :, :R // 2].any() and m[:, :, R // 2 + 1:].any() and not m[:, :, R // 2].any()
