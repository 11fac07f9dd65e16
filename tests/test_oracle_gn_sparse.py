"""CPU tests of the sparse extensions of oracle/gn.py: sparse normal equations, the node_nbr override, the float64
block-Jacobi PCG restatement of the device solve and the sparse-LU step.  The GPU tests of the solver
(tests/test_gpu_gn_shapes.py) judge the device against these, so they are pinned here against the dense oracle."""
import numpy as np
import pytest

from oracle import gn as ogn


@pytest.fixture(scope="module")
def system():
    from dynamicfusion_body_b200 import synth
    sc = synth.make_scene(res=64, k=4, n_nodes=60, seed=0, rows=48, cols=64)
    d = synth.make_gn_problem(sc, 2000, seed=1, noise=0.05)
    nw = float(np.float32(sc.node_w))
    args = (d.vertices, d.normals, d.corr, d.vert_knn, sc.node_pos, nw, d.node_vertex_idx, sc.lw, 0.05)
    return sc, d, args


def test_sparse_normal_equations_equal_dense(system):
    sc, d, args = system
    J, f = ogn.jacobian(d.x0, *args)
    for huber in (False, True):
        Hd, gd = ogn.normal_equations(J, f, 0.3, huber)
        Hs, gs = ogn.normal_equations(J, f, 0.3, huber, dense=False)
        assert Hs.format == "csr" and Hs.has_sorted_indices
        assert np.array_equal(Hs.toarray(), Hd)
        assert np.array_equal(gs, gd)


def test_node_nbr_default_reproduces_output(system):
    sc, d, args = system
    nbr = ogn.reg_neighbours(d.vert_knn, d.node_vertex_idx)
    f0 = ogn.computef(d.x0, *args)
    f1 = ogn.computef(d.x0, *args, node_nbr=nbr)
    assert np.array_equal(f0, f1)
    J0, r0 = ogn.jacobian(d.x0, *args)
    J1, r1 = ogn.jacobian(d.x0, *args, node_nbr=nbr)
    assert np.array_equal(r0, r1)
    assert (J0 != J1).nnz == 0
    # a different table changes the regularisation rows only
    f2 = ogn.computef(d.x0, *args, node_nbr=np.roll(nbr, 1, axis=0))
    V = len(d.vertices)
    assert np.array_equal(f2[:V], f0[:V]) and not np.array_equal(f2[V:], f0[V:])


@pytest.mark.parametrize("lam", [1e-1, 1e-3])
def test_pcg_block_jacobi_and_sparse_step_reach_gn_step(system, lam):
    sc, d, args = system
    J, f = ogn.jacobian(d.x0, *args)
    Hd, g = ogn.normal_equations(J, f)
    Hs, _ = ogn.normal_equations(J, f, dense=False)
    ref = ogn.gn_step(Hd, g, lam)
    ds = ogn.sparse_gn_step(Hs, g, lam)
    assert np.linalg.norm(ds - ref) <= 1e-10 * np.linalg.norm(ref)
    dp, it = ogn.pcg_block_jacobi(Hs, g, lam, 1e-14, 5000)
    assert 0 < it < 5000
    assert np.linalg.norm(dp - ref) <= 1e-9 * np.linalg.norm(ref)
    # the iteration count is the number of updates applied: max_iter caps it exactly, and the iterates are those of CG
    d1, it1 = ogn.pcg_block_jacobi(Hs, g, lam, 0.0, 1)
    assert it1 == 1
    n = Hs.shape[0] // 8
    mu = lam * np.trace(Hd) / (8 * n)
    M = np.zeros_like(Hd)
    for i in range(n):
        M[8 * i:8 * i + 8, 8 * i:8 * i + 8] = np.linalg.inv(Hd[8 * i:8 * i + 8, 8 * i:8 * i + 8] + mu * np.eye(8))
    z0 = M @ -g
    A = Hd + mu * np.eye(8 * n)
    alpha = (-g @ z0) / (z0 @ A @ z0)
    assert np.linalg.norm(d1 - alpha * z0) <= 1e-12 * np.linalg.norm(d1)
    # the stopping rule is the device's: (r, z) <= tol^2 (r0, z0)
    d4, it4 = ogn.pcg_block_jacobi(Hs, g, lam, 1e-4, 5000)
    r = -g - A @ d4
    rz0 = float(-g @ z0)
    assert r @ (M @ r) <= 1e-8 * rz0 * (1 + 1e-6)
    _, it4m = ogn.pcg_block_jacobi(Hs, g, lam, 1e-4, it4 - 1)
    assert it4m == it4 - 1


def test_gauss_newton_loop_sparse_equals_dense(system):
    sc, d, args = system
    xd, c0d, cd, ad = ogn.gauss_newton_loop(d.x0, *args, max_iter=3)
    xs, c0s, cs, as_ = ogn.gauss_newton_loop(d.x0, *args, max_iter=3, sparse=True)
    assert ad == as_ and c0d == c0s
    assert abs(cs - cd) <= 1e-10 * cd
    assert np.linalg.norm(xs - xd) <= 1e-9 * np.linalg.norm(xd)
