"""CPU oracle, part 3: the warp-field least-squares path -- TEST INFRASTRUCTURE ONLY (see oracle/dq.py).

residual functions  computef / computef_lw   restate core/fusion.py:459-491 / :444-456 op for op
                                             (pinned against the reference by tests/test_oracle_vs_reference.py);
Jacobian            analytic, float64; validated against scipy's 2-point finite differences of the residual
                    function -- exactly what the reference's least_squares(jac='2-point') call differentiates
                    (core/fusion.py:382-392) -- by tests/test_oracle_gn.py;
Gauss-Newton step   the reference has none (it calls scipy TRF/LSMR, SURVEY 8a a12): the step oracle is DEFINED
                    here as  delta = solve(J^T W J + lam * mean(diag) * I, -J^T W f)  in float64 numpy with the
                    Huber IRLS weights W = min(1, f_scale/|f|); "parity unpinned" for the optimiser trajectory.
"""
import numpy as np

from . import dq as _dq


# ---------------------------------------------------------------------------------------------------
# residuals (reference arithmetic)
# ---------------------------------------------------------------------------------------------------
def reg_neighbours(vert_knn, node_vertex_idx):
    """`self._neighbor_look_up[self._nodes[idx][0]]` (core/fusion.py:477): the k node ids around each node."""
    return np.asarray(vert_knn)[np.asarray(node_vertex_idx)]


def computef(x, vertices, normals, corr, vert_knn, node_pos, node_w, node_vertex_idx, lw, rw, node_nbr=None):
    """core/fusion.py:459-491.  x (8N,) (its dtype matters exactly like in the reference: `dqs = np.split(x, ...)`).
    node_nbr (N,k): regularisation neighbours of every node (default reg_neighbours(vert_knn, node_vertex_idx)); a problem over a
    subset of the vertices passes the rows of the full vertex->node table, like gn.Problem(node_nbr=)."""
    x = np.asarray(x)
    dqs = x.reshape(-1, 8)
    n_nodes = len(dqs)
    node_w = np.broadcast_to(np.asarray(node_w, dtype=np.float64), (n_nodes,))
    vw, nw = _dq.warp(vertices, node_pos[vert_knn], dqs[vert_knn], node_w[vert_knn], lw=lw, normal=normals)
    f_data = np.einsum('ij,ij->i', nw, vw - corr)
    nbr = reg_neighbours(vert_knn, node_vertex_idx) if node_nbr is None else np.asarray(node_nbr)   # (N,k)
    k = nbr.shape[1]
    pj = node_pos[nbr]                                           # (N,k,3) dgj_v
    di = _dq.dqb_warp(dqs[:, None, :], pj)                       # dqb_warp(dgi_se3, dgj_v)
    dj = _dq.dqb_warp(dqs[nbr], pj)                              # dqb_warp(dgj_se3, dgj_v)
    diff = di - dj
    # rw * max(w_i, w_j) * diff[i]  -- python floats: (rw*max)*diff
    c = rw * np.maximum(node_w[:, None], node_w[nbr])
    f_reg = (c[..., None] * diff).reshape(-1)
    return np.concatenate([f_data, f_reg])


def computef_lw(x, vertices, normals, corr, vert_knn, node_pos, node_dq, node_w):
    """core/fusion.py:444-456: data term only, as a function of the global rigid dq x (8,)."""
    n_nodes = len(node_pos)
    node_w = np.broadcast_to(np.asarray(node_w, dtype=np.float64), (n_nodes,))
    vw, nw = _dq.warp(vertices, node_pos[vert_knn], node_dq[vert_knn], node_w[vert_knn], lw=np.asarray(x), normal=normals)
    return np.einsum('ij,ij->i', nw, vw - corr)


def sparsity_pattern(vert_knn, node_vertex_idx, n_nodes):
    """Correct Jacobian pattern (rows V + 3kN, cols 8N) as a scipy CSR of ones.  (The reference's computeSparsity,
    core/fusion.py:416-442, covers only 3N of the 3kN regularisation rows -- SURVEY Q7 -- and is not reproduced.)"""
    from scipy.sparse import csr_matrix
    vert_knn = np.asarray(vert_knn)
    V, k = vert_knn.shape
    rows, cols = [], []
    r = np.repeat(np.arange(V), k * 8)
    c = (vert_knn[:, :, None] * 8 + np.arange(8)[None, None, :]).reshape(-1)
    rows.append(r); cols.append(c)
    nbr = reg_neighbours(vert_knn, node_vertex_idx)
    base = V
    for i in range(n_nodes):
        for jj in range(k):
            j = nbr[i, jj]
            for comp in range(3):
                row = base + (i * k + jj) * 3 + comp
                cc = np.concatenate([i * 8 + np.arange(8), j * 8 + np.arange(8)])
                rows.append(np.full(16, row)); cols.append(cc)
    rows = np.concatenate(rows); cols = np.concatenate(cols)
    m = csr_matrix((np.ones(len(rows)), (rows, cols)), shape=(V + 3 * k * n_nodes, 8 * n_nodes))
    m.data[:] = 1
    return m


# ---------------------------------------------------------------------------------------------------
# analytic derivatives (float64, smooth model: the float32 roundings of the reference are not differentiated)
# ---------------------------------------------------------------------------------------------------
def _skew(v):
    z = np.zeros(v.shape[:-1])
    return np.stack([np.stack([z, -v[..., 2], v[..., 1]], -1),
                     np.stack([v[..., 2], z, -v[..., 0]], -1),
                     np.stack([-v[..., 1], v[..., 0], z], -1)], -2)


def W(q, p):
    """dqb_warp closed form (quadratic in q): (w^2-|v|^2)p + 2(v.p)v + 2w(v x p) + 2(w dv - dw v + v x dv)."""
    w, v, dw, dv = q[..., 0:1], q[..., 1:4], q[..., 4:5], q[..., 5:8]
    return (w * w - (v * v).sum(-1, keepdims=True)) * p + 2 * (v * p).sum(-1, keepdims=True) * v + 2 * w * np.cross(v, p) \
        + 2 * (w * dv - dw * v + np.cross(v, dv))


def dW_dq(q, p, rotation_only=False):
    """(...,3,8) Jacobian of W(q,p) w.r.t. q.  rotation_only: the dqb_warp_normal variant (dual part zeroed)."""
    shape = np.broadcast_shapes(q.shape[:-1], p.shape[:-1])
    q = np.broadcast_to(q, shape + (8,))
    p = np.broadcast_to(p, shape + (3,))
    w, v, dw, dv = q[..., 0:1], q[..., 1:4], q[..., 4:5], q[..., 5:8]
    if rotation_only:
        dw = np.zeros_like(dw); dv = np.zeros_like(dv)
    I = np.broadcast_to(np.eye(3), shape + (3, 3))
    J = np.zeros(shape + (3, 8))
    J[..., :, 0] = 2 * w * p + 2 * np.cross(v, p) + 2 * dv
    J[..., :, 1:4] = (-2 * p[..., :, None] * v[..., None, :] + 2 * v[..., :, None] * p[..., None, :]
                      + 2 * (v * p).sum(-1)[..., None, None] * I - 2 * w[..., None] * _skew(p)
                      - 2 * dw[..., None] * I - 2 * _skew(dv))
    if not rotation_only:
        J[..., :, 4] = -2 * v
        J[..., :, 5:8] = 2 * w[..., None] * I + 2 * _skew(v)
    return J


def affine_of(q):
    """(A 3x3, t 3) with W(q,p) = A p + t."""
    e = np.eye(3)
    t = W(q, np.zeros(3))
    A = np.stack([W(q, e[i]) - t for i in range(3)], -1)
    return A, t


def data_jacobian_parts(x, vertices, normals, corr, vert_knn, node_pos, node_w, lw):
    """Per data residual: r (V,), g (V,8) = d r / d b  (b = un-normalised blend), wts (V,k) so that
    d r / d dq_a = wts[:,a] * g.  float64 smooth model."""
    dqs = np.asarray(x, dtype=np.float64).reshape(-1, 8)
    n_nodes = len(dqs)
    node_w = np.broadcast_to(np.asarray(node_w, dtype=np.float64), (n_nodes,))
    p = np.asarray(vertices, dtype=np.float64)
    n = np.asarray(normals, dtype=np.float64)
    npk = node_pos.astype(np.float64)[vert_knn]
    d2 = ((p[:, None, :] - npk) ** 2).sum(-1)
    wts = np.exp(-d2 / (4.0 * node_w[vert_knn] ** 2))
    b = (wts[..., None] * dqs[vert_knn]).sum(1)
    s = np.linalg.norm(b, axis=1, keepdims=True)
    bh = b / s
    A, t = affine_of(np.asarray(lw, dtype=np.float64))
    v1 = W(bh, p)
    rq = bh.copy(); rq[:, 4:] = 0
    n1 = W(rq, n)
    v2 = v1 @ A.T + t
    n2 = n1 @ A.T
    r = np.einsum('ij,ij->i', n2, v2 - corr)
    Jv = dW_dq(bh, p)                       # (V,3,8)
    Jn = dW_dq(bh, n, rotation_only=True)
    gt = np.einsum('vi,ij,vjc->vc', n2, A, Jv) + np.einsum('vi,ij,vjc->vc', v2 - corr, A, Jn)
    g = (gt - bh * (bh * gt).sum(1, keepdims=True)) / s
    return r, g, wts


def jacobian(x, vertices, normals, corr, vert_knn, node_pos, node_w, node_vertex_idx, lw, rw, node_nbr=None):
    """Sparse analytic Jacobian (CSR, rows V + 3kN, cols 8N) of computef and its residual vector.  node_nbr: as in computef."""
    from scipy.sparse import csr_matrix
    dqs = np.asarray(x, dtype=np.float64).reshape(-1, 8)
    n_nodes = len(dqs)
    vert_knn = np.asarray(vert_knn)
    V, k = vert_knn.shape
    node_wa = np.broadcast_to(np.asarray(node_w, dtype=np.float64), (n_nodes,))
    r, g, wts = data_jacobian_parts(x, vertices, normals, corr, vert_knn, node_pos, node_w, lw)
    rows = np.repeat(np.arange(V), k * 8)
    cols = (vert_knn[:, :, None] * 8 + np.arange(8)[None, None, :]).reshape(-1)
    vals = (wts[:, :, None] * g[:, None, :]).reshape(-1)
    nbr = reg_neighbours(vert_knn, node_vertex_idx) if node_nbr is None else np.asarray(node_nbr)
    pj = node_pos.astype(np.float64)[nbr]                        # (N,k,3)
    c = rw * np.maximum(node_wa[:, None], node_wa[nbr])          # (N,k)
    Ji = c[..., None, None] * dW_dq(dqs[:, None, :], pj)         # (N,k,3,8)
    Jj = -c[..., None, None] * dW_dq(dqs[nbr], pj)
    f_reg = (c[..., None] * (W(dqs[:, None, :], pj) - W(dqs[nbr], pj))).reshape(-1)
    rr = (V + np.arange(n_nodes * k * 3)).reshape(n_nodes, k, 3)
    rows_i = np.broadcast_to(rr[..., None], Ji.shape).reshape(-1)
    cols_i = np.broadcast_to((np.arange(n_nodes)[:, None, None, None] * 8 + np.arange(8)), Ji.shape).reshape(-1)
    cols_j = np.broadcast_to((nbr[:, :, None, None] * 8 + np.arange(8)), Jj.shape).reshape(-1)
    rows_all = np.concatenate([rows, rows_i, rows_i])
    cols_all = np.concatenate([cols, cols_i, cols_j])
    vals_all = np.concatenate([vals, Ji.reshape(-1), Jj.reshape(-1)])
    J = csr_matrix((vals_all, (rows_all, cols_all)), shape=(V + 3 * k * n_nodes, 8 * n_nodes))   # duplicates (j == i) sum to 0
    return J, np.concatenate([r, f_reg])


def lw_jacobian(lw, vertices, normals, corr, vert_knn, node_pos, node_dq, node_w):
    """Dense (V,8) Jacobian of computef_lw w.r.t. the global rigid dq, and the residuals (smooth model)."""
    dqs = np.asarray(node_dq, dtype=np.float64)
    n_nodes = len(dqs)
    node_wa = np.broadcast_to(np.asarray(node_w, dtype=np.float64), (n_nodes,))
    p = np.asarray(vertices, dtype=np.float64); n = np.asarray(normals, dtype=np.float64)
    npk = node_pos.astype(np.float64)[vert_knn]
    d2 = ((p[:, None, :] - npk) ** 2).sum(-1)
    wts = np.exp(-d2 / (4.0 * node_wa[vert_knn] ** 2))
    b = (wts[..., None] * dqs[vert_knn]).sum(1)
    bh = b / np.linalg.norm(b, axis=1, keepdims=True)
    v1 = W(bh, p)
    rq = bh.copy(); rq[:, 4:] = 0
    n1 = W(rq, n)
    q = np.broadcast_to(np.asarray(lw, dtype=np.float64), (len(p), 8))
    v2 = W(q, v1)
    qr = q.copy(); qr[:, 4:] = 0
    n2 = W(qr, n1)
    r = np.einsum('ij,ij->i', n2, v2 - corr)
    J = np.einsum('vi,vic->vc', n2, dW_dq(q, v1)) + np.einsum('vi,vic->vc', v2 - corr, dW_dq(q, n1, rotation_only=True))
    return J, r


# ---------------------------------------------------------------------------------------------------
# Gauss-Newton step oracle (definition; see module docstring)
# ---------------------------------------------------------------------------------------------------
def huber_weights(f, f_scale=1.0, huber=True):
    if not huber:
        return np.ones_like(f)
    a = np.abs(f) / f_scale
    return np.where(a <= 1.0, 1.0, 1.0 / np.maximum(a, 1e-300))


def robust_cost(f, f_scale=1.0, huber=True):
    """0.5 * f_scale^2 * sum rho((f/f_scale)^2) with scipy's huber rho (z<=1: z, else 2 sqrt(z) - 1)."""
    if not huber:
        return 0.5 * float(f @ f)
    z = (f / f_scale) ** 2
    return 0.5 * f_scale ** 2 * float(np.where(z <= 1, z, 2 * np.sqrt(z) - 1).sum())


def normal_equations(J, f, f_scale=1.0, huber=True, dense=True):
    """H = J^T W J, g = J^T W f.  dense=False returns H as a scipy CSR (sorted indices, duplicates summed): at 5 k nodes the
    dense matrix is 40 k^2 doubles."""
    w = huber_weights(f, f_scale, huber)
    JW = J.multiply(w[:, None]).tocsr()
    H = (J.T.tocsr() @ JW).tocsr()
    H.sum_duplicates()
    H.sort_indices()
    g = np.asarray(J.T @ (w * f)).ravel()
    return (H.toarray() if dense else H), g


def gn_step(H, g, lam):
    """delta of (H + lam * mean(diag H) * I) delta = -g."""
    n = H.shape[0]
    mu = lam * np.trace(H) / n
    return np.linalg.solve(H + mu * np.eye(n), -g)


def _damping(H, lam):
    return lam * H.diagonal().sum() / H.shape[0]


def sparse_gn_step(H, g, lam):
    """gn_step for a scipy sparse H, by a sparse LU of H + mu I."""
    from scipy.sparse import identity
    from scipy.sparse.linalg import splu
    n = H.shape[0]
    A = (H + _damping(H, lam) * identity(n, format="csr")).tocsc()
    return splu(A).solve(-np.asarray(g, dtype=np.float64))


def pcg_block_jacobi(H, g, lam, tol, max_iter):
    """float64 restatement of the device solve dfb_gn_solve: (H + mu I) delta = -g with mu = lam * trace(H) / (8N), conjugate
    gradients preconditioned by the inverses of the damped 8x8 diagonal blocks, starting at delta = 0, stopping once
    (r, z) <= tol^2 (r0, z0) or after max_iter updates.  Returns (delta, number of updates applied) -- the count the device
    reports in workspace[6].  H: scipy sparse (8N, 8N) or dense."""
    from scipy.sparse import csr_matrix
    H = csr_matrix(H)
    n8 = H.shape[0]
    n = n8 // 8
    mu = _damping(H, lam)
    C = H.tocoo()
    on = (C.row // 8) == (C.col // 8)
    D = np.zeros((n, 8, 8))
    np.add.at(D, (C.row[on] // 8, C.row[on] % 8, C.col[on] % 8), C.data[on])
    Minv = np.linalg.inv(D + mu * np.eye(8))

    def prec(v):
        return np.einsum("iab,ib->ia", Minv, v.reshape(n, 8)).reshape(-1)

    delta = np.zeros(n8)
    r = -np.asarray(g, dtype=np.float64)
    z = prec(r)
    p = z.copy()
    rz = rz0 = float(r @ z)
    it = 0
    while it < max_iter and rz > tol * tol * rz0:
        q = H @ p + mu * p
        alpha = rz / float(p @ q)
        delta += alpha * p
        r -= alpha * q
        z = prec(r)
        rz_new = float(r @ z)
        p = z + (rz_new / rz) * p
        rz = rz_new
        it += 1
    return delta, it


def gauss_newton_loop(x0, vertices, normals, corr, vert_knn, node_pos, node_w, node_vertex_idx, lw, rw, max_iter=15, huber=True, f_scale=1.0,
                      lam0=1e-3, lam_min=1e-5, sparse=False):
    """The damped Gauss-Newton (Levenberg-Marquardt accept / reject) iteration of dynamicfusion_body_b200.gn.Problem.gauss_newton with
    every linear system solved densely in float64 -- the oracle of the PRODUCT's optimiser loop (the reference hands `computef` to
    scipy's TRF, whose trajectory is not a parity target: SURVEY 8a row a12).  Returns (x, cost0, cost, accepted).
    sparse=True: the same systems through scipy sparse matrices and a sparse LU (sparse_gn_step), for graphs of thousands of nodes."""
    x = np.asarray(x0, dtype=np.float64).copy()

    def assemble(xx):
        J, f = jacobian(xx, vertices, normals, corr, vert_knn, node_pos, node_w, node_vertex_idx, lw, rw)
        H, g = normal_equations(J, f, f_scale, huber, dense=not sparse)
        return H, g, robust_cost(f, f_scale, huber)

    H, g, cost = assemble(x)
    cost0, lam, accepted = cost, lam0, 0
    for _ in range(max_iter):
        x_new = x + (sparse_gn_step(H, g, lam) if sparse else gn_step(H, g, lam))
        H2, g2, cost_new = assemble(x_new)
        if np.isfinite(cost_new) and cost_new < cost:
            x, H, g, cost = x_new, H2, g2, cost_new
            lam = max(lam / 3.0, lam_min)
            accepted += 1
        else:
            lam *= 4.0
            if lam > 1e8:
                break
    return x, cost0, cost, accepted
