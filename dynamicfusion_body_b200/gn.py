"""Host side of the warp-field Gauss-Newton path (Fusion.solve, core/fusion.py:327-491) over the C ABI.

The reference delegates to scipy.optimize.least_squares with a finite-difference Jacobian; here one iteration is
  dfb_gn_normal_eq  (analytic J -> block-sparse J^T W J, J^T W f, cost)        [optionally NCCL all-reduced]
  dfb_gn_solve      (damped block-Jacobi PCG in node space, x_new = x + delta)
under a Levenberg-Marquardt accept/reject loop driven from the host (one 16-byte cost read per iteration).
"""
import ctypes as C
import dataclasses

import numpy as np
import torch

from . import _capi
from .engine import _ptr, _stream, _to_dev, fill_lw


def dq_blend_points(wf, pts, idx):
    p = _to_dev(pts, torch.float32, wf.device).reshape(-1, 3)
    i = _to_dev(idx, torch.int32, wf.device).reshape(p.shape[0], -1)
    out = torch.empty((p.shape[0], 8), dtype=torch.float64, device=wf.device)
    s = wf.struct(None, None, k=i.shape[1])
    _capi.check(_capi.lib().dfb_dq_blend_points(_ptr(p), p.shape[0], _ptr(i), C.byref(s), _ptr(out), _stream()))
    return out.cpu().numpy()


def sparsity(vert_knn, node_vertex_idx, n_vert, n_nodes, n, m):
    """scipy lil_matrix (n, m) of ones: the correct Jacobian pattern of computef (see Fusion.computeSparsity)."""
    from scipy.sparse import lil_matrix
    vert_knn = np.asarray(vert_knn)
    k = vert_knn.shape[1]
    sp = lil_matrix((n, m), dtype=np.float32)
    for idx in range(n_vert):
        for loc in vert_knn[idx]:
            sp[idx, 8 * loc:8 * loc + 8] = 1
    nbr = vert_knn[np.asarray(node_vertex_idx)]
    for i in range(n_nodes):
        for jj in range(k):
            j = nbr[i, jj]
            for c in range(3):
                row = n_vert + (i * k + jj) * 3 + c
                sp[row, 8 * i:8 * i + 8] = 1
                sp[row, 8 * j:8 * j + 8] = 1
    return sp


@dataclasses.dataclass
class GNResult:
    x: torch.Tensor          # (8N,) float64 on the device
    cost0: float             # robust cost before
    cost: float              # robust cost after
    iterations: int
    accepted: int
    history: list            # per iteration dicts (cost, lambda, accepted, pcg_iterations)
    cost0_l2: float = 0.0    # 0.5 |f(x0)|^2 -- the reference's `cost_before` (core/fusion.py:376)


class Problem:
    """Device-resident least-squares problem: vertices, normals, correspondences, vertex->node kNN, nodes."""

    def __init__(self, wf, vertices, normals, corr, vert_knn, node_vertex_idx, shard=None, reg_owner=True, *, node_nbr=None):
        """node_nbr (optional, (N,k)): the regularisation neighbours of every node.  Default: vert_knn[node_vertex_idx]
        (core/fusion.py:477), which needs vert_knn to cover every vertex; a problem over a subset of the vertices (the data term
        of the associated ones only) passes the rows of the full vertex->node table here."""
        dev = wf.device
        self.wf = wf
        self.device = dev
        self.vertices = _to_dev(vertices, torch.float32, dev).reshape(-1, 3)
        self.normals = _to_dev(normals, torch.float32, dev).reshape(-1, 3)
        self.corr = _to_dev(corr, torch.float64, dev).reshape(-1, 3)
        self.vert_knn = _to_dev(vert_knn, torch.int32, dev).reshape(self.vertices.shape[0], -1)
        self.k = int(self.vert_knn.shape[1]) if self.vert_knn.numel() else wf.k
        self.n_vert = int(self.vertices.shape[0])
        self.n_nodes = wf.n_nodes
        nvi = np.asarray(node_vertex_idx, dtype=np.int64)
        if node_nbr is not None:
            self.node_nbr = _to_dev(node_nbr, torch.int32, dev).reshape(self.n_nodes, self.k)
        elif isinstance(vert_knn, torch.Tensor):
            self.node_nbr = self.vert_knn[torch.from_numpy(nvi).to(dev)].contiguous()
        else:
            self.node_nbr = _to_dev(np.asarray(vert_knn)[nvi], torch.int32, dev).reshape(self.n_nodes, self.k)
        # multi-GPU: every rank holds the (small) full problem so that the block pattern is identical everywhere, but
        # assembles only the data residuals of its vertex range `shard`; the regularisation rows belong to one rank.
        self.shard = (0, self.n_vert) if shard is None else (int(shard[0]), int(shard[1]))
        self.reg_owner = bool(reg_owner)
        self._pattern = None
        self._ws = None
        self._orders = {}

    def _order(self, v0, v1):
        """Processing order of the data residuals [v0, v1) for the assembly kernel: sorted by their (ascending) node tuple, so
        that residuals adding to the same 8x8 blocks follow each other (dfb_gn_problem.order).  Once per correspondence set; the
        sort is torch plumbing, not part of an iteration."""
        key = (v0, v1)
        o = self._orders.get(key)
        if o is None:
            rows = torch.sort(self.vert_knn[v0:v1].long(), dim=1).values
            o = torch.arange(v1 - v0, device=self.device)
            for c in range(rows.shape[1] - 1, -1, -1):          # lexicographic: stable sorts from the last column to the first
                o = o[torch.sort(rows[o, c], stable=True).indices]
            o = o.to(torch.int32).contiguous()
            self._orders[key] = o
        return o

    # -- struct ------------------------------------------------------------------------------------------
    def struct(self, lw, rw=1.0, huber=False, f_scale=1.0, sharded=False, ordered=False):
        p = _capi.GNProblem()
        v0, v1 = self.shard if sharded else (0, self.n_vert)
        if ordered and v1 > v0:
            p.order = self._order(v0, v1).data_ptr()
        p.n_vert = v1 - v0
        p.vertices = self.vertices.data_ptr() + 12 * v0; p.normals = self.normals.data_ptr() + 12 * v0
        p.corr = self.corr.data_ptr() + 24 * v0
        p.vert_knn = self.vert_knn.data_ptr() + 4 * self.k * v0
        if sharded and not self.reg_owner:
            rw = 0.0                                     # regularisation rows are assembled by their owner rank only
        p.n_nodes = self.n_nodes; p.k = self.k
        p.node_pos = self.wf.node_pos.data_ptr(); p.node_w = self.wf.node_w.data_ptr(); p.node_nbr = self.node_nbr.data_ptr()
        tmp = _capi.WarpField()
        fill_lw(tmp, lw if lw is not None else np.array([1.0, 0, 0, 0, 0, 0, 0, 0]))
        for i in range(8):
            p.lw[i] = tmp.lw[i]
        p.lw_is_f32 = tmp.lw_is_f32
        p.rw = float(rw); p.huber = 1 if huber else 0; p.f_scale = float(f_scale)
        return p

    # -- residual values (reference arithmetic) -------------------------------------------------------------
    def residuals(self, x, lw, rw):
        """Fusion.computef: (V + 3kN,) float64 CUDA tensor.  x: numpy (its dtype selects the reference's dtype flow) or CUDA f64."""
        is_f32 = 0
        if isinstance(x, np.ndarray):
            is_f32 = 1 if x.dtype == np.float32 else 0
        xd = _to_dev(x, torch.float64, self.device).reshape(-1)
        f = torch.empty(self.n_vert + 3 * self.k * self.n_nodes, dtype=torch.float64, device=self.device)
        p = self.struct(lw, rw)
        _capi.check(_capi.lib().dfb_gn_residuals(C.byref(p), _ptr(xd), is_f32, _ptr(f), _stream()))
        return f

    def residuals_lw(self, lw):
        """Fusion.computef_lw with the current node transforms."""
        lw = np.asarray(lw)
        f = torch.empty(self.n_vert, dtype=torch.float64, device=self.device)
        p = self.struct(lw)
        dq = self.wf.node_dq.double().contiguous()
        lwd = np.ascontiguousarray(lw, dtype=np.float64)
        _capi.check(_capi.lib().dfb_gn_residuals_lw(C.byref(p), _ptr(dq), 1, lwd.ctypes.data_as(_capi.c_f64p),
                                                    1 if lw.dtype == np.float32 else 0, _ptr(f), _stream()))
        return f

    # -- pattern ---------------------------------------------------------------------------------------------
    def pattern(self):
        """(row_ptr int32 [N+1], col_idx int32 [nnzb]) of the node co-occurrence graph; cached."""
        if self._pattern is None:
            n = self.n_nodes
            words = (n + 31) // 32
            bitmap = torch.empty(n * words, dtype=torch.int32, device=self.device)
            row_ptr = torch.empty(n + 1, dtype=torch.int32, device=self.device)
            p = self.struct(None)
            _capi.check(_capi.lib().dfb_gn_pattern_rows(C.byref(p), _ptr(bitmap), _ptr(row_ptr), _stream()))
            nnzb = int(row_ptr[-1].item())
            col_idx = torch.empty(nnzb, dtype=torch.int32, device=self.device)
            _capi.check(_capi.lib().dfb_gn_pattern_cols(n, _ptr(bitmap), _ptr(row_ptr), _ptr(col_idx), _stream()))
            self._pattern = (row_ptr, col_idx, nnzb)
        return self._pattern

    # -- normal equations ----------------------------------------------------------------------------------------
    def normal_equations(self, x, lw, rw, huber=False, f_scale=1.0, out=None):
        """(H [nnzb,8,8], g [8N], cost [2]) float64 CUDA tensors for x (CUDA f64 [8N])."""
        row_ptr, col_idx, nnzb = self.pattern()
        if out is None:
            # one flat buffer [H | g | cost]: the sharded solve sums it over ranks with ONE collective, in place (dist.py)
            nH, ng = nnzb * 64, 8 * self.n_nodes
            flat = torch.empty(nH + ng + 2, dtype=torch.float64, device=self.device)
            H, g, cost = flat[:nH].view(nnzb, 8, 8), flat[nH:nH + ng], flat[nH + ng:]
        else:
            H, g, cost = out
        p = self.struct(lw, rw, huber, f_scale, sharded=True, ordered=True)
        _capi.check(_capi.lib().dfb_gn_normal_eq(C.byref(p), _ptr(x), _ptr(row_ptr), _ptr(col_idx), nnzb, _ptr(H), _ptr(g), _ptr(cost), _stream()))
        return H, g, cost

    def solve_step(self, H, g, x, lam, max_iter=200, tol=1e-10):
        """x_new = x + delta with (H + lam*mean(diag H)*I) delta = -g.  Returns (x_new, delta, info tensor[8])."""
        row_ptr, col_idx, nnzb = self.pattern()
        n = self.n_nodes
        nws = int(_capi.lib().dfb_gn_solve_workspace_doubles(n))
        if self._ws is None or self._ws.numel() < nws:
            self._ws = torch.empty(nws, dtype=torch.float64, device=self.device)
        x_new = torch.empty_like(x)
        delta = torch.empty_like(x)
        _capi.check(_capi.lib().dfb_gn_solve(n, _ptr(row_ptr), _ptr(col_idx), _ptr(H), _ptr(g), float(lam), int(max_iter), float(tol),
                                             _ptr(x), _ptr(x_new), _ptr(delta), _ptr(self._ws), _stream()))
        return x_new, delta, self._ws[:8]

    def gauss_newton(self, x0, lw, rw, max_iter=15, huber=True, f_scale=1.0, lam0=1e-3, lam_min=1e-5, pcg_iters=400,
                     pcg_tol=1e-4, ftol=1e-9, verbose=False, allreduce=None, broadcast=None):
        """Damped Gauss-Newton (Levenberg-Marquardt accept/reject).  `allreduce(H, g, cost)` is called after every
        assembly when the residuals are sharded over ranks (dist.py); `broadcast(x)` (rank 0 -> all, in place) after every solve: the
        PCG's inner products are accumulated with atomics, so the replicated solves agree only to rounding -- broadcasting the
        iterate keeps every rank's transforms (and with them the sharded TSDF updates) bit-identical.  The linear systems are solved inexactly (PCG stops at a
        relative residual of `pcg_tol`): at 1 k nodes / 300 k residuals 1e-3 reaches the cost of a 1e-9 solve to 2e-6 relative
        in 2.0 instead of 3.2 ms per iteration (the damping shrinks as the iteration converges and the late, ill-conditioned
        systems need 350-400 PCG iterations to 1e-9 for no gain in cost); scripts/gn_forcing.py, DESIGN section 4."""
        x = _to_dev(x0, torch.float64, self.device).reshape(-1).clone()

        def assemble(xx):
            H, g, c = self.normal_equations(xx, lw, rw, huber, f_scale)
            if allreduce is not None:
                allreduce(H, g, c)
            return H, g, c

        H, g, c = assemble(x)
        c_host = c.tolist()
        cost, cost0_l2 = float(c_host[0]), float(c_host[1])
        cost0 = cost
        lam = lam0
        hist = []
        accepted = 0
        it = 0
        for it in range(1, max_iter + 1):
            x_new, delta, info = self.solve_step(H, g, x, lam, pcg_iters, pcg_tol)
            if broadcast is not None:
                broadcast(x_new)
            H2, g2, c2 = assemble(x_new)
            cost_new = float(c2[0].item())
            ok = np.isfinite(cost_new) and cost_new < cost
            # the PCG iteration count stays on the device until the loop is over (one host sync per iteration: the cost)
            hist.append({"cost": cost_new, "lambda": lam, "accepted": bool(ok), "pcg_iterations": info[6:7].clone()})
            if verbose:
                print("GN it %d: cost %.6e -> %.6e  lambda %.2e  %s  pcg %d" % (it, cost, cost_new, lam, "ok" if ok else "rejected", int(info[6].item())))
            if ok:
                rel = (cost - cost_new) / max(cost, 1e-300)
                x, H, g, cost = x_new, H2, g2, cost_new
                lam = max(lam / 3.0, lam_min)
                accepted += 1
                if rel < ftol:
                    break
            else:
                lam *= 4.0
                if lam > 1e8:
                    break
        if hist:
            its = torch.cat([h["pcg_iterations"] for h in hist]).cpu().numpy()
            for h, n_it in zip(hist, its):
                h["pcg_iterations"] = int(n_it)
        return GNResult(x=x, cost0=cost0, cost=cost, iterations=it, accepted=accepted, history=hist, cost0_l2=cost0_l2)

    # -- rigid fit of the global dq (core/fusion.py:350-362) -----------------------------------------------------------
    def lw_normal_equations(self, lw, huber=False, f_scale=1.0):
        lw = np.ascontiguousarray(lw, dtype=np.float64)
        H = torch.empty(64, dtype=torch.float64, device=self.device)
        g = torch.empty(8, dtype=torch.float64, device=self.device)
        c = torch.empty(2, dtype=torch.float64, device=self.device)
        p = self.struct(lw, 1.0, huber, f_scale)
        dq = self.wf.node_dq.double().contiguous()
        _capi.check(_capi.lib().dfb_gn_lw_normal_eq(C.byref(p), _ptr(dq), lw.ctypes.data_as(_capi.c_f64p), _ptr(H), _ptr(g), _ptr(c), _stream()))
        out = torch.cat([H, g, c]).cpu().numpy()
        return out[:64].reshape(8, 8), out[64:72], out[72:74]

    def solve_lw(self, lw0, max_iter=20, lam0=1e-6, verbose=False):
        """Damped GN on the 8 unknowns of the global rigid dq (plain L2 like the reference's default loss)."""
        lw = np.asarray(lw0, dtype=np.float64).copy()
        H, g, c = self.lw_normal_equations(lw)
        cost = c[1]
        lam = lam0
        for it in range(max_iter):
            mu = lam * np.trace(H) / 8.0
            try:
                d = np.linalg.solve(H + mu * np.eye(8), -g)
            except np.linalg.LinAlgError:
                lam *= 10
                continue
            H2, g2, c2 = self.lw_normal_equations(lw + d)
            if np.isfinite(c2[1]) and c2[1] < cost:
                rel = (cost - c2[1]) / max(cost, 1e-300)
                lw, H, g, cost = lw + d, H2, g2, c2[1]
                lam = max(lam / 3, 1e-15)
                if verbose:
                    print("lw it %d cost %.6e" % (it, cost))
                if rel < 1e-12:
                    break
            else:
                lam *= 10
                if lam > 1e10:
                    break
        return lw
