"""Device Gauss-Newton at the shapes where its code paths change (run with -m gpu): every PCG kernel and block-caching mode,
every normal_eq_data_kernel<K> instantiation, multi-batch warps, sharded and subset assembly, against the float64 oracle.

The solve tests call dfb_gn_solve directly on a BSR system built from the oracle's H, so they do not depend on the device
assembly.  The kernel that runs depends on the node count, the device (SM count, opt-in shared memory per block) and three
environment switches read once per process (DFB_PCG_GLOBAL, DFB_PCG_RPW, DFB_PCG_TWO_BARRIERS); `dispatch` restates that
choice from the device properties and every case asserts that it reached the path it is named for, so a device with other
limits fails loudly instead of testing something else.  Forced variants run in a child process (this file run as a script).

Bars.  Fixed iteration counts m (tol = 0) against oracle/gn.py:pcg_block_jacobi after m updates: <= 1e-9 relative for
m <= 10.  At m = 50 the bar is 1e-7: CG in floating point loses orthogonality at a rate set by the conditioning, the device
sums its inner products with atomics in no fixed order and the pipelined kernel carries extra recurrences, so two correct
implementations drift apart by rounding amplified over the iterations (DESIGN section 4: pipelined vs two-barrier 1e-7).
Some intermediate iterates are ill-conditioned in their own right: on the dense-row system at lam = 1e-3 the host PCG's own 50th
iterate moves by 9e-4 when g is perturbed by 1e-15 relative (10th: 4e-14, 80th: 3e-8), and every device variant lands ~8e-4 from it.
So each fixed-count bar is max(bar, 10 x that sensitivity), measured per case and printed ("sens"); m = 1 and 2, which pin the
preconditioner, the block layout and the first recurrences, stay at ~1e-9 wherever the iterate is well conditioned.
Converged (tol 1e-12): <= 1e-6 relative to the sparse-LU step and true residual |(H + mu I) d + g| / |g| <= 1e-9 -- when the
solve meets its tolerance.  The pipelined kernel does not always meet 1e-12: at lam = 1e-3 (cond ~1e6) its recurrences (u = M^-1 r,
w = A u, m, n carried next to r and x) accumulate rounding that the textbook iteration does not, (r,u) stalls above 1e-24 (r0,u0) and
the solve runs to its iteration cap.  A float64 numpy restatement of the same recurrences does the same on the CPU (N = 1184 and
2369, k = 4: 5000 updates, error 6e-8 / 3e-8, residual 2e-10 / 9e-11, where the textbook PCG stops after ~600 at 3e-11 / 6e-13), so
this is the attainable accuracy of the pipelined arrangement, not a defect of the kernel; the benchmarked tolerance 1e-4 is far
above it.  Such a capped solve is held to FLOOR_ERR / FLOOR_RES instead: on a B200 (1000 W) the capped S1 solves end at errors of
1.5e-7 ... 1.1e-6 and residuals of 8.9e-10 ... 2.2e-9 (N = 1184 ... 4736, k = 4 and 8); the bars leave a factor of ~10.
Assembly: every block (the mirrored lower ones too), g and both costs to 1e-10 relative."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu

MS = (1, 2, 10, 50)
CONV_ITERS = 5000
FLOOR_ERR, FLOOR_RES = 1e-5, 2e-8     # capped solves of the pipelined kernel (see above)
GD = 20          # blocks per gather round of pcg_pipelined_kernel (4 lane groups x GU = 5)
GR = 16          # the same for pcg_resident_kernel


# ---------------------------------------------------------------------------------------------------------------------
# problems
# ---------------------------------------------------------------------------------------------------------------------
def make_problem(n_nodes, k, seed=0, pts_per_node=12, pool=None, noise=0.05):
    """A least-squares problem over exactly `n_nodes` distinct vertices of the body mesh (64^3 units) as nodes, with points
    sampled near the mesh and their k nearest node ids (or k ids drawn from their `pool` nearest nodes: denser rows)."""
    from scipy.spatial import cKDTree
    from dynamicfusion_body_b200 import synth
    rng = np.random.default_rng(seed)
    v, nrm, _ = synth.load_body_mesh()
    v = v.astype(np.float64)
    node_idx = np.sort(rng.choice(len(v), n_nodes, replace=False))
    node_pos = v[node_idx].astype(np.float32)
    k = min(k, n_nodes)
    n_pts = max(pts_per_node * n_nodes, 64)
    src = rng.integers(0, len(v), n_pts)
    pts = (v[src] + rng.normal(size=(n_pts, 3)) * 0.3).astype(np.float32)
    norms = nrm[src].astype(np.float32)
    tree = cKDTree(node_pos.astype(np.float64))
    if pool is None:
        _, knn = tree.query(pts.astype(np.float64), k=k)
        knn = np.asarray(knn).reshape(n_pts, k)
    else:
        _, cand = tree.query(pts.astype(np.float64), k=min(pool, n_nodes))
        pick = np.argsort(rng.random(cand.shape), axis=1)[:, :k]
        knn = np.take_along_axis(cand, pick, axis=1)
    knn = knn.astype(np.int64)
    # node support radius: twice the mean distance to the nearest other node, so that the kNN weights are not negligible
    spacing = float(np.mean(tree.query(node_pos.astype(np.float64), k=2)[0][:, 1])) if n_nodes > 1 else 1.0
    node_w = np.float32(2.0 * spacing if pool is None else 6.0 * spacing)
    node_dq = synth.smooth_warp_field(node_pos, rng, 0.3, extent=64.0)
    lw = np.array([1, 0, 0, 0, 0, 0.05, -0.02, 0.01], np.float64)
    corr = synth.blend_warp(pts, node_pos, node_dq, np.full(n_nodes, node_w), knn, lw=lw) + rng.normal(size=(n_pts, 3)) * noise
    _, nvi = cKDTree(pts.astype(np.float64)).query(node_pos.astype(np.float64))
    x = node_dq.reshape(-1).astype(np.float64) + rng.normal(size=8 * n_nodes) * 2e-3
    return dict(verts=pts, norms=norms, corr=corr, knn=knn, nvi=nvi.astype(np.int64), node_pos=node_pos, nw=float(node_w),
                node_dq=node_dq, lw=lw, x=x, k=k, n=n_nodes)


def oracle_args(p, sl=slice(None)):
    return (p["verts"][sl], p["norms"][sl], p["corr"][sl], p["knn"][sl], p["node_pos"], p["nw"], p["nvi"], p["lw"])


def oracle_system(p, rw=0.05, huber=True, f_scale=1.0):
    from oracle import gn as ogn
    J, f = ogn.jacobian(p["x"], *oracle_args(p), rw)
    H, g = ogn.normal_equations(J, f, f_scale, huber, dense=False)
    return H, g


def to_bsr(H):
    """(row_ptr, col_idx, blocks [nnzb,8,8]) of a CSR H: ascending columns and every diagonal block present (dfb_gn_solve's
    contract, include/dfb.h)."""
    B = H.tobsr(blocksize=(8, 8))
    B.sum_duplicates()
    B.sort_indices()
    rp, ci = B.indptr.astype(np.int32), B.indices.astype(np.int32)
    n = len(rp) - 1
    for i in range(n):
        assert i in ci[rp[i]:rp[i + 1]], "row %d has no diagonal block" % i
    return rp, ci, np.ascontiguousarray(B.data, dtype=np.float64)


# ---------------------------------------------------------------------------------------------------------------------
# dispatch arithmetic of dfb_gn_solve (csrc/gn.cu), restated from the device properties
# ---------------------------------------------------------------------------------------------------------------------
def device_limits():
    import torch
    pr = torch.cuda.get_device_properties(0)
    return pr.multi_processor_count, pr.shared_memory_per_block_optin


def dispatch(row_ptr, sms, optin, rpw_min=1, force_global=False, two_barriers=False):
    rp = np.asarray(row_ptr, dtype=np.int64)
    n = len(rp) - 1
    warps = 8 * sms
    rpw = max(-(-n // warps), min(rpw_min, 4))
    row_len = int(np.diff(rp).max())
    if rpw > 4 or force_global:
        return dict(kernel="global", n=n, max_row_blocks=row_len)
    rows = 8 * rpw
    cap = (optin - 1024 - rows * 512) // 516
    starts = np.arange(0, n, rows)
    per_cta = rp[np.minimum(starts + rows, n)] - rp[starts]
    gather = GR if two_barriers else GD
    return dict(kernel="resident" if two_barriers else "pipelined", n=n, rpw=rpw, cap_blocks=int(cap), ctas=len(starts),
                max_cta_blocks=int(per_cta.max()), spilled_ctas=int((per_cta > cap).sum()), max_row_blocks=row_len,
                multi_round=row_len > gather)


# ---------------------------------------------------------------------------------------------------------------------
# the device solve
# ---------------------------------------------------------------------------------------------------------------------
def device_solve(rp, ci, Hb, g, lam, max_iter, tol):
    """dfb_gn_solve on the BSR system; returns (delta, workspace[:8])."""
    import torch
    from dynamicfusion_body_b200 import _capi
    from dynamicfusion_body_b200.engine import _ptr, _stream
    n = len(rp) - 1
    dev = torch.device("cuda")
    t = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (rp, ci, Hb, g)]
    lib = _capi.lib()
    ws = torch.empty(int(lib.dfb_gn_solve_workspace_doubles(n)), dtype=torch.float64, device=dev)
    x = torch.zeros(8 * n, dtype=torch.float64, device=dev)
    x_new, delta = torch.empty_like(x), torch.empty_like(x)
    _capi.check(lib.dfb_gn_solve(n, _ptr(t[0]), _ptr(t[1]), _ptr(t[2]), _ptr(t[3]), float(lam), int(max_iter), float(tol),
                                 _ptr(x), _ptr(x_new), _ptr(delta), _ptr(ws), _stream()))
    torch.cuda.synchronize()
    d = delta.cpu().numpy()
    assert np.array_equal(x_new.cpu().numpy(), d)
    return d, ws[:8].cpu().numpy()


def fixed_counts(n):
    """MS below the dimension 8N of the system (CG on an 8-dimensional system is done after 8 updates)."""
    return [m for m in MS if m < 8 * n]


def solve_runs(rp, ci, Hb, g, lam):
    """The device runs a case is judged on: fixed counts MS (tol 0), converged (tol 1e-12) and the benchmarked tol 1e-4."""
    out = {}
    for m in fixed_counts(len(rp) - 1):
        out["m%d" % m] = device_solve(rp, ci, Hb, g, lam, m, 0.0)
    out["tol12"] = device_solve(rp, ci, Hb, g, lam, CONV_ITERS, 1e-12)
    out["tol4"] = device_solve(rp, ci, Hb, g, lam, 400, 1e-4)
    return out


def check_runs(name, kernel, H, g, lam, runs, step=None):
    """Device runs against pcg_block_jacobi (fixed counts, tol 1e-4) and the sparse-LU step (converged); prints the errors."""
    from oracle import gn as ogn
    errs, sens = {}, {}
    g_ulp = g * (1 + 1e-15 * np.random.default_rng(0).standard_normal(len(g)))
    for m in fixed_counts(H.shape[0] // 8):
        d, ws = runs["m%d" % m]
        ref, it = ogn.pcg_block_jacobi(H, g, lam, 0.0, m)
        assert it == m and ws[6] == m, (name, m, ws[6])
        errs[m] = np.linalg.norm(d - ref) / np.linalg.norm(ref)
        # how far the host's own m-th iterate moves when g changes in its last bits (see the module docstring)
        sens[m] = np.linalg.norm(ogn.pcg_block_jacobi(H, g_ulp, lam, 0.0, m)[0] - ref) / np.linalg.norm(ref)
    mu = lam * H.diagonal().sum() / H.shape[0]
    d, ws = runs["tol12"]
    if step is None:
        step = ogn.sparse_gn_step(H, g, lam)
    e_conv = np.linalg.norm(d - step) / np.linalg.norm(step)
    res = np.linalg.norm(H @ d + mu * d + g) / np.linalg.norm(g)
    _, it4 = ogn.pcg_block_jacobi(H, g, lam, 1e-4, 400)
    d4, ws4 = runs["tol4"]
    print("  %s lam %.0e: rel err %s | tol1e-12: err %.2e residual %.2e (%d its) | tol1e-4: %d its, host %d"
          % (name, lam, " ".join("m=%d %.2e (sens %.1e)" % (m, errs[m], sens[m]) for m in errs), e_conv, res, int(ws[6]), int(ws4[6]),
             it4))
    for m in errs:
        assert errs[m] <= max(1e-9 if m <= 10 else 1e-7, 10 * sens[m]), (name, lam, m, errs[m], sens[m])
    if ws[6] < CONV_ITERS:
        assert e_conv <= 1e-6 and res <= 1e-9, (name, lam, e_conv, res)
    else:
        # the pipelined recurrences stalled at their attainable accuracy before (r,z) reached 1e-24 (r0,z0); see the docstring
        assert kernel == "pipelined", (name, lam, kernel, e_conv, res)
        assert e_conv <= FLOOR_ERR and res <= FLOOR_RES, (name, lam, e_conv, res)
    assert abs(int(ws4[6]) - it4) <= 2, (name, lam, ws4[6], it4)


# ---------------------------------------------------------------------------------------------------------------------
# S1: natural dispatch at node counts picked from the SM count
# ---------------------------------------------------------------------------------------------------------------------
def _s1_counts(sms, k):
    w = 8 * sms
    return [1, k, w, w + 1, 2 * w + 1, 3 * w + 1, 4 * w, 4 * w + 1]


_SYSTEMS = {}


def _system(n, k):
    key = (n, k)
    if key not in _SYSTEMS:
        p = make_problem(n, k, seed=n + 17 * k, pts_per_node=6)
        H, g = oracle_system(p)
        _SYSTEMS[key] = (p, H, g, to_bsr(H))
    return _SYSTEMS[key]


@pytest.mark.parametrize("k", [4, 8])
def test_s1_natural_dispatch(k):
    sms, optin = device_limits()
    w = 8 * sms
    seen = set()
    for n in _s1_counts(sms, k):
        p, H, g, (rp, ci, Hb) = _system(n, k)
        info = dispatch(rp, sms, optin)
        print("N %d k %d: %s" % (n, p["k"], json.dumps(info)))
        if n > 4 * w:
            assert info["kernel"] == "global"
        else:
            assert info["kernel"] == "pipelined" and info["rpw"] == -(-n // w)
        seen.add((info["kernel"], info.get("rpw"), info.get("spilled_ctas", 0) > 0, info.get("multi_round", False)))
        for lam in (1e-1, 1e-3):
            runs = solve_runs(rp, ci, Hb, g, lam)
            check_runs("S1 N=%d k=%d" % (n, p["k"]), info["kernel"], H, g, lam, runs, step=None if n <= 2 * w + 1 else step_pcg(H, g, lam))
    # every resident rpw, the global kernel, and (k = 8: 30 blocks per row) spilled CTAs and multi-round rows
    kinds = {(s[0], s[1]) for s in seen}
    assert {("pipelined", r) for r in (1, 2, 3, 4)} <= kinds and ("global", None) in kinds, seen
    if k == 8:
        assert any(s[2] for s in seen) and any(s[3] for s in seen), seen


def step_pcg(H, g, lam):
    """The converged step of a system too large for a quick sparse LU: the host PCG driven to 1e-14 (pinned against the LU
    step by tests/test_oracle_gn_sparse.py)."""
    from oracle import gn as ogn
    d, _ = ogn.pcg_block_jacobi(H, g, lam, 1e-14, 20000)
    return d


# ---------------------------------------------------------------------------------------------------------------------
# S2: forced kernel variants (environment switches), in a child process
# ---------------------------------------------------------------------------------------------------------------------
VARIANTS = ([("two_barriers_rpw%d" % r, {"DFB_PCG_TWO_BARRIERS": "1", "DFB_PCG_RPW": str(r)}) for r in (1, 2, 3, 4)]
            + [("pipelined_rpw%d" % r, {"DFB_PCG_RPW": str(r)}) for r in (2, 3, 4)]
            + [("global", {"DFB_PCG_GLOBAL": "1"})])


@pytest.fixture(scope="module")
def s2_systems(tmp_path_factory):
    """A sparse system (every block cached) and a dense-row one (k = 8 ids drawn from each point's 40 nearest nodes: some CTA
    spills even at one row per warp, rows run past one gather round)."""
    out = []
    d = tmp_path_factory.mktemp("s2")
    for name, kw in (("sparse", dict(n_nodes=300, k=4)), ("dense_rows", dict(n_nodes=400, k=8, pool=40, pts_per_node=20))):
        p = make_problem(**kw, seed=7)
        H, g = oracle_system(p)
        rp, ci, Hb = to_bsr(H)
        path = str(d / ("%s.npz" % name))
        np.savez(path, rp=rp, ci=ci, Hb=Hb, g=g)
        out.append((name, H, g, rp, path))
    return out


@pytest.mark.parametrize("variant", [v[0] for v in VARIANTS])
def test_s2_forced_variants(variant, s2_systems, tmp_path):
    env_add = dict(VARIANTS)[variant]
    sms, optin = device_limits()
    env = {k: v for k, v in os.environ.items() if not k.startswith("DFB_PCG_")}
    env.update(env_add)
    env["PYTHONPATH"] = ROOT + os.pathsep + env.get("PYTHONPATH", "")
    for name, H, g, rp, path in s2_systems:
        info = dispatch(rp, sms, optin, rpw_min=int(env_add.get("DFB_PCG_RPW", 1)), force_global="DFB_PCG_GLOBAL" in env_add,
                        two_barriers="DFB_PCG_TWO_BARRIERS" in env_add)
        print("%s / %s: %s" % (variant, name, json.dumps(info)))
        if variant == "global":
            assert info["kernel"] == "global"
        else:
            assert info["kernel"] == ("resident" if "DFB_PCG_TWO_BARRIERS" in env_add else "pipelined")
            assert info["rpw"] == int(env_add["DFB_PCG_RPW"])
            if name == "sparse":
                assert info["spilled_ctas"] == 0
            elif info["rpw"] == 1:
                assert info["spilled_ctas"] > 0 and info["multi_round"], info
        for lam in (1e-1, 1e-3):
            res = str(tmp_path / ("%s_%g.npz" % (name, lam)))
            subprocess.run([sys.executable, os.path.abspath(__file__), path, str(lam), res], env=env, cwd=ROOT, check=True, timeout=600)
            r = np.load(res)
            runs = {key: (r[key + "_d"], r[key + "_ws"]) for key in ["m%d" % m for m in fixed_counts(len(rp) - 1)] + ["tol12", "tol4"]}
            check_runs("S2 %s %s" % (variant, name), info["kernel"], H, g, lam, runs)


# ---------------------------------------------------------------------------------------------------------------------
# assembly: device Problem.normal_equations against the oracle
# ---------------------------------------------------------------------------------------------------------------------
def device_problem(p, sl=slice(None), **kw):
    from dynamicfusion_body_b200 import engine, gn
    wf = engine.DeviceWarpField(p["k"])
    wf.set_nodes(p["node_pos"], p["node_dq"], np.float32(p["nw"]))
    return gn.Problem(wf, p["verts"][sl], p["norms"][sl], p["corr"][sl], p["knn"][sl], p["nvi"], **kw)


def block_pattern(knn, nbr, n):
    """Node pairs (a, b) of the block pattern of J^T J (structural), plus every diagonal block."""
    from scipy.sparse import csr_matrix
    V, k = knn.shape
    rows = np.concatenate([np.repeat(np.arange(V), k), V + np.repeat(np.arange(n * k), 2)])
    cols = np.concatenate([knn.reshape(-1), np.stack([np.repeat(np.arange(n), k), nbr.reshape(-1)], 1).reshape(-1)])
    B = csr_matrix((np.ones(len(rows)), (rows, cols)), shape=(V + n * k, n))
    P = (B.T @ B).tocoo()
    return set(zip(P.row.tolist(), P.col.tolist())) | {(i, i) for i in range(n)}


def check_assembly(name, prob, x, lw, rw, huber, f_scale, Ho, go, fo, nbr, knn, sharded_cost=True):
    """Device H (all blocks), g and both costs against the oracle (Ho CSR, go, residual vector fo); pattern as exact sets."""
    import torch
    from oracle import gn as ogn
    H, g, cost = prob.normal_equations(torch.from_numpy(x).cuda(), lw, rw, huber=huber, f_scale=f_scale)
    rp, ci, nnzb = prob.pattern()
    rp, ci, Hb = rp.cpu().numpy(), ci.cpu().numpy(), H.cpu().numpy()
    n = len(rp) - 1
    rows = np.repeat(np.arange(n), np.diff(rp))
    assert all((np.diff(ci[rp[i]:rp[i + 1]]) > 0).all() for i in range(n))
    pat = set(zip(rows.tolist(), ci.tolist()))
    assert pat == block_pattern(knn, nbr, n), name
    Bo = Ho.tobsr(blocksize=(8, 8))
    Bo.sum_duplicates()
    ref = np.zeros_like(Hb)
    brow = np.repeat(np.arange(n), np.diff(Bo.indptr))
    slot = {(a, b): s for s, (a, b) in enumerate(zip(rows.tolist(), ci.tolist()))}
    for s, (a, b) in enumerate(zip(brow.tolist(), Bo.indices.tolist())):
        ref[slot[(a, b)]] += Bo.data[s]
    scale = np.abs(ref).max()
    e_H = np.abs(Hb - ref).max() / scale
    e_g = np.abs(g.cpu().numpy() - go).max() / np.abs(go).max()
    c = cost.cpu().numpy()
    c_rob, c_l2 = ogn.robust_cost(fo, f_scale, huber), 0.5 * float(fo @ fo)
    e_c = max(abs(c[0] - c_rob) / c_rob, abs(c[1] - c_l2) / c_l2)
    print("  %s: %d blocks, err H %.2e g %.2e cost %.2e" % (name, nnzb, e_H, e_g, e_c))
    assert e_H <= 1e-10 and e_g <= 1e-10 and e_c <= 1e-10, name
    return Hb, g.cpu().numpy(), c


def _oracle_neq(p, sl=slice(None), rw=0.3, huber=True, f_scale=0.5, node_nbr=None, lw=None):
    from oracle import gn as ogn
    a = list(oracle_args(p, sl))
    if lw is not None:
        a[-1] = lw
    J, f = ogn.jacobian(p["x"], *a, rw, node_nbr=node_nbr)
    H, g = ogn.normal_equations(J, f, f_scale, huber, dense=False)
    return H, g, f


@pytest.mark.parametrize("k", range(1, 9))
def test_a1_assembly_every_k(k):
    from oracle import gn as ogn
    p = make_problem(90, k, seed=100 + k, pts_per_node=30, noise=0.3)
    nbr = ogn.reg_neighbours(p["knn"], p["nvi"])
    for lw in (p["lw"], p["lw"].astype(np.float32)):
        for huber in (False, True):
            prob = device_problem(p)
            Ho, go, fo = _oracle_neq(p, huber=huber, lw=lw)
            check_assembly("A1 k=%d huber=%s lw=%s" % (k, huber, lw.dtype), prob, p["x"], lw, 0.3, huber, 0.5, Ho, go, fo, nbr, p["knn"])


@pytest.mark.parametrize("n_vert", [400_003, 700_011])
def test_a2_multi_batch_warps(n_vert):
    """More residuals than 1184 warps x 256: each warp walks 2 (3) consecutive batches and carries tuple runs across the batch
    ends; V is not a multiple of 32.  Sorted order and natural order."""
    import torch
    from oracle import gn as ogn
    sms, _ = device_limits()
    nblk = min(-(-n_vert // 256), sms * 8)
    per_warp = -(-(-(-n_vert // 32)) // (nblk * 8))
    print("A2 V=%d: %d batches per warp" % (n_vert, per_warp))
    assert per_warp >= 2
    p = make_problem(1000, 4, seed=11, pts_per_node=1)
    rng = np.random.default_rng(12)
    src = rng.integers(0, len(p["verts"]), n_vert)
    for key in ("verts", "norms", "knn"):
        p[key] = p[key][src]
    p["corr"] = p["corr"][src] + rng.normal(size=(n_vert, 3)) * 0.05
    nbr = ogn.reg_neighbours(p["knn"], p["nvi"])
    Ho, go, fo = _oracle_neq(p)
    prob = device_problem(p)
    H1, g1, c1 = check_assembly("A2 V=%d sorted" % n_vert, prob, p["x"], p["lw"], 0.3, True, 0.5, Ho, go, fo, nbr, p["knn"])
    prob._orders[(0, n_vert)] = torch.arange(n_vert, dtype=torch.int32, device="cuda")
    check_assembly("A2 V=%d natural" % n_vert, prob, p["x"], p["lw"], 0.3, True, 0.5, Ho, go, fo, nbr, p["knn"])


def test_a3_repeated_node_id():
    """A residual whose kNN row lists a node twice: the diagonal block gets (w_a + w_b)^2, the 2.0 branch of the kernel."""
    from oracle import gn as ogn
    for k in (2, 4, 8):
        p = make_problem(80, k, seed=30 + k, pts_per_node=20)
        nbr = ogn.reg_neighbours(p["knn"], p["nvi"])
        knn = p["knn"].copy()
        knn[::7, 1] = knn[::7, 0]
        knn[::11, -1] = knn[::11, 0]
        p["knn"] = knn
        Ho, go, fo = _oracle_neq(p, node_nbr=nbr)
        prob = device_problem(p, node_nbr=nbr)
        check_assembly("A3 k=%d" % k, prob, p["x"], p["lw"], 0.3, True, 0.5, Ho, go, fo, nbr, knn)


@pytest.mark.parametrize("n_shards", [2, 3, 4])
def test_a4_sharded_assembly(n_shards):
    """Shards of [0, V) (regularisation on the first only), each with its own sorted order: every shard matches the oracle
    on its slice, and the shards sum to the full system."""
    import torch
    from oracle import gn as ogn
    p = make_problem(200, 4, seed=40, pts_per_node=25, noise=0.2)
    nbr = ogn.reg_neighbours(p["knn"], p["nvi"])
    V = len(p["verts"])
    cuts = np.linspace(0, V, n_shards + 1).astype(int)
    cuts[1:-1] += 13
    full = device_problem(p)
    Hf, gf, cf = full.normal_equations(torch.from_numpy(p["x"]).cuda(), p["lw"], 0.3, huber=True, f_scale=0.5)
    Hs = torch.zeros_like(Hf); gs = torch.zeros_like(gf); cs = torch.zeros_like(cf)
    for s in range(n_shards):
        v0, v1 = int(cuts[s]), int(cuts[s + 1])
        prob = device_problem(p, shard=(v0, v1), reg_owner=(s == 0), node_nbr=nbr)
        rw = 0.3 if s == 0 else 0.0
        Ho, go, fo = _oracle_neq(p, slice(v0, v1), rw=rw, node_nbr=nbr)
        if s > 0:
            fo = fo[:v1 - v0]      # the regularisation rows (all zero at rw = 0) belong to the first shard
        # the pattern covers every vertex: compare the shard's blocks against the oracle on the full pattern
        H, g, c = prob.normal_equations(torch.from_numpy(p["x"]).cuda(), p["lw"], 0.3, huber=True, f_scale=0.5)
        rp, ci, _ = prob.pattern()
        rp, ci = rp.cpu().numpy(), ci.cpu().numpy()
        rows = np.repeat(np.arange(len(rp) - 1), np.diff(rp))
        Hd = np.zeros(Ho.shape)
        Hb = H.cpu().numpy()
        for t in range(len(ci)):
            Hd[8 * rows[t]:8 * rows[t] + 8, 8 * ci[t]:8 * ci[t] + 8] = Hb[t]
        Hod = Ho.toarray()
        assert np.abs(Hd - Hod).max() <= 1e-10 * np.abs(Hod).max()
        assert np.abs(g.cpu().numpy() - go).max() <= 1e-10 * np.abs(go).max()
        assert abs(c[0].item() - ogn.robust_cost(fo, 0.5, True)) <= 1e-10 * abs(c[0].item())
        Hs += H; gs += g; cs += c
    e = (Hs - Hf).abs().max().item() / Hf.abs().max().item()
    print("A4 %d shards: sum vs full %.2e" % (n_shards, e))
    assert e <= 1e-12
    assert (gs - gf).abs().max().item() <= 1e-12 * gf.abs().max().item()
    assert (cs - cf).abs().max().item() <= 1e-12 * cf.abs().max().item()


def test_a5_subset_with_node_nbr():
    """The data term of a subset of the vertices, regularisation neighbours from the full vertex->node table (projective path)."""
    from oracle import gn as ogn
    p = make_problem(150, 4, seed=50, pts_per_node=20, noise=0.2)
    nbr = ogn.reg_neighbours(p["knn"], p["nvi"])
    sel = np.sort(np.random.default_rng(51).choice(len(p["verts"]), len(p["verts"]) // 3, replace=False))
    Ho, go, fo = _oracle_neq(p, sel, node_nbr=nbr)
    prob = device_problem(p, sel, node_nbr=nbr)
    check_assembly("A5 subset", prob, p["x"], p["lw"], 0.3, True, 0.5, Ho, go, fo, nbr, p["knn"][sel])


def test_a6_pattern_beyond_one_scan_chunk():
    """N > 1024: pattern_scan_kernel carries its sum across 1024-row chunks; row_ptr and col_idx equal the oracle pattern."""
    from oracle import gn as ogn
    for n in (1025, 2500):
        p = make_problem(n, 4, seed=60, pts_per_node=4)
        nbr = ogn.reg_neighbours(p["knn"], p["nvi"])
        prob = device_problem(p)
        rp, ci, nnzb = prob.pattern()
        pat = sorted(block_pattern(p["knn"], nbr, n))
        rows = np.array([a for a, _ in pat])
        assert np.array_equal(rp.cpu().numpy(), np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=n))]))
        assert np.array_equal(ci.cpu().numpy(), np.array([b for _, b in pat]))
        print("A6 N=%d: %d blocks" % (n, nnzb))


# ---------------------------------------------------------------------------------------------------------------------
# the loop at k = 8: two block rows per warp, spilled CTAs
# ---------------------------------------------------------------------------------------------------------------------
def test_loop_k8_spilled_matches_oracle_loop():
    import torch
    from oracle import gn as ogn
    sms, optin = device_limits()
    n = 2 * 8 * sms - 800             # two rows per warp on 148 SMs (1568 nodes)
    p = make_problem(n, 8, seed=70, pts_per_node=40, noise=0.02)
    prob = device_problem(p)
    rp, _, _ = prob.pattern()
    info = dispatch(rp.cpu().numpy(), sms, optin)
    print("loop: %s" % json.dumps(info))
    assert info["kernel"] == "pipelined" and info["rpw"] == 2 and info["spilled_ctas"] > 0
    xo, c0o, co, acc_o = ogn.gauss_newton_loop(p["x"], *oracle_args(p), 0.05, max_iter=5, huber=True, sparse=True)
    res = prob.gauss_newton(torch.from_numpy(p["x"]).cuda(), p["lw"], 0.05, max_iter=5, huber=True, ftol=0.0)
    x = res.x.cpu().numpy()
    rel = np.linalg.norm(x - xo) / np.linalg.norm(xo)
    print("loop: rel err of x %.3e, accepted %d vs %d, pcg its %s" % (rel, res.accepted, acc_o, [h["pcg_iterations"] for h in res.history]))
    assert res.accepted == acc_o
    assert rel <= 1e-4


# ---------------------------------------------------------------------------------------------------------------------
# child process: python test_gpu_gn_shapes.py SYSTEM.npz LAMBDA OUT.npz  (environment selects the kernel)
# ---------------------------------------------------------------------------------------------------------------------
def _child(path, lam, out):
    s = np.load(path)
    runs = solve_runs(s["rp"], s["ci"], s["Hb"], s["g"], lam)
    np.savez(out, **{k + "_d": v[0] for k, v in runs.items()}, **{k + "_ws": v[1] for k, v in runs.items()})


if __name__ == "__main__":
    _child(sys.argv[1], float(sys.argv[2]), sys.argv[3])
