"""Generate tests/golden/reference_vectors.npz by EXECUTING THE UNMODIFIED REFERENCE (a checkout at oracle/_ref/,
see oracle/refload.py) on small seeded inputs:   python tests/golden/make_golden.py

The reference has no golden vectors of its own beyond three quaternion doctests (core/util.py:146-153,176-194,
258-260); these fixtures pin the oracle (oracle/*.py) to the reference's actual behaviour for every hot-path
function (SURVEY 8a rows a1-a11), including its dtype-dependent roundings (numpy 2.3.5 / scipy 1.18.1 here).
Inputs are stored alongside outputs so the tests need nothing but numpy.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import refload  # noqa: E402


def rand_dq(rng, n, scale_t=0.3, ang=0.2):
    ax = rng.normal(size=(n, 3)); ax /= np.linalg.norm(ax, axis=1, keepdims=True)
    a = rng.random(n) * ang
    q = np.concatenate([np.cos(a / 2)[:, None], np.sin(a / 2)[:, None] * ax], 1)
    t = rng.normal(size=(n, 3)) * scale_t
    qe = np.zeros((n, 4))
    for i in range(n):
        qe[i] = 0.5 * refload.load()[0].quaternion_multiply([0, t[i, 0], t[i, 1], t[i, 2]], q[i])
    return np.concatenate([q, qe], 1)


def main():
    util, Fusion, FusionDM = refload.load()
    rng = np.random.default_rng(20240)
    out = {}

    # --- a6: dual-quaternion algebra ------------------------------------------------------------------------
    out["qmul_kat"] = util.quaternion_multiply([4, 1, -2, 3], [8, -5, 6, 7])      # core/util.py:258-260 doctest
    for tag, dt1, dt2 in (("ff", np.float32, np.float32), ("df", np.float64, np.float32), ("fd", np.float32, np.float64), ("dd", np.float64, np.float64)):
        dq = rng.normal(size=(16, 8)).astype(dt1)
        p = (rng.normal(size=(16, 3)) * 20).astype(dt2)
        out["dqw_dq_" + tag] = dq; out["dqw_p_" + tag] = p
        out["dqw_out_" + tag] = np.array([util.dqb_warp(dq[i], p[i]) for i in range(16)])
        out["dqwn_out_" + tag] = np.array([util.dqb_warp_normal(dq[i], p[i]) for i in range(16)])

    # --- a7: interpolate_tsdf incl. the None cases printed by test.py:216-230 ---------------------------------
    vol = rng.normal(size=(6, 7, 8))
    pts = np.concatenate([rng.random((40, 3)) * np.array([5, 6, 7]), np.array([[0, 0, 0], [5, 6, 7], [5.0001, 1, 1], [-1e-9, 2, 2], [2, 6.5, 1], [1, 1, 7.2], [3, 2, 1]])])
    vals = [util.interpolate_tsdf(p, vol) for p in pts]
    out["interp_vol"] = vol; out["interp_pts"] = pts
    out["interp_valid"] = np.array([v is not None for v in vals])
    out["interp_val"] = np.array([0.0 if v is None else v for v in vals])

    # --- a1/a4/a5/a8: Fusion.updateTSDF, warp, dq_blend, KD-tree kNN ---------------------------------------------
    R, N, k = 10, 30, 4
    node_pos = (rng.random((N, 3)) * R).astype(np.float32)
    node_dq32 = rand_dq(rng, N).astype(np.float32)
    node_w = 5.0
    tsdf0 = rng.normal(size=(R, R, R)) * 0.3
    w0 = np.where(rng.random((R, R, R)) < 0.5, 0.0, np.floor(rng.random((R, R, R)) * 120))
    curr = rng.normal(size=(R + 2, R, R - 1)) * 0.5
    tdist = 0.6
    for tag, lw, dq in (("f32", np.array([1, 0, 0, 0, 0, 0.1, 0, 0], dtype=np.float32), node_dq32),
                        ("f64", rand_dq(rng, 1, 0.2, 0.1)[0], node_dq32)):
        nodes = [(i, node_pos[i], dq[i], node_w) for i in range(N)]
        f = refload.make_fusion(nodes, tsdf0.copy(), w0.copy(), tdist, k, lw)
        with refload.quiet():
            f.updateTSDF(curr)
        out["a1_lw_" + tag] = lw; out["a1_tsdf_" + tag] = f._tsdf; out["a1_w_" + tag] = f._tsdfw
    out.update(a1_node_pos=node_pos, a1_node_dq=node_dq32, a1_node_w=node_w, a1_tsdf0=tsdf0, a1_w0=w0, a1_curr=curr, a1_tdist=tdist, a1_k=k)
    f = refload.make_fusion([(i, node_pos[i], node_dq32[i], node_w) for i in range(N)], tsdf0, w0, tdist, k, np.array([1, 0, 0, 0, 0, 0.1, 0, 0], dtype=np.float32))
    grid = np.indices((R, R, R)).reshape(3, -1).T.astype(np.float32)
    out["knn_idx"] = np.array([f._kdtree.query(v, k=k + 1)[1][:-1] for v in grid])
    vv = (rng.random((24, 3)) * R).astype(np.float32); nn = rng.normal(size=(24, 3)).astype(np.float32)
    kk = np.array([f._kdtree.query(v, k=k)[1] for v in vv])
    wp = [f.warp(vv[i], [node_dq32[j] for j in kk[i]], kk[i], nn[i], m_lw=f._lw) for i in range(24)]
    out.update(warp_pts=vv, warp_nrm=nn, warp_knn=kk, warp_out_p=np.array([w[0] for w in wp]), warp_out_n=np.array([w[1] for w in wp]))
    out["blend_out"] = np.array([f.dq_blend(vv[i], [node_dq32[j] for j in kk[i]], kk[i]) for i in range(24)])
    out["warp_auto_p"] = np.array([f.warp(vv[i], m_lw=f._lw) for i in range(24)])   # warp() looking up its own k nearest (:503-506)

    # --- a2: FusionDM.fuseDepths, FusionDM.updateTSDF ---------------------------------------------------------------
    K = np.array([[60., 0, 31.5], [0, 60., 23.5], [0, 0, 1]])
    fdm = FusionDM(tdist, K, tsdf_res=R)
    H, Wd = 48, 64
    dm = -(rng.random((H, Wd)) * 8 + 14).astype(np.float32); dm[rng.random((H, Wd)) < 0.2] = 0
    ang = 0.2
    Rm = np.array([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]])
    lw34 = np.concatenate([Rm, np.array([[0.3], [-0.2], [18.]])], 1)
    center = np.array([0.1, 0.2, -0.3])
    with refload.quiet():
        rt, rw_ = fdm.fuseDepths(dm, lw34, tsdf0.copy(), w0.copy(), scale=1.3, center=center)
    out.update(a2_K=K, a2_dm=dm, a2_lw34=lw34, a2_center=center, a2_scale=1.3, a2_tsdf=rt, a2_w=rw_)
    fdm._tsdf = tsdf0.copy(); fdm._tsdfw = w0.copy(); fdm._lw = np.array([1, 0, 0, 0, 0, 0.1, 0, 0], dtype=np.float32)
    with refload.quiet():
        fdm.updateTSDF(curr)
    out.update(rigidvol_tsdf=fdm._tsdf, rigidvol_w=fdm._tsdfw)

    # --- a9/a11: computef / computef_lw ---------------------------------------------------------------------------------
    V = 60
    verts = (rng.random((V, 3)) * R).astype(np.float32); norms = rng.normal(size=(V, 3)).astype(np.float32)
    norms /= np.linalg.norm(norms, axis=1, keepdims=True)
    corr = verts.astype(np.float64) + rng.normal(size=(V, 3)) * 0.1
    vknn = np.array([f._kdtree.query(v, k=k)[1] for v in verts])
    nvi = rng.integers(0, V, size=N)
    nodes = [(int(nvi[i]), node_pos[i], node_dq32[i], node_w) for i in range(N)]
    for tag, lw in (("f32", np.array([1, 0, 0, 0, 0, 0.1, 0, 0], dtype=np.float32)), ("f64", out["a1_lw_f64"])):
        f = refload.make_fusion(nodes, None, None, tdist, k, lw, vertices=verts, normals=norms, neighbor_look_up=list(vknn), correspondences=corr)
        x32 = np.concatenate([n[2] for n in nodes])
        x64 = x32.astype(np.float64) + rng.normal(size=x32.shape) * 1e-3
        out["cf_x64_" + tag] = x64
        out["cf_f32_" + tag] = f.computef(x32, 0.2, 0.001, 0.5)
        out["cf_f64_" + tag] = f.computef(x64, 0.2, 0.001, 0.5)
        out["cflw_" + tag] = f.computef_lw(lw.astype(np.float64) + 1e-3, 0.2, 1)
    out.update(cf_verts=verts, cf_norms=norms, cf_corr=corr, cf_knn=vknn, cf_nvi=nvi)

    path = os.path.join(HERE, "reference_vectors.npz")
    np.savez_compressed(path, **{k_: np.asarray(v) for k_, v in out.items()})
    print("wrote", path, os.path.getsize(path), "bytes,", len(out), "arrays")


if __name__ == "__main__":
    main()
