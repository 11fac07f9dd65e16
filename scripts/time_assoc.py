"""Projective data association vs the closest-point path on one GPU: association time, the Gauss-Newton solve each
correspondence set leads to, and the coverage of the default gates.  Writes one JSON file (default profiles/r3_assoc.json)
and prints the card name and power limit (queried, never set) beside the numbers.

Workload: the gn_depth_frame one of bench.py (256^3 scene, focal 775, ~1k nodes, k=4, one 640x480 frame): canonical samples
= the back-projected valid pixels of a depth frame rendered from the canonical mesh; closest-point live points = the
back-projected pixels of the live frame.  The association timings are repeated on 300 k area-weighted canonical samples."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from scipy.spatial import cKDTree

from dynamicfusion_body_b200 import engine, synth
from dynamicfusion_body_b200.fusion import Fusion


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:                                  # the number is still reported, marked as lacking the limit
        q = "unavailable (%s)" % e
    return {"name": name, "power_limit_and_max_sm_clock": q}


def event_ms(fn, reps=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "r3_assoc.json"))
    ap.add_argument("--gn-iters", type=int, default=15)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(0)
    sc = synth.make_scene(res=256, k=4, n_nodes=1000, seed=0, background=False, focal=775.0)
    K, Kinv = sc.K, sc.Kinv
    E = np.stack([synth.dq_apply(sc.lw[None, :].astype(np.float64), e[None, :])[0] for e in np.eye(3)], 1)
    t = synth.dq_apply(sc.lw[None, :].astype(np.float64), np.zeros((1, 3)))[0]
    Rm = E - t[:, None]

    def backproject(dm):
        v, u = np.nonzero(dm < 0)
        z = -dm[v, u].astype(np.float64)
        return (Kinv @ np.stack([u * z, v * z, z])).T

    canon_cam = backproject(synth.render_depth(sc.vertices.astype(np.float64) @ Rm.T + t, sc.faces, K, sc.rows, sc.cols))
    canon = ((canon_cam - t) @ Rm).astype(np.float32)
    _, nn = cKDTree(sc.vertices.astype(np.float64)).query(canon.astype(np.float64))
    normals = -sc.normals[nn]                               # the fixture's normals point into the body: turned outward
    live = backproject(sc.depths[0]).astype(np.float32)
    rng = np.random.default_rng(0)
    x0 = sc.node_dq.reshape(-1).astype(np.float64) + rng.normal(size=8 * sc.n_nodes) * 2e-3
    _, nvi = cKDTree(canon.astype(np.float64)).query(sc.node_pos.astype(np.float64))
    nodes = [(int(nvi[i]),) + n[1:] for i, n in enumerate(sc.nodes_as_reference_tuples())]

    def make_fusion():
        f = Fusion(sc.tdist, knn=4, device=dev, use_cnn=False, write_warpfield=False)
        f.InitializeCanonicalSpace(tsdf_shape=(8, 8, 8), K=K, vertices=canon, normals=normals, nodes=nodes)
        f._lw = sc.lw
        f.set_node_dqs(x0.reshape(-1, 8).astype(np.float32))
        return f

    out = {"card": card(), "workload": {"scene": "256^3, focal 775, one 640x480 frame, %d nodes, k=4" % sc.n_nodes,
                                        "canonical_pixels": int(len(canon)), "live_pixels": int(len(live)),
                                        "default_gates": {"max_distance": sc.tdist, "max_distance_is": "the truncation distance",
                                                          "min_normal_dot": 0.5}}}
    depth = torch.from_numpy(sc.depths).to(dev)
    views = engine.make_views(depth, K, Kinv, None)
    live_d = torch.from_numpy(live).to(dev)
    wf = make_fusion()._wf

    # ---- association time ----------------------------------------------------------------------------------------------
    def timings(verts, norms, loc, label):
        v = torch.from_numpy(np.ascontiguousarray(verts)).to(dev)
        n = torch.from_numpy(np.ascontiguousarray(norms)).to(dev)
        lc = torch.from_numpy(np.ascontiguousarray(loc, dtype=np.int32)).to(dev)

        def warp():
            return engine.warp_points(wf, sc.lw, v, n, idx=lc, k=4)
        wv, wn = warp()

        def proj():
            a, b = warp()
            return engine.corr_projective(a, b, views, sc.tdist, 0.5)

        def clpts():
            a, b = warp()
            nn_ = engine.PointGrid(live_d, device=dev).knn(a, 4)
            return engine.corr_select(a, b, live_d, nn_)
        r = {"points": int(len(verts)), "warp_ms": event_ms(warp),
             "corr_projective_only_ms": event_ms(lambda: engine.corr_projective(wv, wn, views, sc.tdist, 0.5)),
             "projective_warp_plus_assoc_ms": event_ms(proj), "closest_point_warp_grid_knn_select_ms": event_ms(clpts)}
        view = engine.corr_projective(wv, wn, views, sc.tdist, 0.5)[0]
        r["associated_fraction_default_gates"] = float((view >= 0).float().mean().item())
        out["association_" + label] = r

    timings(canon, normals, make_fusion()._neighbor_look_up, "gn_depth_frame")
    pd = synth.make_gn_problem(sc, 300000, seed=0)
    timings(pd.vertices, -pd.normals, pd.vert_knn, "300k_samples")

    # ---- Gauss-Newton with each correspondence set ------------------------------------------------------------------------
    def solve(fus, label):
        prob = fus._problem()
        x = torch.from_numpy(x0).to(dev)
        prob.pattern()
        prob.gauss_newton(x, sc.lw, 0.05, max_iter=2, huber=True)       # warm-up
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        res = prob.gauss_newton(x, sc.lw, 0.05, max_iter=args.gn_iters, huber=True, ftol=0.0)
        b.record()
        torch.cuda.synchronize()
        pcg = [h["pcg_iterations"] for h in res.history]
        out["gn_" + label] = {"data_residuals": prob.n_vert, "iterations": res.iterations, "accepted": res.accepted,
                              "rejected": res.iterations - res.accepted, "pcg_iterations": pcg,
                              "pcg_iterations_mean": float(np.mean(pcg)) if pcg else 0.0, "pcg_at_cap_400": int(sum(p >= 400 for p in pcg)),
                              "cost0": res.cost0, "final_cost": res.cost, "ms_per_iteration": a.elapsed_time(b) / max(1, res.iterations)}

    fp = make_fusion()
    fp.setupCorrespondences(None, method='projective', depths=depth, prune_result=False)
    out["gn_depth_frame_projective_associated"] = int(len(fp._corridx))
    solve(fp, "projective")
    fc = make_fusion()
    fc.setupCorrespondences(None, method='clpts', prune_result=False, live_vertices=live)
    solve(fc, "closest_point")
    out["config"] = ("gn: rw 0.05, huber, %d iterations from node transforms perturbed by N(0, 2e-3), PCG cap 400 at rel. tol 1e-4 "
                     "(Problem.gauss_newton defaults); the projective problem holds the associated pixels only, the closest-point one all "
                     "canonical pixels (prune_result=False)" % args.gn_iters)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
