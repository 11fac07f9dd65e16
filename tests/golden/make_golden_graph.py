"""Generate tests/golden/reference_graph_vectors.npz by EXECUTING THE UNMODIFIED REFERENCE (a checkout at oracle/_ref/,
see oracle/refload.py) for the SURVEY 8f rows next to the hot paths: closest-point correspondences (Fusion /
FusionDM.setupCorrespondences), `uniform_sample`, and `Fusion.update_graph`:

    python tests/golden/make_golden_graph.py

scikit-image is not installed, so `marching_cubes` is replaced on the INSTANCE by a function returning the supplied
live vertices (setupCorrespondences) or doing nothing (update_graph: the canonical vertices are set by hand); every
line of the reference after that call runs unmodified.  Inputs are stored alongside the outputs.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import refload  # noqa: E402
from make_golden import rand_dq  # noqa: E402


def main():
    util, Fusion, FusionDM = refload.load()
    rng = np.random.default_rng(777)
    mesh = np.load(os.path.join(HERE, "body_mesh.npz"))
    mv, mn = mesh["vertices"], mesh["normals"]
    out = {}
    k = 4
    radius = 4.0

    # canonical surface = every 12th mesh vertex; deformation nodes by the reference's own sampler
    verts = np.ascontiguousarray(mv[::12]); norms = np.ascontiguousarray(mn[::12])
    node_pos, node_idx = util.uniform_sample(verts, radius)
    N = len(node_pos)
    node_dq = rand_dq(rng, N, scale_t=0.4, ang=0.15).astype(np.float32)
    lw = rand_dq(rng, 1, scale_t=0.5, ang=0.1)[0]
    out.update(verts=verts, norms=norms, radius=radius, k=k, node_pos=node_pos, node_idx=node_idx, node_dq=node_dq, lw=lw)

    # live surface: another subset of the mesh, displaced a little (plays marching cubes of the live TSDF)
    lverts = (mv[5::7] + rng.normal(size=mv[5::7].shape) * 0.3 + np.array([0.4, -0.2, 0.3])).astype(np.float32)
    out["lverts"] = lverts

    nodes = [(int(node_idx[i]), node_pos[i], node_dq[i], 2 * radius) for i in range(N)]
    f = refload.make_fusion(nodes, None, None, 1.0, k, lw)
    vknn = np.array([f._kdtree.query(v, k=k)[1] for v in verts])
    f._vertices, f._normals, f._neighbor_look_up = verts.copy(), norms.copy(), list(vknn)
    f.marching_cubes = lambda *a, **kw: (lverts, None, None, None)
    with refload.quiet():
        f.setupCorrespondences(np.zeros((2, 2, 2)), method='clpts', prune_result=False)
    out["vknn"] = vknn
    out["corr_fusion"] = np.array(f._correspondences)

    fdm = FusionDM(0.5, np.eye(3), tsdf_res=4, knn=k)
    fdm._lw = lw
    fdm._vertices, fdm._normals = verts.copy(), norms.copy()
    fdm.marching_cubes = lambda *a, **kw: (lverts, None, None, None)
    with refload.quiet():
        fdm.setupCorrespondences(None, tolerance=0.25)
    out["dm_tolerance"] = 0.25
    out["dm_corridx"] = np.array(fdm._corridx)
    out["dm_corr"] = np.array(fdm._correspondences)

    # uniform_sample on its own (second radius)
    us_v, us_i = util.uniform_sample(lverts[:1200], 2.5)
    out["us_radius"] = 2.5
    out["us_idx"] = us_i

    # update_graph: the new canonical surface is the live one -> parts of it are unsupported by the old graph
    g = refload.make_fusion(nodes, None, None, 1.0, k, lw)
    new_verts = np.ascontiguousarray(np.concatenate([verts, (mv[3::40] + np.array([9.0, 0, 0])).astype(np.float32)]))
    g._vertices, g._radius = new_verts, radius
    g.marching_cubes = lambda *a, **kw: None
    with refload.quiet():
        g.update_graph()
    out["ug_verts"] = new_verts
    out["ug_node_vidx"] = np.array([n[0] for n in g._nodes])
    out["ug_node_pos"] = np.array([n[1] for n in g._nodes])
    out["ug_node_dq"] = np.array([np.asarray(n[2], dtype=np.float64) for n in g._nodes])
    out["ug_lookup"] = np.array(g._neighbor_look_up)

    path = os.path.join(HERE, "reference_graph_vectors.npz")
    np.savez_compressed(path, **{k_: np.asarray(v) for k_, v in out.items()})
    print("wrote", path, os.path.getsize(path), "bytes,", len(out), "arrays;", N, "nodes ->", len(g._nodes))


if __name__ == "__main__":
    main()
