"""Z-buffer rasteriser (csrc/dfb_render.h, compiled for the host by tests/hostshim/render_shim.cpp) against the oracle
(oracle/render.py): bit-for-bit agreement on synthetic scenes and on knife-edge constructions, known answers, coverage against
the test scenes' point-splat renderer, and the C-ABI argument validation of dfb_render.  tests/test_gpu_render.py runs the
device kernels."""
import ctypes

import numpy as np
import pytest

import hostshim_api as hs
from dynamicfusion_body_b200 import synth
from oracle import render as orr

# dyadic intrinsics: camera points built from dyadic pixel coordinates and depths project exactly
F, CX, CY = 2.0, 8.0, 6.0
K = np.array([[F, 0, CX], [0, F, CY], [0, 0, 1.0]])
ROWS, COLS = 13, 17


def _cam(x, y, z):
    """The camera-frame point that projects onto pixel coordinates (x, y) at depth z."""
    return np.array([(x - CX) * z / F, (y - CY) * z / F, z], np.float64)


def _assert_bits(h, o):
    assert np.array_equal(h[0].view(np.uint32), o[0].view(np.uint32))
    assert np.array_equal(h[1], o[1])
    assert np.array_equal(h[2].view(np.uint32), o[2].view(np.uint32))


def _both(pts, faces, extrinsics=None, rows=ROWS, cols=COLS, k=K):
    """host build and oracle on the same input; asserts they agree bit for bit and returns the oracle's view 0 (or all views)."""
    pts = np.asarray(pts, np.float64).reshape(-1, 3)
    faces = np.asarray(faces, np.int32).reshape(-1, 3)
    h = hs.render(pts, faces, k, rows, cols, extrinsics)
    o = orr.render(pts, faces, k, rows, cols, extrinsics)
    _assert_bits(h, o)
    return tuple(a[0] for a in o) if extrinsics is None else o


def _tri(*xyz):
    return np.stack([_cam(*p) for p in xyz])


def test_fronto_parallel_quad():
    z0 = 3.7
    pts = _tri((2.5, 1.5, z0), (14.5, 1.5, z0), (14.5, 10.5, z0), (2.5, 10.5, z0))
    depth, face, normal = _both(pts, [[0, 1, 2], [0, 2, 3]])
    cov = face >= 0
    assert cov.sum() == 12 * 9                                   # columns 3..14, rows 2..10
    ref = np.float32(z0)
    ulp = np.spacing(ref)
    assert np.all(np.abs(-depth[cov] - ref) <= ulp)
    assert np.all(depth[~cov] == 0) and np.all(normal[~cov] == 0)
    # (Pb - Pa) x (Pc - Pa) of these windings points along +z in the camera frame (away from the camera): not flipped
    assert np.array_equal(normal[cov], np.tile(np.float32([0, 0, 1]), (cov.sum(), 1)))


def test_tilted_plane_is_the_ray_plane_intersection():
    nrm = np.array([0.07, -0.05, 1.0])
    d = 5.0
    corners = []
    for x, y in ((-1.0, -1.0), (18.0, -1.0), (18.0, 14.0), (-1.0, 14.0)):
        ray = np.linalg.solve(K, [x, y, 1.0])
        corners.append(ray * d / nrm.dot(ray))                  # on the plane nrm . X = d
    depth, face, _ = _both(np.stack(corners), [[0, 1, 2], [0, 2, 3]])
    assert (face >= 0).all()
    r, c = np.mgrid[0:ROWS, 0:COLS]
    rays = np.stack([(c - CX) / F, (r - CY) / F, np.ones_like(c, dtype=np.float64)], -1)
    z = d / (rays @ nrm)                                         # depth of the intersection (ray z component is 1)
    zf = -depth.astype(np.float64)
    # zf is float32(z') for a z' within 1e-12 of z, relative
    assert np.all(np.abs(zf - z) <= 0.5 * np.spacing(np.float32(zf)) + 1e-12 * z)


def test_nearer_face_wins_and_ties_go_to_the_lower_id():
    box = ((1.5, 1.5), (15.5, 1.5), (1.5, 11.5))
    near = _tri(*[(x, y, 3.0) for x, y in box])
    far = _tri(*[(x, y, 4.0) for x, y in box])
    for order, winner in (((far, near), 1), ((near, far), 0)):
        _, face, _ = _both(np.concatenate(order), [[0, 1, 2], [3, 4, 5]])
        assert set(np.unique(face[face >= 0])) == {winner}
    # equal float32 depth: face 0 is farther in float64 by 1e-12, the same in float32, and wins by its lower id
    z = 3.0
    a = _tri(*[(x, y, z * (1 + 1e-12)) for x, y in box])
    b = _tri(*[(x, y, z) for x, y in box])
    depth, face, _ = _both(np.concatenate([a, b]), [[0, 1, 2], [3, 4, 5]])
    assert set(np.unique(face[face >= 0])) == {0} and np.all(depth[face >= 0] == -np.float32(z))


def test_inclusive_edges_and_vertices():
    # vertices on pixel centres; the hypotenuse passes through pixel centres: all of them are covered
    pts = _tri((2, 2, 4.0), (10, 2, 4.0), (2, 10, 4.0))
    _, face, _ = _both(pts, [[0, 1, 2]])
    r, c = np.mgrid[0:ROWS, 0:COLS]
    inside = (c >= 2) & (r >= 2) & ((c - 2) + (r - 2) <= 8)
    assert np.array_equal(face == 0, inside) and inside.sum() == 45
    # the same with the opposite winding (negative area)
    _, face, _ = _both(pts, [[0, 2, 1]])
    assert np.array_equal(face == 0, inside)
    # two faces sharing the diagonal through pixel centres: both cover it, the depth test decides (here the nearer face 1)
    quad = np.concatenate([_tri((2, 2, 4.0), (10, 2, 4.0), (10, 10, 4.0)), _tri((2, 2, 3.0), (10, 10, 3.0), (2, 10, 3.0))])
    _, face, _ = _both(quad, [[0, 1, 2], [3, 4, 5]])
    diag = np.arange(2, 11)
    assert np.all(face[diag, diag] == 1)
    assert np.all(face[2:11, 2:11][np.triu_indices(9, 1)] == 0) and np.all(face[2:11, 2:11][np.tril_indices(9, -1)] == 1)


def test_culled_faces():
    good = _tri((2, 2, 4.0), (10, 2, 4.0), (2, 10, 4.0))
    behind = good.copy(); behind[1, 2] = -1.0                     # a vertex behind the camera
    on = good.copy(); on[1] = 0.0                                 # a vertex at the centre of projection (z = 0)
    line = _tri((2, 2, 4.0), (6, 6, 4.0), (10, 10, 4.0))          # collinear: zero area
    pts = np.concatenate([good, behind, on, line])
    n = len(pts)
    faces = [[3, 4, 5], [6, 7, 8], [9, 10, 11], [0, 1, n], [0, -1, 2], [0, 1, 2]]
    depth, face, _ = _both(pts, faces)
    assert set(np.unique(face)) == {-1, 5}                        # only the last face renders
    assert (face == 5).sum() == 45
    for f in faces[:-1]:
        _, face, _ = _both(pts, [f])
        assert (face == -1).all(), f


def test_partly_outside_and_whole_image_faces():
    # a face reaching past every border: covered pixels are exactly those inside the triangle
    pts = _tri((-7.3, -4.1, 4.0), (25.6, 3.2, 5.0), (4.4, 22.7, 6.0))
    _, face, _ = _both(pts, [[0, 1, 2]])
    x, y = [], []
    for p in pts:
        q = K @ p
        x.append(q[0] / q[2]); y.append(q[1] / q[2])
    r, c = np.mgrid[0:ROWS, 0:COLS]
    e = [(x[(i + 2) % 3] - x[(i + 1) % 3]) * (r - y[(i + 1) % 3]) - (y[(i + 2) % 3] - y[(i + 1) % 3]) * (c - x[(i + 1) % 3]) for i in range(3)]
    inside = (e[0] >= 0) & (e[1] >= 0) & (e[2] >= 0)
    assert np.array_equal(face == 0, inside) and 0 < inside.sum() < ROWS * COLS
    # one face covering the whole image
    pts = _tri((-100, -100, 5.0), (300, -100, 5.0), (-100, 300, 5.0))
    depth, face, _ = _both(pts, [[0, 1, 2]])
    assert (face == 0).all() and np.all(depth == -np.float32(5.0))
    # and its box entirely outside the image: nothing
    pts = _tri((20, 20, 5.0), (30, 20, 5.0), (20, 30, 5.0))
    assert (_both(pts, [[0, 1, 2]])[1] == -1).all()


def test_extrinsics_and_normals_stay_in_the_frame_of_the_points():
    # the camera looks down -x of the point frame; normals are reported in the point frame
    Rm = np.array([[0, 1.0, 0], [0, 0, 1.0], [1.0, 0, 0]])       # camera (x, y, z) = point (y, z, x)
    t = np.array([0.5, -0.25, 2.0])
    E = np.concatenate([Rm, t[:, None]], 1)
    cam = _tri((2, 2, 4.0), (10, 2, 4.0), (2, 10, 4.0))
    pts = (cam - t) @ Rm                                          # R^T (cam - t)
    _, face, normal = _both(pts, [[0, 1, 2]], extrinsics=E[None])
    n = np.cross(pts[1] - pts[0], pts[2] - pts[0])
    assert (face[0] == 0).sum() == 45
    assert np.allclose(normal[0][face[0] == 0], n / np.linalg.norm(n), atol=1e-7)


@pytest.mark.parametrize("n_views,k", [(1, 4), (1, 8), (3, 4), (3, 8)])
def test_scene_host_equals_oracle(n_views, k):
    sc = synth.make_scene(res=64, k=k, n_nodes=300, seed=11, n_views=n_views)
    out = _both(sc.warped_vertices, sc.faces, sc.extrinsics, sc.rows, sc.cols, sc.K)
    face = out[1] if n_views > 1 else out[1][None]
    assert all((f >= 0).mean() > 0.1 for f in face)                # the body fills a good part of every view
    assert len(np.unique(face[face >= 0])) > 0.3 * len(sc.faces)


@pytest.mark.parametrize("n_views", [1, 3])
def test_coverage_against_the_point_splatter(n_views):
    """synth.render_depth splats dense surface samples over 2x2 pixel blocks into a min z-buffer: its silhouette grows by up to a
    pixel and its surface moves up to about a pixel toward the camera.  The two renderings of the same warped mesh still agree:
    the non-empty masks differ on under 2 % of covered pixels, and the median depth difference is under the median pixel
    footprint (oracle at this size: 1.8 % / 1.5 % of pixels differ, median |dz| 0.14 / 0.12 against a footprint of 0.16)."""
    sc = synth.make_scene(res=64, k=4, n_nodes=300, seed=11, n_views=n_views)
    depth, _, _ = orr.render(sc.warped_vertices, sc.faces, sc.K, sc.rows, sc.cols, sc.extrinsics)
    ours, theirs = depth != 0, sc.depths != 0
    diff = float((ours ^ theirs).sum()) / float((ours | theirs).sum())
    both = ours & theirs
    dz = float(np.median(np.abs(depth[both].astype(np.float64) - sc.depths[both])))
    footprint = float(np.median(-depth[ours])) / sc.K[0, 0]
    print("mask difference %.4f of covered pixels, median |dz| %.4f, footprint %.4f" % (diff, dz, footprint))
    assert diff < 0.02
    assert dz < footprint


def test_argument_validation_without_gpu():
    from dynamicfusion_body_b200 import _capi
    lib = _capi.lib()
    p = ctypes.c_void_p(8)
    good = _capi.Views()
    good.n_views, good.rows, good.cols = 2, 8, 8
    words = lib.dfb_render_workspace_words(5, 2, 8, 8)
    assert words == 1 + 2 * 64 + 5 * 2
    for bad in ((-1, 1, 8, 8), (5, 0, 8, 8), (5, 1, 0, 8), (5, 1, 8, 0)):
        assert lib.dfb_render_workspace_words(*bad) == -1

    def call(views=good, pts=p, n_pts=4, faces=p, n_faces=5, ws=p, n_ws=words, depth=p, face=p, normal=p):
        return lib.dfb_render(pts, n_pts, faces, n_faces, ctypes.byref(views) if views is not None else None, ws, n_ws, depth, face,
                              normal, None)

    cases = [(dict(pts=None), b"null pointer"), (dict(faces=None), b"null pointer"), (dict(views=None), b"null pointer"),
             (dict(ws=None), b"null pointer"), (dict(depth=None), b"null pointer"), (dict(face=None), b"null pointer"),
             (dict(normal=None), b"null pointer"), (dict(n_pts=-1), b"negative count"), (dict(n_faces=-1), b"negative count"),
             (dict(n_faces=1 << 31), b"int32 face ids"), (dict(n_ws=words - 1), b"workspace")]
    for kw, msg in cases:
        assert call(**kw) == -1, kw
        assert msg in lib.dfb_last_error(), (kw, lib.dfb_last_error())
    for field, val, msg in (("n_views", 0, b"n_views"), ("n_views", 9, b"n_views"), ("rows", 0, b"is empty"), ("cols", 0, b"is empty")):
        bad = _capi.Views.from_buffer_copy(good)
        setattr(bad, field, val)
        assert call(bad) == -1 and msg in lib.dfb_last_error(), field
