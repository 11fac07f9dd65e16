"""Projective data association (csrc/dfb_math.h assoc_projective_ref, compiled for the host by tests/hostshim/assoc_shim.cpp) against the
oracle (oracle/assoc.py): known answers on hand-built depth maps, bit-for-bit agreement on synthetic scenes and on knife-edge
constructions, and the C-ABI argument validation of dfb_corr_projective.  tests/test_gpu_assoc.py runs the device kernel."""
import ctypes

import numpy as np
import pytest

import assoc_shim
import hostshim_api as hs
from dynamicfusion_body_b200 import synth
from oracle import assoc as oa

# dyadic intrinsics: Kinv is exact, so back-projections of integer pixels at dyadic depths are exact
F, CX, CY = 2.0, 8.0, 6.0
K = np.array([[F, 0, CX], [0, F, CY], [0, 0, 1.0]])
KINV = np.linalg.inv(K)
ROWS, COLS = 13, 17
MD = 0.5                                   # max_distance
Z = 4.0                                    # plane depth


def _plane(z=Z):
    return np.full((ROWS, COLS), -z, np.float32)


def _pixel_point(u, v, z=Z):
    """Kinv [z u, z v, z], summed like the kernel: the back-projection of pixel (u, v) at depth z."""
    c = [z * u, z * v, z * 1.0]
    return np.array([(KINV[r, 0] * c[0] + KINV[r, 1] * c[1]) + KINV[r, 2] * c[2] for r in range(3)])


FACING = np.array([0.0, 0.0, -1.0])


def _both(pts, nrm, dms, md=MD, mnd=0.5, extrinsics=None):
    """host build and oracle on the same input; asserts they agree bit for bit and returns the result."""
    pts = np.atleast_2d(np.asarray(pts, np.float64))
    nrm = np.atleast_2d(np.asarray(nrm, np.float64))
    dms = np.asarray(dms, np.float32).reshape(-1, ROWS, COLS) if np.ndim(dms) == 2 else np.asarray(dms, np.float32)
    hv, hc, hp = assoc_shim.corr_projective(pts, nrm, dms, K, KINV, md, mnd, extrinsics)
    ov, oc, op = oa.associate(pts, nrm, dms, K, KINV, md, mnd, extrinsics)
    _assert_bits(hv, hc, hp, ov, oc, op)
    return ov, oc, op


def _assert_bits(hv, hc, hp, ov, oc, op):
    assert np.array_equal(hv, ov)
    assert np.array_equal(hc.view(np.uint64), oc.view(np.uint64))
    assert np.array_equal(hp.view(np.uint64), op.view(np.uint64))


def test_fronto_parallel_plane_maps_vertex_onto_itself():
    w = _pixel_point(7, 5)
    v, c, p = _both(w, FACING, _plane())
    assert v[0] == 0 and c[0] == 0.0 and np.array_equal(p[0], w)


def test_rejections():
    dm = _plane()
    cases = {
        "occluded": (_pixel_point(7, 5, Z + 2.0), FACING, dm),                 # behind the measured surface, beyond max_distance
        "back_facing": (_pixel_point(7, 5), -FACING, dm),
        "outside_frustum": (_pixel_point(-2, 5), FACING, dm),
        "border_ring_u0": (_pixel_point(0, 5), FACING, dm),
        "border_ring_u_last": (_pixel_point(COLS - 1.4, 5), FACING, dm),      # inside the frustum, rounds onto column cols-1
        "border_ring_v_last": (_pixel_point(7, ROWS - 1.4), FACING, dm),
        "behind_camera": (-_pixel_point(7, 5), -FACING, dm),
    }
    nodata = dm.copy(); nodata[5, 7] = 0
    cases["no_data"] = (_pixel_point(7, 5), FACING, nodata)
    nbr_nodata = dm.copy(); nbr_nodata[4, 7] = 0
    cases["neighbour_no_data"] = (_pixel_point(7, 5), FACING, nbr_nodata)
    step = dm.copy(); step[5, 8:] = -(Z + 2 * MD)
    cases["neighbour_across_step"] = (_pixel_point(7, 5), FACING, step)
    for name, (w, n, d) in cases.items():
        v, c, p = _both(w, n, d)
        assert v[0] == -1 and c[0] == np.inf and not p.any(), name
    # the control: the same vertex against the clean plane associates
    assert _both(_pixel_point(7, 5), FACING, dm)[0][0] == 0


def test_two_views_lower_index_wins_tie_and_argmin():
    w = _pixel_point(7, 5, Z + 0.25)
    v, c, _ = _both(w, FACING, np.stack([_plane(), _plane()]))
    assert v[0] == 0 and c[0] == 0.25
    v, c, p = _both(w, FACING, np.stack([_plane(), _plane(Z + 0.25)]))        # view 1 is closer: it wins
    assert v[0] == 1 and c[0] == 0.0 and np.array_equal(p[0], w)


def test_extrinsics_map_back_into_the_frame_of_the_points():
    # view 0: camera frame = point frame shifted by t; corr must come back in the point frame
    t = np.array([0.5, -0.25, 1.0])
    E = np.concatenate([np.eye(3), t[:, None]], 1)
    w = _pixel_point(7, 5) - t
    v, c, p = _both(w, FACING, _plane(), extrinsics=E[None])
    assert v[0] == 0 and c[0] == 0.0 and np.array_equal(p[0], w)


def test_knife_edges():
    dm = _plane()
    # projection exactly on a half-integer pixel: round half to even (u = 6.5 -> 6, u = 7.5 -> 8); half a pixel is 1 unit here
    for u, ui in ((6.5, 6), (7.5, 8)):
        w = _pixel_point(u, 5)
        v, c, p = _both(w, FACING, dm, md=1.0)
        assert v[0] == 0 and np.array_equal(p[0], _pixel_point(ui, 5))
    # a depth step of exactly max_distance is kept, one ulp more is not
    for dz, ok in ((MD, True), (np.nextafter(np.float32(Z + MD), np.float32(10)) - Z, False)):
        d = dm.copy(); d[5, 8] = -np.float32(Z + dz)
        assert (_both(_pixel_point(7, 5), FACING, d)[0][0] == 0) == ok
    # normal dot exactly at min_normal_dot: ln = (3,0,-4) against the plane normal (0,0,-|g|) has cos = 0.8 exactly
    ln = np.array([3.0, 0.0, -4.0])
    assert _both(_pixel_point(7, 5), ln, dm, mnd=0.8)[0][0] == 0
    assert _both(_pixel_point(7, 5), ln, dm, mnd=np.nextafter(0.8, 1.0))[0][0] == -1
    # distance gate exactly at max_distance (|l - c|^2 == max_distance^2): a point on the optical axis MD in front of the plane
    assert _both(_pixel_point(CX, CY, Z - MD), FACING, dm)[0][0] == 0
    assert _both(_pixel_point(CX, CY, Z - MD), FACING, dm, md=np.nextafter(MD, 0.0))[0][0] == -1


def test_knife_edge_battery_matches_oracle():
    """Random points on the half-integer pixel lattice at dyadic depths, depth maps with steps of exactly max_distance and
    holes, dyadic normals at exact cosines: every decision on its edge, host build == oracle bit for bit."""
    rng = np.random.default_rng(5)
    n = 4000
    md = 1.0                                                     # = half a pixel's footprint at depth Z: half-pixel offsets sit on the gate
    u = rng.integers(-2, 2 * COLS + 2, n) * 0.5
    v = rng.integers(-2, 2 * ROWS + 2, n) * 0.5
    z = Z + rng.integers(-2, 3, n) * (md / 2)
    pts = np.stack([_pixel_point(a, b, c) for a, b, c in zip(u, v, z)])
    normals = np.array([[0, 0, -1], [3, 0, -4], [0, 3, -4], [4, 0, -3], [0, -4, -3], [0, 0, 1], [1, 0, 0]], np.float64)
    nrm = normals[rng.integers(0, len(normals), n)] * rng.choice([0.5, 1.0, 2.0], n)[:, None]
    steps = rng.choice([0, 0, 0, 0, 0, 0, 1, -1, 2], (3, ROWS, COLS)) * md              # steps of exactly max_distance, and beyond
    dms = -(Z + steps).astype(np.float32)
    dms[rng.random(dms.shape) < 0.03] = 0
    for mnd in (0.8, 0.6, -1.0, 1.0):
        view, cost, corr = _both(pts, nrm, dms, md=md, mnd=mnd)
        if mnd < 1.0:
            assert (view >= 0).sum() > 100 and (view < 0).sum() > 100
    E = np.stack([np.concatenate([np.eye(3), np.array([[0.5 * i], [-0.25 * i], [0.0]])], 1) for i in range(3)])
    _both(pts, nrm, dms, md=md, mnd=0.6, extrinsics=E)


@pytest.mark.parametrize("n_views,k", [(1, 4), (1, 8), (3, 4), (3, 8)])
def test_scene_host_equals_oracle(n_views, k):
    sc = synth.make_scene(res=64, k=k, n_nodes=300, seed=11, n_views=n_views, rows=240, cols=320)
    wf = hs.HostWarpField(sc.node_pos, sc.node_dq, np.float32(sc.node_w), sc.k, lw=sc.lw)
    # the body-mesh fixture's normals point into the body; association wants them pointing out (as marching cubes of a TSDF)
    wv, wn = hs.warp_points(sc.vertices, -sc.normals, sc.vert_knn, wf)
    hv, hc, hp = assoc_shim.corr_projective(wv, wn, sc.depths, sc.K, sc.Kinv, sc.tdist, 0.5, sc.extrinsics)
    ov, oc, op = oa.associate(wv, wn, sc.depths, sc.K, sc.Kinv, sc.tdist, 0.5, sc.extrinsics)
    _assert_bits(hv, hc, hp, ov, oc, op)
    frac = float((ov >= 0).mean())
    assert frac > 0.2, frac                                      # a depth camera sees the front of the body
    if n_views > 1:
        assert len(np.unique(ov[ov >= 0])) > 1


def test_argument_validation_without_gpu():
    from dynamicfusion_body_b200 import _capi
    lib = _capi.lib()
    p = ctypes.c_void_p(8)
    good = _capi.Views()
    good.n_views, good.rows, good.cols = 1, 8, 8
    good.depth[0] = 8

    def call(views, m=4, md=1.0, mnd=0.5, pts=p):
        return lib.dfb_corr_projective(pts, p, m, ctypes.byref(views) if views is not None else None, md, mnd, p, p, p, None)

    cases = [(dict(pts=None), b"null pointer"), (dict(views=None), b"null pointer"), (dict(m=-1), b"negative count"),
             (dict(md=0.0), b"max_distance"), (dict(md=float("nan")), b"max_distance"), (dict(md=-1.0), b"max_distance"),
             (dict(mnd=1.5), b"min_normal_dot"), (dict(mnd=float("nan")), b"min_normal_dot"), (dict(mnd=-1.01), b"min_normal_dot")]
    for kw, msg in cases:
        args = dict(views=good)
        args.update(kw)
        assert call(**args) == -1, kw
        assert msg in lib.dfb_last_error(), (kw, lib.dfb_last_error())
    for field, val, msg in (("n_views", 0, b"n_views"), ("n_views", 9, b"n_views"), ("rows", 2, b"smaller than 3x3"),
                            ("cols", 2, b"smaller than 3x3")):
        bad = _capi.Views.from_buffer_copy(good)
        setattr(bad, field, val)
        assert call(bad) == -1 and msg in lib.dfb_last_error()
    nulldepth = _capi.Views()
    nulldepth.n_views, nulldepth.rows, nulldepth.cols = 2, 8, 8
    nulldepth.depth[0] = 8
    assert call(nulldepth) == -1 and b"depth[1] is null" in lib.dfb_last_error()
