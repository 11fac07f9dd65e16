"""Raycasting the fused volume on the device (run with -m gpu): dfb_raycast against oracle/raycast.py bit for bit at 64^3, 81^3
and 256^3 volumes fused on the device, at 1 and 8 views; 8 views in one call against 8 single-view calls; FusionDM.raycast on
numpy, CUDA and resident volumes; tracking a raycast frame back to its pose on the device; the slab refusal."""
import numpy as np
import pytest

from track_scenes import Ring, perturb, pose_error

pytestmark = pytest.mark.gpu


def _device_fused(res):
    """Ring scene at res^3 (tdist 3 voxels per 64) fused on the device by FusionDM.fuseDepths from the views at -20 and +20 degrees;
    returns (ring, FusionDM, tsdf, weight) with the volume as float32 CUDA tensors."""
    import torch
    from dynamicfusion_body_b200.fusion import FusionDM
    rg = Ring(res, tdist=3.0 * res / 64)
    fus = FusionDM(rg.tdist, rg.K, tsdf_res=res)
    T = torch.full((res,) * 3, rg.tdist, dtype=torch.float32, device="cuda")
    W = torch.zeros((res,) * 3, dtype=torch.float32, device="cuda")
    for a in (-20.0, 20.0):
        lw = rg.pose(a)
        fus.fuseDepths(rg.frame(lw), lw, T, W, rg.scale, rg.center)
    torch.cuda.synchronize()
    return rg, fus, T, W


@pytest.fixture(scope="module", params=[64, 81, 256])
def fused(request):
    return _device_fused(request.param)


def _poses(rg, n):
    return np.stack([perturb(rg.pose(-35.0 + 10.0 * i, 1.2 + 0.2 * i), 1.0, rg.res / 64, 20 + i) for i in range(n)])


@pytest.mark.parametrize("n_views", [1, 8])
def test_device_equals_oracle(fused, n_views):
    from dynamicfusion_body_b200 import engine
    from oracle import raycast as orc
    rg, fus, T, W = fused
    E = _poses(rg, n_views)
    views = engine.camera_views(rg.K, rg.rows, rg.cols, E)
    z_far = engine.raycast_far(T.shape, rg.res, views, rg.scale, rg.center)
    d, n = engine.raycast((T, W), rg.res, views, rg.scale, rg.center, rg.tdist)
    do, no = orc.raycast(T.cpu().numpy(), W.cpu().numpy(), rg.res, rg.scale, rg.center, rg.tdist, rg.K, rg.rows, rg.cols, E,
                         rg.scale, 0.0, z_far)
    assert np.array_equal(d.cpu().numpy().view(np.uint32), do.view(np.uint32))
    assert np.array_equal(n.cpu().numpy().view(np.uint32), no.view(np.uint32))
    assert (do != 0).mean(axis=(1, 2)).min() > 0.05


def test_eight_views_equal_single_views(fused):
    from dynamicfusion_body_b200 import engine
    rg, fus, T, W = fused
    E = _poses(rg, 8)
    z_far = 3.0 * rg.res
    d8, n8 = engine.raycast((T, W), rg.res, engine.camera_views(rg.K, rg.rows, rg.cols, E), rg.scale, rg.center, rg.tdist,
                            0.75 * rg.scale, 1.0, z_far)
    for v in range(8):
        d1, n1 = engine.raycast((T, W), rg.res, engine.camera_views(rg.K, rg.rows, rg.cols, E[v:v + 1]), rg.scale, rg.center,
                                rg.tdist, 0.75 * rg.scale, 1.0, z_far)
        assert d1[0].cpu().numpy().tobytes() == d8[v].cpu().numpy().tobytes()
        assert n1[0].cpu().numpy().tobytes() == n8[v].cpu().numpy().tobytes()


def test_fusiondm_raycast_api():
    import torch
    from dynamicfusion_body_b200 import engine
    rg, fus, T, W = _device_fused(64)
    lw = rg.pose(5.0)
    on_dev = fus.raycast(lw, T, W, rg.scale, rg.center)
    on_host = fus.raycast(lw, T.cpu().numpy(), W.cpu().numpy(), rg.scale, rg.center)
    fus._tsdf, fus._tsdfw = T.cpu().numpy(), W.cpu().numpy()
    resident = fus.raycast(lw, None, None, rg.scale, rg.center)
    stack = fus.raycast(np.stack([lw, rg.pose(-5.0)]), T, W, rg.scale, rg.center, rows=240, cols=320, K=rg.K * [[0.5], [0.5], [1]])
    assert on_dev.depth.shape == (1, rg.rows, rg.cols) and on_dev.normal.shape == (1, rg.rows, rg.cols, 3)
    assert stack.depth.shape == (2, 240, 320)
    for r in (on_host, resident):
        assert r.depth.cpu().numpy().tobytes() == on_dev.depth.cpu().numpy().tobytes()
        assert r.normal.cpu().numpy().tobytes() == on_dev.normal.cpu().numpy().tobytes()
    views = engine.camera_views(rg.K, rg.rows, rg.cols, lw[None])
    d, _ = engine.raycast((T, W), rg.res, views, rg.scale, rg.center, rg.tdist)
    assert d.cpu().numpy().tobytes() == on_dev.depth.cpu().numpy().tobytes()
    # the documented loop: track, fuse, raycast the model from the tracked pose
    truth = perturb(rg.pose(0.0), 2.0, 1.0, 5)
    dm = rg.frame(truth)
    lw_t = fus.track(dm, rg.pose(0.0), T, W, rg.scale, rg.center).lw
    fus.fuseDepths(dm, lw_t, T, W, rg.scale, rg.center)
    model = fus.raycast(lw_t, T, W, rg.scale, rg.center)
    both = (model.depth[0].cpu().numpy() != 0) & (dm != 0)
    assert both.sum() > 0.8 * (dm != 0).sum()
    assert np.median(np.abs(model.depth[0].cpu().numpy()[both] - dm[both])) < 0.5
    with pytest.raises(ValueError, match="3x4"):
        fus.raycast(np.eye(4), T, W, rg.scale, rg.center)
    with pytest.raises(ValueError, match="views"):
        fus.raycast(np.stack([lw] * 9), T, W, rg.scale, rg.center)
    torch.cuda.synchronize()


def test_slab_volume_is_refused():
    import torch
    from dynamicfusion_body_b200 import _capi, engine
    rg, fus, T, W = _device_fused(64)
    fus._vol = engine.DeviceVolume((64,) * 3, 0, 32, device=T.device, tsdf=T[:32], weight=W[:32])
    with pytest.raises(_capi.DfbError, match="slab"):
        fus.raycast(rg.pose(0.0), None, None, rg.scale, rg.center)
    torch.cuda.synchronize()


# measured on a B200: 0.0068 deg and 0.0073 voxel for each seed, as with the oracle backend (tests/test_raycast_host.py)
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_device_tracks_a_raycast_frame_back_to_its_pose(seed):
    rg, fus, T, W = _device_fused(64)
    truth = rg.pose(0.0)
    dm = fus.raycast(truth, T, W, rg.scale, rg.center).depth[0]
    res = fus.track(dm, perturb(truth, 2.0, 1.0, seed), T, W, rg.scale, rg.center)
    rot, tr = pose_error(res.lw, truth)
    print("device, seed %d: %.4f deg, %.4f voxel, iterations %s" % (seed, rot, tr / rg.scale, res.iterations))
    assert rot < 0.02 and tr / rg.scale < 0.03
