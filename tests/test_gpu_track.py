"""Rigid point-to-TSDF tracking on the device (run with -m gpu): dfb_track_normal_eq against oracle/track.py (residual maps bit for
bit, sums to rounding) at 64^3, 81^3 and 256^3, run-to-run determinism, the device-backed Levenberg-Marquardt trajectory against
the oracle-backed one, a 20-frame track-and-fuse sequence, and FusionDM.track."""
import numpy as np
import pytest

from track_scenes import Ring, perturb, pose_error

pytestmark = pytest.mark.gpu


def _assert_sums_close(a, b, rel=1e-12):
    """as tests/test_track_host.py: each sum to `rel` of its Cauchy-Schwarz bound, the cost relative, the count exact."""
    from oracle import track as otr
    Ha, ga, ca, na = otr.unpack(a)
    Hb, gb, cb, nb = otr.unpack(b)
    d = np.sqrt(np.abs(np.diag(Hb)))
    assert np.all(np.abs(Ha - Hb) <= rel * np.outer(d, d) + 1e-300)
    assert np.all(np.abs(ga - gb) <= rel * d * np.sqrt(2 * cb) + 1e-300)
    assert abs(ca - cb) <= rel * cb and na == nb


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


@pytest.mark.parametrize("stride", [1, 2, 4])
def test_device_equals_oracle(fused, stride):
    import torch
    from dynamicfusion_body_b200 import engine
    from oracle import track as otr
    rg, fus, T, W = fused
    Th, Wh = T.cpu().numpy(), W.cpu().numpy()
    delta = 0.5 * rg.tdist
    for lw in (perturb(rg.pose(0.0, 1.2), 2.0, rg.res / 64, 11), perturb(rg.pose(10.0, 2.5), 2.0, rg.res / 64, 12)):   # near, far
        d = engine._to_dev(rg.frame(lw), torch.float32, T.device)
        sums, res = engine.track_normal_eq((T, W), rg.res, d, lw, rg.K, rg.Kinv, rg.scale, rg.center, stride, rg.tdist, delta,
                                           want_residual=True)
        so, ro = otr.normal_eq(Th, Wh, rg.res, rg.scale, rg.center, d.cpu().numpy(), rg.Kinv, lw, stride, rg.tdist, delta,
                               want_residual=True)
        assert np.array_equal(res.cpu().numpy().view(np.uint64), ro.view(np.uint64))
        _assert_sums_close(sums, so)
        assert so[28] > 200


def test_two_calls_give_identical_sums(fused):
    import torch
    from dynamicfusion_body_b200 import engine
    rg, fus, T, W = fused
    lw = rg.pose(5.0)
    d = engine._to_dev(rg.frame(lw), torch.float32, T.device)
    a = engine.track_normal_eq((T, W), rg.res, d, lw, rg.K, rg.Kinv, rg.scale, rg.center, 1, rg.tdist, 0.5 * rg.tdist)
    b = engine.track_normal_eq((T, W), rg.res, d, lw, rg.K, rg.Kinv, rg.scale, rg.center, 1, rg.tdist, 0.5 * rg.tdist)
    assert a.tobytes() == b.tobytes()


def test_device_trajectory_equals_oracle_trajectory():
    import torch
    from dynamicfusion_body_b200 import engine
    from oracle import track as otr
    rg, fus, T, W = _device_fused(64)
    Th, Wh = T.cpu().numpy(), W.cpu().numpy()
    lw0 = rg.pose(0.0)
    truth = perturb(lw0, 2.0, 1.0, 1)
    dm = rg.frame(truth)
    d = engine._to_dev(dm, torch.float32, T.device)
    logs = {"dev": [], "ora": []}

    def dev(lw, s):
        r = engine.track_normal_eq((T, W), rg.res, d, lw, rg.K, rg.Kinv, rg.scale, rg.center, s, rg.tdist, 0.5 * rg.tdist)
        logs["dev"].append((s, int(r[28]), r[27]))
        return r

    def ora(lw, s):
        r = otr.normal_eq(Th, Wh, rg.res, rg.scale, rg.center, dm, rg.Kinv, lw, s, rg.tdist, 0.5 * rg.tdist)
        logs["ora"].append((s, int(r[28]), r[27]))
        return r
    a, b = engine.track_rigid(dev, lw0), engine.track_rigid(ora, lw0)
    assert a.iterations == b.iterations and a.converged == b.converged and a.pixels == b.pixels
    assert [x[:2] for x in logs["dev"]] == [x[:2] for x in logs["ora"]]          # same poses evaluated, same pixel counts
    assert np.allclose([x[2] for x in logs["dev"]], [x[2] for x in logs["ora"]], rtol=1e-9, atol=0)
    assert np.abs(a.lw - b.lw).max() <= 1e-9
    print("device: %.4f deg, %.4f voxel, iterations %s" % (pose_error(a.lw, truth) + (a.iterations,)))


def test_track_and_fuse_sequence():
    """20 frames along a ring arc, 3 degrees apart: frame 0 fused at its true pose, every later frame tracked from the previous
    estimate and fused at its estimate (CUDA volumes, FusionDM.track / fuseDepths)."""
    import torch
    from dynamicfusion_body_b200.fusion import FusionDM
    rg = Ring(64)
    fus = FusionDM(rg.tdist, rg.K, tsdf_res=64)
    T = torch.full((64,) * 3, rg.tdist, dtype=torch.float32, device="cuda")
    W = torch.zeros((64,) * 3, dtype=torch.float32, device="cuda")
    lw = rg.pose(0.0)
    fus.fuseDepths(rg.frame(lw), lw, T, W, rg.scale, rg.center)
    errs = []
    for i in range(1, 20):
        truth = rg.pose(3.0 * i)
        dm = rg.frame(truth)
        lw = fus.track(dm, lw, T, W, rg.scale, rg.center).lw
        fus.fuseDepths(dm, lw, T, W, rg.scale, rg.center)
        errs.append(pose_error(lw, truth))
    rot, tr = errs[-1]
    print("sequence drift after 19 tracked frames: %.4f deg, %.4f voxel (max over frames %.4f deg, %.4f voxel)"
          % (rot, tr, max(e[0] for e in errs), max(e[1] for e in errs)))
    assert rot < 0.5 and tr < 1.0


def test_fusiondm_track_api():
    import torch
    from dynamicfusion_body_b200 import _capi, engine
    from oracle import track as otr
    rg, fus, T, W = _device_fused(64)
    lw0 = rg.pose(0.0)
    truth = perturb(lw0, 2.0, 1.0, 2)
    dm = rg.frame(truth)
    on_dev = fus.track(dm, lw0, T, W, rg.scale, rg.center, want_residual=True)
    on_host = fus.track(dm, lw0, T.cpu().numpy(), W.cpu().numpy(), rg.scale, rg.center)
    fus._tsdf, fus._tsdfw = T.cpu().numpy(), W.cpu().numpy()
    resident = fus.track(dm, lw0, None, None, rg.scale, rg.center)
    assert on_dev.lw.tobytes() == on_host.lw.tobytes() == resident.lw.tobytes()
    assert on_dev.iterations == on_host.iterations == resident.iterations
    assert on_host.residual is None and on_dev.residual.shape == (rg.rows, rg.cols)
    _, ro = otr.normal_eq(T.cpu().numpy(), W.cpu().numpy(), rg.res, rg.scale, rg.center, dm, rg.Kinv, on_dev.lw, 1, rg.tdist,
                          0.5 * rg.tdist, want_residual=True)
    assert np.array_equal(on_dev.residual.cpu().numpy().view(np.uint64), ro.view(np.uint64))
    assert pose_error(on_dev.lw, truth)[0] < 0.15
    with pytest.raises(ValueError, match="pixels"):
        fus.track(np.zeros_like(dm), lw0, T, W, rg.scale, rg.center)
    fus._vol = engine.DeviceVolume((64,) * 3, 0, 32, device=T.device, tsdf=T[:32], weight=W[:32])
    with pytest.raises(_capi.DfbError, match="slab"):
        fus.track(dm, lw0, None, None, rg.scale, rg.center)
    torch.cuda.synchronize()
