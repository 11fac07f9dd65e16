"""C-ABI level GPU tests of the one-launch frame step (dfb_frame_step_*) and the NCCL communicator (dfb_comm_*):
a captured / replayed / updated step must leave exactly the volume the plain dfb_tsdf_update_projective calls leave."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _scene(res=64, n_nodes=300):
    from dynamicfusion_body_b200 import synth
    return synth.make_scene(res=res, k=4, n_nodes=n_nodes, seed=3, rows=120, cols=160, background=True)


def _frames(sc, n):
    rng = np.random.default_rng(5)
    return [(sc.node_dq + (rng.normal(size=sc.node_dq.shape) * 1e-3).astype(np.float32)) for _ in range(n)]


def test_frame_step_graph_equals_direct_calls():
    import torch
    from dynamicfusion_body_b200 import engine
    sc = _scene()
    R = sc.res
    dev = torch.device("cuda", 0)
    dqs = [torch.from_numpy(d).to(dev) for d in _frames(sc, 4)]
    depth = torch.from_numpy(sc.depths).to(dev)
    # reference: plain calls on the default stream
    wf0 = engine.DeviceWarpField(4, dev)
    wf0.set_nodes(sc.node_pos, sc.node_dq, np.float32(sc.node_w))
    vol0 = engine.DeviceVolume((R, R, R), device=dev, fill=sc.tdist)
    for d in dqs:
        wf0.set_dq(d)
        engine.update_projective(vol0, wf0, sc.lw, depth, sc.K, sc.Kinv, sc.extrinsics, sc.tdist)
    lw2 = sc.lw.copy()
    lw2[5] += 0.01
    wf0.set_dq(dqs[0])
    engine.update_projective(vol0, wf0, lw2, depth, sc.K, sc.Kinv, sc.extrinsics, sc.tdist)
    torch.cuda.synchronize()
    # the same frames as graph launches on a capturable stream
    wf = engine.DeviceWarpField(4, dev)
    wf.set_nodes(sc.node_pos, sc.node_dq, np.float32(sc.node_w))
    vol = engine.DeviceVolume((R, R, R), device=dev, fill=sc.tdist)
    views = engine.make_views(depth, sc.K, sc.Kinv, sc.extrinsics)
    step = engine.FrameStep(vol, wf, sc.lw, views, sc.tdist)
    counters = torch.zeros(8, dtype=torch.int32).pin_memory()
    stage = torch.zeros((sc.n_nodes, 8), dtype=torch.float32).pin_memory()
    s = torch.cuda.Stream(device=dev)
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        for i, d in enumerate(dqs):
            if i < 2:                                  # transforms already on the device
                wf.node_dq.copy_(d)
                step.run(step.io(counters_host=counters))
            else:                                      # transforms uploaded from pinned host memory inside the graph
                s.synchronize()
                stage.copy_(d.cpu())
                step.run(step.io(dq_src=stage, counters_host=counters))
        s.synchronize()
        st = step.stats()
        assert st["captures"] == 2 and st["replays"] == 2 and st["direct"] == 0 and st["graph_nodes"] >= 6, st
        dev_counters = vol.workspace.counters.cpu().numpy()
        assert np.array_equal(counters.numpy(), dev_counters) and counters.numpy()[3] > 0
        # a new global rigid dq: the executable graph is updated in place
        step.set_lw(lw2)
        s.synchronize()
        stage.copy_(dqs[0].cpu())
        step.run(step.io(dq_src=stage, counters_host=counters))
        s.synchronize()
        st = step.stats()
        assert st["captures"] == 3 and st["updates"] == 1, st   # the upload node changed the topology (re-instantiated), the new lw only parameters
    assert torch.equal(vol.weight, vol0.weight)
    assert torch.equal(vol.tsdf, vol0.tsdf)
    # the legacy default stream cannot be captured: the step then issues its launches directly
    wf.node_dq.copy_(dqs[1]); wf0.set_dq(dqs[1])
    step.run(step.io())
    engine.update_projective(vol0, wf0, lw2, depth, sc.K, sc.Kinv, sc.extrinsics, sc.tdist)
    torch.cuda.synchronize()
    assert step.stats()["direct"] == 1
    assert torch.equal(vol.tsdf, vol0.tsdf) and torch.equal(vol.weight, vol0.weight)


def test_comm_single_rank_and_step_with_prefetch():
    """World-size-1 communicator through the C ABI (NCCL is initialised for real), broadcasts / reductions are identities, and
    the step's prefetch branch delivers the next frame's sensor data."""
    import torch
    from dynamicfusion_body_b200 import _capi, engine
    assert _capi.lib().dfb_comm_available() > 0
    dev = torch.device("cuda", 0)
    comm = engine.Comm(engine.Comm.unique_id(), 1, 0, dev)
    comm2 = engine.Comm(engine.Comm.unique_id(), 1, 0, dev)
    t = torch.arange(1000, dtype=torch.float64, device=dev)
    comm.allreduce_f64(t)
    comm.broadcast(t)
    torch.cuda.synchronize()
    assert torch.equal(t, torch.arange(1000, dtype=torch.float64, device=dev))
    sc = _scene(48, 200)
    R = sc.res
    depth_host = torch.from_numpy(sc.depths.copy()).pin_memory()
    packets = [torch.zeros(sc.depths.shape, dtype=torch.float32, device=dev) for _ in range(2)]
    wf = engine.DeviceWarpField(4, dev)
    wf.set_nodes(sc.node_pos, sc.node_dq, np.float32(sc.node_w))
    vol = engine.DeviceVolume((R, R, R), device=dev, fill=sc.tdist)
    steps = [engine.FrameStep(vol, wf, sc.lw, engine.make_views(packets[i], sc.K, sc.Kinv, sc.extrinsics), sc.tdist) for i in range(2)]
    s = torch.cuda.Stream(device=dev)
    packets[0].copy_(depth_host)
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        for i in range(4):
            slot = i & 1
            steps[slot].run(steps[slot].io(comm=comm, comm_prefetch=comm2, prefetch_dst=packets[slot ^ 1], prefetch_src=depth_host))
        s.synchronize()
    assert torch.equal(packets[1].cpu(), depth_host)
    wf0 = engine.DeviceWarpField(4, dev)
    wf0.set_nodes(sc.node_pos, sc.node_dq, np.float32(sc.node_w))
    vol0 = engine.DeviceVolume((R, R, R), device=dev, fill=sc.tdist)
    for i in range(4):
        engine.update_projective(vol0, wf0, sc.lw, packets[0], sc.K, sc.Kinv, sc.extrinsics, sc.tdist)
    torch.cuda.synchronize()
    assert torch.equal(vol.tsdf, vol0.tsdf) and torch.equal(vol.weight, vol0.weight)
    comm.close(); comm2.close()


def test_bench_dump_outputs_hold_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs writes the volume the timed path leaves after its last timed step: the same frames (warm-up +
    timed) through plain update calls give the same voxels bit for bit, and the JSON line counts the requested timed steps."""
    import json
    import os
    import subprocess
    import sys
    import torch
    import bench
    from dynamicfusion_body_b200 import engine
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res, nodes, steps, warmup = 64, 200, 2, 3
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
                          "--res", str(res), "--nodes", str(nodes), "--no-gn", "--no-configs", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])["steps"] == steps
    assert sorted(os.listdir(tmp_path)) == ["tsdf.npy", "weight.npy"]
    tsdf, weight = np.load(tmp_path / "tsdf.npy"), np.load(tmp_path / "weight.npy")
    assert tsdf.dtype == weight.dtype == np.float32 and tsdf.shape == weight.shape == (res ** 3,)
    sc = bench.build_scene(res, nodes, 4, 1)
    dqs = bench.frame_dqs(sc, 15)
    dev = torch.device("cuda", 0)
    wf = engine.DeviceWarpField(4, dev)
    wf.set_nodes(sc.node_pos, sc.node_dq, np.float32(sc.node_w))
    vol = engine.DeviceVolume((res, res, res), device=dev, fill=sc.tdist)
    depth = torch.from_numpy(sc.depths).to(dev)
    for i in range(warmup + steps):
        wf.set_dq(torch.from_numpy(dqs[i % len(dqs)]).to(dev))
        engine.update_projective(vol, wf, sc.lw, depth, sc.K, sc.Kinv, sc.extrinsics, sc.tdist)
    torch.cuda.synchronize()
    assert (weight > 0).any()
    assert np.array_equal(weight, vol.weight.cpu().numpy().ravel()) and np.array_equal(tsdf, vol.tsdf.cpu().numpy().ravel())
