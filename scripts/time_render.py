"""Timing of the z-buffer rasteriser (engine.render, include/dfb.h dfb_render) and of Fusion.render_live stage by stage, on one
GPU.  Writes one JSON file (default profiles/r4_render.json) with the card name and power limit (queried, never set).

Workload: the body scene at 256^3 and 512^3, fused from its 8 ring views of 640x480 (one fuseFrame call), surface extracted at
step 1 and warped to the live frame by the scene's field.  engine.render is timed on that mesh at 1 view and at the 8 ring
views; render_live is timed as a whole and split into extraction, kNN, warp and raster, each with CUDA events after warm-up."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from dynamicfusion_body_b200 import engine, synth
from dynamicfusion_body_b200.fusion import Fusion


def card():
    p = torch.cuda.get_device_properties(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:                                  # the numbers are still reported, marked as lacking the limit
        q = "unavailable (%s)" % e
    return {"name": p.name, "sms": p.multi_processor_count, "memory_gb": round(p.total_memory / 2**30, 1), "nvidia_smi_name_power_limit": q}


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


def fused(res):
    sc = synth.make_scene(res=res, k=4, n_nodes=1000, seed=0, n_views=8)
    fus = Fusion(sc.tdist, knn=sc.k, use_cnn=False, write_warpfield=False)
    fus.InitializeCanonicalSpace(tsdf_shape=(res,) * 3, K=sc.K, vertices=sc.vertices, normals=-sc.normals, faces=sc.faces,
                                 nodes=sc.nodes_as_reference_tuples(), radius=sc.radius)
    fus._lw = sc.lw
    fus.fuseFrame(sc.depths, extrinsics=sc.extrinsics)
    return sc, fus


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "r4_render.json"))
    ap.add_argument("--res", type=int, nargs="+", default=[256, 512])
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    out = {"card": card(), "image": [480, 640], "reps": args.reps, "volumes": []}
    for res in args.res:
        sc, fus = fused(res)
        k = sc.k
        v, f, _, _ = fus._device_surface(1, None, keep_on_device=True)
        idx = fus._wf.knn_points(v, k)
        live = engine.warp_points(fus._wf, fus._lw, v, idx=idx, k=k)
        rec = {"res": res, "vertices": int(v.shape[0]), "faces": int(f.shape[0]), "render_ms": {}, "large_face_pairs": {}, "covered": {}}
        for name, E in (("1_view", sc.extrinsics[:1]), ("8_views", sc.extrinsics)):
            views = engine.camera_views(sc.K, sc.rows, sc.cols, E)
            ws = engine.render_workspace(f.shape[0], views)
            rec["render_ms"][name] = event_ms(lambda: engine.render(live, f, views, workspace=ws), args.reps)
            depth, _, _ = engine.render(live, f, views, workspace=ws)
            rec["large_face_pairs"][name] = int(ws[0])
            rec["covered"][name] = float((depth != 0).double().mean())
        # render_live at the first ring camera (the object's K, one extrinsic), whole and stage by stage
        E1 = sc.extrinsics[:1]
        views = engine.camera_views(sc.K, sc.rows, sc.cols, E1)
        stages = {
            "extraction": lambda: fus._device_surface(1, None, keep_on_device=True),
            "knn": lambda: fus._wf.knn_points(v, k),
            "warp": lambda: engine.warp_points(fus._wf, fus._lw, v, idx=idx, k=k),
            "raster": lambda: engine.render(live, f, views),
        }
        rec["render_live_ms"] = {"total": event_ms(lambda: fus.render_live(extrinsics=E1), args.reps)}
        for name, fn in stages.items():
            rec["render_live_ms"][name] = event_ms(fn, args.reps)
        out["volumes"].append(rec)
        print(json.dumps(rec), flush=True)
        del fus
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
