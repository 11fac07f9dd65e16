"""Timing of raycasting the fused volume (include/dfb.h dfb_raycast, engine.raycast) on one GPU, beside the mesh path it replaces
for a FusionDM user (surface extraction, engine.marching_cubes at step 1 and level 0, then engine.render of the mesh) on the same
volume and poses.  Writes one JSON file (default profiles/r6_raycast.json) with the card name and power limit (queried, never set).

Workload: the body mesh on the test ring (tests/track_scenes.py), fused on the device by FusionDM.fuseDepths from the views at
-20 and +20 degrees into a 256^3 and a 512^3 volume; 640x480 images at 1 view (the 0-degree ring camera) and at 8 ring views;
step one voxel, z_far the default.  Every number is CUDA events around `reps` calls after warm-up; the volumes (64 MB and 512 MB
each for tsdf and weight at 256^3 / 512^3) are not flushed from L2 between calls, and the raycast reads only the voxels near
its rays."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "scripts")]
import numpy as np
import torch

from dynamicfusion_body_b200 import engine
from dynamicfusion_body_b200.fusion import FusionDM
from time_render import card, event_ms
from track_scenes import Ring


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_raycast.json"))
    ap.add_argument("--res", type=int, nargs="+", default=[256, 512])
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    out = {"card": card(), "image": [480, 640], "reps": args.reps, "step_voxels": 1.0, "volumes": []}
    for res in args.res:
        rg = Ring(res, tdist=3.0 * res / 64)
        fus = FusionDM(rg.tdist, rg.K, tsdf_res=res)
        T = torch.full((res,) * 3, rg.tdist, dtype=torch.float32, device="cuda")
        W = torch.zeros((res,) * 3, dtype=torch.float32, device="cuda")
        for a in (-20.0, 20.0):
            fus.fuseDepths(rg.frame(rg.pose(a)), rg.pose(a), T, W, rg.scale, rg.center)
        rec = {"res": res, "raycast_ms": {}, "hit_fraction": {}, "extract_ms": None, "render_ms": {}, "mesh_faces": None}
        ext = lambda: engine.marching_cubes(T, 1, level=0.0, keep_on_device=True)
        rec["extract_ms"] = event_ms(ext, args.reps)
        v, f, _, _ = ext()
        pts = rg.scale * (v.double() - res / 2.0) + torch.as_tensor(rg.center, device="cuda")
        rec["mesh_faces"] = int(f.shape[0])
        for name, E in (("1_view", np.stack([rg.pose(0.0)])), ("8_views", np.stack([rg.pose(-35.0 + 10.0 * i) for i in range(8)]))):
            views = engine.camera_views(rg.K, rg.rows, rg.cols, E)
            call = lambda: engine.raycast((T, W), res, views, rg.scale, rg.center, rg.tdist)
            rec["raycast_ms"][name] = event_ms(call, args.reps)
            rec["hit_fraction"][name] = float((call()[0] != 0).double().mean())
            ws = engine.render_workspace(f.shape[0], views)
            rec["render_ms"][name] = event_ms(lambda: engine.render(pts, f, views, workspace=ws), args.reps)
        rec["extract_plus_render_ms"] = {k: rec["extract_ms"] + r for k, r in rec["render_ms"].items()}
        out["volumes"].append(rec)
        print(json.dumps(rec), flush=True)
        del fus, T, W, v, f, pts
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
