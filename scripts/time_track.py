"""Timing of rigid point-to-TSDF tracking (include/dfb.h dfb_track_normal_eq, FusionDM.track) on one GPU.  Writes one JSON file
(default profiles/r5_track.json) with the card name and power limit (queried, never set).

Workload: the body mesh on the test ring (tests/track_scenes.py), fused on the device by FusionDM.fuseDepths from the views at
-20 and +20 degrees into a 256^3 and a 512^3 volume; frames of 640x480.  dfb_track_normal_eq (both kernels and the 232-byte read
of the sums) is timed with CUDA events after warm-up at strides 1, 2 and 4; FusionDM.track is timed per frame with a host clock
around a synchronised call, tracking a frame rendered 2 degrees and res/64 voxels away from the starting pose."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "scripts")]
import torch

from dynamicfusion_body_b200 import engine
from dynamicfusion_body_b200.fusion import FusionDM
from time_render import card, event_ms
from track_scenes import Ring, perturb, pose_error


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_track.json"))
    ap.add_argument("--res", type=int, nargs="+", default=[256, 512])
    ap.add_argument("--reps", type=int, default=50)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    out = {"card": card(), "image": [480, 640], "reps": args.reps, "volumes": []}
    for res in args.res:
        rg = Ring(res, tdist=3.0 * res / 64)
        fus = FusionDM(rg.tdist, rg.K, tsdf_res=res)
        T = torch.full((res,) * 3, rg.tdist, dtype=torch.float32, device="cuda")
        W = torch.zeros((res,) * 3, dtype=torch.float32, device="cuda")
        for a in (-20.0, 20.0):
            fus.fuseDepths(rg.frame(rg.pose(a)), rg.pose(a), T, W, rg.scale, rg.center)
        lw0 = rg.pose(0.0)
        truth = perturb(lw0, 2.0, res / 64, 1)
        dm = rg.frame(truth)
        d = engine._to_dev(dm, torch.float32, T.device)
        rec = {"res": res, "normal_eq_ms": {}, "pixels": {}}
        for s in (1, 2, 4):
            n = int(engine._capi.lib().dfb_track_workspace_doubles(rg.rows, rg.cols, s))
            ws = torch.empty(n, dtype=torch.float64, device="cuda")
            call = lambda: engine.track_normal_eq((T, W), res, d, truth, rg.K, rg.Kinv, rg.scale, rg.center, s, rg.tdist,
                                                  0.5 * rg.tdist, workspace=ws)
            rec["normal_eq_ms"]["stride_%d" % s] = event_ms(call, args.reps)
            rec["pixels"]["stride_%d" % s] = int(call()[28])
        walls = []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = fus.track(dm, lw0, T, W, rg.scale, rg.center)
            torch.cuda.synchronize()
            walls.append((time.perf_counter() - t0) * 1e3)
        rec["track_ms_per_frame"] = {"min": min(walls[1:]), "median": sorted(walls[1:])[len(walls[1:]) // 2], "first": walls[0]}
        rec["track_iterations"] = list(r.iterations)
        rec["track_error_deg_voxel"] = [pose_error(r.lw, truth)[0], pose_error(r.lw, truth)[1] / rg.scale]
        out["volumes"].append(rec)
        print(json.dumps(rec), flush=True)
        del fus, T, W
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
