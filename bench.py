#!/usr/bin/env python
"""bench.py -- headline benchmark of the warped-TSDF hot path (BASELINE.json metric:
"warped-TSDF voxels/sec ... (% HBM roofline); GN solve ms/iter").

  python bench.py --gpus 1 --steps 20 --warmup 5
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
         bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference ...          (CPU: the reference path restated in oracle/, all host cores)

A step = one frame of the a3 path over one GPU's slab: new depth frame + new node transforms ->
node records packed -> warped projective TSDF update (fast pass + reference-exact pass).
Workload at N=1: 512^3 voxels, ~4k nodes, k=4 DQB, one 640x480 depth view (north_star target config;
BASELINE configs[4] at one GPU).  N>1: weak scaling -- the grid is ~(512*N^(1/3))^3 (y/z a multiple of 32: 640 / 800 /
1024 at N = 2 / 4 / 8) so every rank owns an x-slab of >= 512^3 voxels of it; rank 0 broadcasts the depth views of the
next frame on a side stream and the node transforms inside the step, over NCCL.

`value`   : voxels/s with the frame already resident in HBM.
`e2e`     : voxels/s through the reference-facing class call (Fusion.fuseFrame) with HOST numpy buffers:
            H2D of depth + node transforms and D2H of the per-frame statistics are inside the timed region.
            The TSDF volume itself is persistent device state (Fusion._tsdf), as in the reference where it
            is an attribute that lives across frames.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALG_BYTES_PER_VOXEL = 16.0  # read v, read w, write v, write w (fp32) -- SURVEY 8d
DUMP_VOXELS = 4_000_000     # --dump-outputs: voxels sampled per array (2 float32 arrays, <= 32 MB in all)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
            return
        t0 = time.time()                       # nvidia-smi needs a moment before its first sample
        while time.time() - t0 < 5.0:
            try:
                if os.path.getsize(self.path) > 0:
                    break
            except OSError:
                pass
            time.sleep(0.02)
        self.skip = sum(1 for _ in open(self.path))   # samples taken before the timed region starts

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for ln, line in enumerate(open(self.path)):
                if ln < getattr(self, "skip", 0):
                    continue
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}
        return out


def dump_sample(n_voxels, dev):
    """Voxel indices that --dump-outputs writes: every voxel of a volume up to DUMP_VOXELS, else a fixed seeded sample (sorted,
    unique), so that two builds run with the same arguments dump the same voxels."""
    import torch
    if n_voxels <= DUMP_VOXELS:
        idx = np.arange(n_voxels)
    else:
        idx = np.unique(np.random.default_rng(0).integers(0, n_voxels, DUMP_VOXELS))
    return torch.from_numpy(idx).to(dev)


def build_scene(res, n_nodes, k, n_views, seed=0):
    from dynamicfusion_body_b200 import synth
    return synth.make_scene(res=res, k=k, n_nodes=n_nodes, seed=seed, n_views=n_views, background=True)


def frame_dqs(sc, n_frames, seed=1):
    """Per-frame node transforms: the scene's field plus a small per-frame perturbation (15-frame sequence shape)."""
    rng = np.random.default_rng(seed)
    return [(sc.node_dq + (rng.normal(size=sc.node_dq.shape) * 1e-4).astype(np.float32)) for _ in range(n_frames)]


# ------------------------------------------------------------------------------------------------------
class RankState:
    """Everything one rank needs to step its x-slab [x0, x1) of the grid: the drop-in Fusion object, the double-buffered frame
    packets, and one captured frame step (CUDA graph) per packet with its resident / end-to-end I/O descriptors."""

    def __init__(self, args, sc, grid, x0, x1, dev, rank, comm, comm_pre, frames):
        import torch
        from dynamicfusion_body_b200 import engine
        from dynamicfusion_body_b200 import dist as ddist
        from dynamicfusion_body_b200.fusion import Fusion
        self.x0, self.x1, self.rank, self.dev, self.sc, self.comm_pre = x0, x1, rank, dev, sc, comm_pre
        self.nvox = (x1 - x0) * grid[1] * grid[2]
        fus = Fusion(sc.tdist, knn=args.k, device=dev, use_cnn=False, write_warpfield=False)
        fus.InitializeCanonicalSpace(tsdf_shape=grid, slab=(x0, x1), K=sc.K, vertices=sc.vertices, normals=sc.normals,
                                     nodes=sc.nodes_as_reference_tuples())
        fus._lw = sc.lw
        self.fus, self.vol, self.wf = fus, fus._vol, fus._wf
        # graph revision: voxel kNN table + brick / region candidate sets (once per update_graph, core/fusion.py:229); the revision
        # kernels are loaded on a throw-away field first (the first launch of a kernel pays for loading its module)
        warm = engine.DeviceWarpField(args.k, dev)
        warm.set_nodes(sc.node_pos, sc.node_dq, np.float32(sc.node_w))
        warm.knn_table((32, 32, 32), 0, 32)
        warm.brick_nodes((32, 32, 32), 0, 32)
        del warm
        torch.cuda.synchronize()
        rev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        rev[0].record()
        fus.build_knn()
        rev[1].record()
        torch.cuda.synchronize()
        self.graph_revision_ms = ddist.max_over_ranks(rev[0].elapsed_time(rev[1]), dev)
        self.stream = torch.cuda.Stream(device=dev)      # a capturable (non-default) stream: the step is one CUDA-graph launch
        shape = sc.depths.shape
        self.frames = frames
        self.packets = [torch.zeros(shape, dtype=torch.float32, device=dev) for _ in range(2)]
        self.dq_stage = [torch.zeros((sc.n_nodes, 8), dtype=torch.float32).pin_memory() for _ in range(2)]
        self.counters_host = [torch.zeros(8, dtype=torch.int32).pin_memory() for _ in range(2)]
        self.slot_done = [torch.cuda.Event(), torch.cuda.Event()]
        self.steps, self.ios_res, self.ios_e2e, self.ios_nobcast, self.ios_local = [], [], [], [], []
        for slot in range(2):
            views = engine.make_views(self.packets[slot], sc.K, sc.Kinv, sc.extrinsics)
            st = engine.FrameStep(self.vol, self.wf, sc.lw, views, sc.tdist)
            self.steps.append(st)
            # resident frame: the transforms are already in wf.node_dq on the root, the next depth frame is a device buffer
            self.ios_res.append(st.io(comm=comm, comm_prefetch=comm_pre, root=0, prefetch_dst=self.packets[slot ^ 1], prefetch_src=frames["depth_dev"]))
            # end to end: transforms and depth come from pinned host memory, the counters go back to pinned host memory
            self.ios_e2e.append(st.io(comm=comm, comm_prefetch=comm_pre, root=0, dq_src=self.dq_stage[slot], prefetch_dst=self.packets[slot ^ 1],
                                      prefetch_src=frames["depth_host"], counters_host=self.counters_host[slot]))
            # limiter analysis (N > 1): the same step without the in-step transform broadcast / without any communication
            self.ios_nobcast.append(st.io(comm=None, comm_prefetch=comm_pre, root=0, prefetch_dst=self.packets[slot ^ 1], prefetch_src=frames["depth_dev"]))
            self.ios_local.append(st.io())

    def reset(self):
        self.vol.tsdf.fill_(self.sc.tdist)
        self.vol.weight.zero_()

    def prime(self, src):
        """frame 0's sensor data into packet 0 (every later frame arrives through the prefetch branch of the step before it)"""
        import torch
        with torch.cuda.stream(self.stream):
            if self.rank == 0:
                self.packets[0].copy_(src, non_blocking=True)
            if self.comm_pre is not None:
                self.comm_pre.broadcast(self.packets[0])
        self.stream.synchronize()

    def step_resident(self, i):
        import torch
        slot = i & 1
        with torch.cuda.stream(self.stream):
            if self.rank == 0:
                self.wf.node_dq.copy_(self.frames["dq_dev"][i % len(self.frames["dq_dev"])], non_blocking=True)
            self.steps[slot].run(self.ios_res[slot])

    def step_with(self, ios, all_ranks_own_transforms=True):
        """step function over another set of I/O descriptors (limiter analysis): every rank copies the frame's transforms itself"""
        import torch

        def f(i):
            slot = i & 1
            with torch.cuda.stream(self.stream):
                self.wf.node_dq.copy_(self.frames["dq_dev"][i % len(self.frames["dq_dev"])], non_blocking=True)
                self.steps[slot].run(ios[slot])
        return f

    def step_e2e(self, i):
        import torch
        slot = i & 1
        self.slot_done[slot].synchronize()                             # step i-2 has consumed this slot's staging buffers
        stats = self.counters_host[slot].numpy().copy()                # D2H result of step i-2, read on the host
        if self.rank == 0:
            self.dq_stage[slot].numpy()[...] = self.frames["dqs"][i % len(self.frames["dqs"])]   # host -> pinned staging (the solver's output)
        with torch.cuda.stream(self.stream):
            self.steps[slot].run(self.ios_e2e[slot])
            self.slot_done[slot].record()
        return stats

    def timed(self, step_fn, steps, warmup, src, barrier, per_rank=False):
        import torch
        from dynamicfusion_body_b200 import dist as ddist
        self.prime(src)
        for i in range(warmup):
            step_fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for i in range(warmup, warmup + steps):
            step_fn(i)
        e1.record(self.stream)
        barrier()
        if per_rank:
            return e0.elapsed_time(e1)
        return ddist.max_over_ranks(e0.elapsed_time(e1), self.dev)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from dynamicfusion_body_b200 import _capi, engine
    from dynamicfusion_body_b200 import dist as ddist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run for --gpus > 1")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs is implemented for one GPU")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # STRONG scaling (BASELINE configs[4]): ONE res^3 grid, one x-slab per rank
    res = args.res
    grid = (res, res, res)
    sc = build_scene(res, args.nodes, args.k, args.views)
    nvox_total = res ** 3
    n_frames = 15
    dqs = frame_dqs(sc, n_frames)
    frames = {"dqs": dqs, "dq_dev": [torch.from_numpy(d).to(dev) for d in dqs], "depth_dev": torch.from_numpy(sc.depths.copy()).to(dev),
              "depth_host": torch.from_numpy(sc.depths.copy()).pin_memory()}
    depth_dev, depth_host, dq_dev = frames["depth_dev"], frames["depth_host"], frames["dq_dev"]

    # communicators (raw NCCL through the C ABI): one for the in-step transform broadcast, one for the sensor prefetch
    comm = comm_pre = None
    if world > 1:
        comm = engine.Comm.from_torch(dev)
        comm_pre = engine.Comm.from_torch(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    parts_equal = ddist.slab_partition(res, world)
    st = RankState(args, sc, grid, parts_equal[rank][0], parts_equal[rank][1], dev, rank, comm, comm_pre, frames)
    partition = {"kind": "equal", "slabs": parts_equal}
    equal_info = None
    if world > 1:
        # the step time of a sharded volume is the maximum over ranks: measure the equal slabs, then move the slab boundaries
        # (multiples of 16 planes) so that the estimated cost -- brick classes of a frame -- is the same on every rank
        UNIT = 4                                                       # slab boundaries on brick layers (4 planes)
        ms_eq = st.timed(st.step_resident, args.steps, args.warmup, depth_dev, barrier)
        equal_info = {"ms_per_step": ms_eq / args.steps, "value": nvox_total * args.steps / (ms_eq * 1e-3), "slabs": parts_equal}
        if not args.equal_slabs:
            parts = parts_equal
            for rnd in range(2):
                # cost of every 4-plane layer from the brick classes of a frame, rescaled per rank by what the rank's step really
                # takes on its own (no communication) minus the per-step floor -- the second round corrects the first one's model
                prof = engine.slab_cost_profile(st.vol, UNIT)
                t_local = st.timed(st.step_with(st.ios_local), max(10, args.steps // 2), 3, depth_dev, barrier, per_rank=True) / max(10, args.steps // 2)
                floor_ms = 0.03
                scale = max(t_local - floor_ms, 0.2 * t_local) / max(float(prof.sum()), 1e-9)
                gathered = [None] * world
                dist.all_gather_object(gathered, (prof * scale).tolist())
                unit_cost = np.concatenate([np.asarray(g) for g in gathered])[:res // UNIT]
                new_parts = ddist.balanced_slab_partition(unit_cost, world, UNIT, res)
                if rnd == 0:
                    equal_info["rank_compute_ms"] = [float(np.sum(g)) + floor_ms for g in gathered]
                if new_parts == parts:
                    break
                parts = new_parts
                del st
                torch.cuda.empty_cache()
                st = RankState(args, sc, grid, parts[rank][0], parts[rank][1], dev, rank, comm, comm_pre, frames)
                st.timed(st.step_resident, 3, 2, depth_dev, barrier)   # a few frames so that the brick classes exist
            if parts != parts_equal:
                partition = {"kind": "balanced", "slabs": parts,
                             "how": "x-slab boundaries on brick layers (multiples of 4 planes) minimising the largest slab cost; cost per layer = "
                                    "brick classes of a frame (0.6 / 1.6 / 10.7 per brick / CLAMP brick / MIXED brick) scaled by the measured "
                                    "compute time of the rank that owned the layer, two rounds"}
        st.reset()
    x0, x1 = st.x0, st.x1
    nvox_rank = st.nvox
    fus = st.fus

    # ---- untimed parity check on the hardware (N > 1): slabs gathered over NCCL == a single-volume run on rank 0 ----
    parity = None
    if world > 1:
        parity = parity_check(args, sc, st, partition["slabs"], comm, rank, world, dev)
        st.reset()

    dump_idx = dump_sample(nvox_rank, dev) if args.dump_outputs else None
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_total = st.timed(st.step_resident, args.steps, args.warmup, depth_dev, barrier)
    dumped = None
    if dump_idx is not None:
        # what a caller of the timed path receives: the (tsdf, weight) volume after the last timed step, gathered before any
        # later (untimed) step changes it
        dumped = {"tsdf": st.vol.tsdf.view(-1)[dump_idx], "weight": st.vol.weight.view(-1)[dump_idx]}
        torch.cuda.synchronize()
    # the K timed steps last only a few tens of ms; keep the same step running (untimed, identical count on every rank so
    # that the collectives match) until the 20 ms sampler has seen ~0.4 s of this load
    n_extra = max(0, int(400.0 / max(ms_total / args.steps, 1e-3)) - args.steps)
    for i in range(min(n_extra, 4000)):
        st.step_resident(i)
        if i % 64 == 63:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    limiter = None
    if world > 1:
        # where the N-GPU step goes: (a) every rank's own compute (no communication at all; each rank uploads the transforms itself),
        # (b) the step with the sensor prefetch but without the in-step transform broadcast, (c) the real step
        ms_local = st.timed(st.step_with(st.ios_local), args.steps, args.warmup, depth_dev, barrier, per_rank=True) / args.steps
        allms = [None] * world
        dist.all_gather_object(allms, float(ms_local))
        ms_nob = st.timed(st.step_with(st.ios_nobcast), args.steps, args.warmup, depth_dev, barrier) / args.steps
        step_now = ms_total / args.steps
        limiter = {"step_ms": step_now, "rank_compute_ms": allms, "max_rank_compute_ms": max(allms), "mean_rank_compute_ms": float(np.mean(allms)),
                   "step_without_transform_broadcast_ms": ms_nob, "transform_broadcast_on_critical_path_ms": step_now - ms_nob,
                   "prefetch_branch_and_rank_skew_ms": ms_nob - max(allms),
                   "note": "rank_compute = one CUDA-graph launch per step of [node records, counters memset, region bounds, brick classify, "
                           "update, exact] on the rank's slab, no communication; an N-th of the one-GPU step would be the ideal"}
    for e in st.slot_done:
        e.record(st.stream)
    ms_e2e = st.timed(st.step_e2e, args.steps, max(3, args.warmup // 2), depth_host, barrier)
    stats = fus.frame_stats()
    gstats = st.steps[0].stats()

    # ---- roofline leg: every kernel of the step timed alone with CUDA events on its stream ----
    kk = 4 if args.k <= 4 else 8
    # the update pass as tsdf.cu dispatches it: node table in shared memory (TMA) for several views or k > 4, global records otherwise
    upd_name = ("brick_update_smem_kernel<%d>" % kk) if (sc.depths.shape[0] > 1 or args.k > 4) else ("brick_update_kernel<%d, 1, 1>" % kk)
    prod = [("region_bounds_kernel+brick_classify_kernel", _capi.MODE_BRICK_CLASSIFY), (upd_name, _capi.MODE_BRICK_UPDATE),
            ("proj_exact_kernel<%d>" % kk, _capi.MODE_LIST_ONLY)]
    parts = [("region_bounds_kernel+brick_classify_kernel", _capi.MODE_BRICK_CLASSIFY), ("brick_stream_kernel", _capi.MODE_BRICK_STREAM),
             ("brick_mixed_kernel<%d>" % kk, _capi.MODE_BRICK_MIXED)]

    def time_modes(seq, reps):
        acc = {n: [] for n, _ in seq}
        for i in range(reps):
            fus.set_node_dqs(dq_dev[i % n_frames])
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(seq) + 1)]
            ev[0].record()
            for j, (n, mode) in enumerate(seq):
                fus.fuseFrame(depth_dev, extrinsics=sc.extrinsics, mode=mode)
                ev[j + 1].record()
            torch.cuda.synchronize()
            for j, (n, _) in enumerate(seq):
                acc[n].append(ev[j].elapsed_time(ev[j + 1]))
        return {n: float(np.mean(v[2:])) for n, v in acc.items()}

    reps = max(6, min(args.steps, 20))
    kms = time_modes(prod, reps)
    stats = fus.frame_stats()
    pms = time_modes(parts, reps)
    vox_per_brick = 4 * 4 * 32
    n_stream, n_mixed = stats["bricks_streamed"] * vox_per_brick, stats["bricks_mixed"] * vox_per_brick
    units = {prod[0][0]: 0, prod[1][0]: n_stream + n_mixed, prod[2][0]: stats["deferred"]}
    punits = {parts[1][0]: n_stream, parts[2][0]: n_mixed}
    names = prod
    # dominant = the slowest kernel that moves volume data (the classifier reads 48 B per brick, no voxels)
    dominant = max([n for n, _ in prod[1:]], key=kms.get)
    value = nvox_total * args.steps / (ms_total * 1e-3)
    e2e_value = nvox_total * args.steps / (ms_e2e * 1e-3)
    peak, peak_src = measured_peaks()
    step_ms = ms_total / args.steps
    kernels = [{"kernel": n, "ms": kms[n], "voxels": int(units[n]),
                "achieved_GBps": ALG_BYTES_PER_VOXEL * units[n] / (kms[n] * 1e-3) / 1e9,
                "frac": ALG_BYTES_PER_VOXEL * units[n] / (kms[n] * 1e-3) / 1e9 / peak} for n, _ in names]
    kernels += [{"kernel": n + " (half of the fused pass, timed alone)", "ms": pms[n], "voxels": int(punits[n]),
                 "achieved_GBps": ALG_BYTES_PER_VOXEL * punits[n] / (pms[n] * 1e-3) / 1e9,
                 "frac": ALG_BYTES_PER_VOXEL * punits[n] / (pms[n] * 1e-3) / 1e9 / peak} for n, _ in parts[1:]]
    achieved = ALG_BYTES_PER_VOXEL * units[dominant] / (kms[dominant] * 1e-3) / 1e9
    step_achieved = ALG_BYTES_PER_VOXEL * nvox_rank / (step_ms * 1e-3) / 1e9
    traffic = measured_traffic(dominant) if world == 1 else None
    slab_mb = nvox_rank * (8 + 2 * args.k) / 1e6
    out = {
        "metric": "warped_tsdf_voxels_per_sec", "value": value, "unit": "voxels/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "%d^3 voxels total (ONE grid, %s x-slabs over %d GPU(s): %s), warped projective TSDF update (a3), k=%d DQB, "
                               "%d nodes, %d view(s) 640x480, 15-frame dq sequence"
                               % (res, partition["kind"], world, "/".join(str(b - a) for a, b in partition["slabs"]), args.k, sc.n_nodes, args.views),
                   "l2": ("inputs larger than L2 (%.0f MB of v,w,kNN per GPU)" % slab_mb) if slab_mb > 250 else
                         ("slab of %.0f MB (v,w,kNN) per GPU, each step streams it once: a 512^3/N slab approaches the 126 MB L2 from N=4 on, "
                          "so part of it is served from L2 -- that is the configuration BASELINE configs[4] names" % slab_mb),
                   "parallelism": ("one CUDA-graph launch per rank and step: NCCL broadcast of the node transforms (dfb_comm, raw NCCL) -> node "
                                   "records -> classify / update / exact kernels, next depth frame broadcast as a concurrent graph branch")
                                  if world > 1 else "single GPU, one CUDA-graph launch per step",
                   "partition": partition,
                   "deferred_voxel_fraction": stats["deferred"] / nvox_rank,
                   "dqb_voxel_fraction_of_mixed": stats.get("dqb_voxels", 0) / max(1, n_mixed)},
        "e2e": {"value": e2e_value, "unit": "voxels/s", "h2d_bytes_per_step": int(sc.depths.nbytes + dqs[0].nbytes),
                "d2h_bytes_per_step": 32, "ms_per_step": ms_e2e / args.steps,
                "pipeline": "per step: host copies the frame's node transforms into pinned staging, ONE graph launch = [H2D transforms -> "
                            "(NCCL bcast) -> node records -> classify/update/exact kernels -> D2H of the 8 frame counters] with the H2D (+bcast) "
                            "of the next frame's pinned depth image as a concurrent branch; the host reads step t-2's counters before "
                            "re-using its slot; every step's H2D and D2H lie inside the timed region"},
        "gpu_launches": 5 * args.steps,
        "step_graph": gstats,
        "clocks": clocks,
        "graph_revision_ms": st.graph_revision_ms,
        "value_amortised": {"revision_every_frame": nvox_total / ((step_ms + st.graph_revision_ms) * 1e-3),
                            "revision_every_15_frames": nvox_total / ((step_ms + st.graph_revision_ms / 15.0) * 1e-3),
                            "note": "the reference rebuilds its KD-tree in update_graph (core/fusion.py:229) and queries it per voxel per frame "
                                    "(:175); here the voxel kNN table + brick/region sets belong to a graph revision: `graph_revision_ms` is "
                                    "the FULL rebuild, `graph_revision_incremental` the update after +1 % appended nodes; `value` excludes both"},
        "roofline": {"bound": "hbm", "kernel": dominant, "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic,
                     "note": "dominant kernel by time; its units = the voxels that launch processes x 16 B. The step as a whole "
                             "(all voxels of the slab x 16 B / step time) is in `step`.",
                     "algorithmic_bytes_per_voxel": ALG_BYTES_PER_VOXEL,
                     "step": {"achieved": step_achieved, "frac": step_achieved / peak, "ms": step_ms},
                     "kernels": kernels,
                     "bricks": {"total": stats["bricks"], "streamed": stats["bricks_streamed"], "mixed": stats["bricks_mixed"]}},
    }
    if equal_info is not None:
        out["equal_slabs"] = equal_info
    if parity is not None:
        out["parity_check"] = parity
    if limiter is not None:
        out["limiter"] = limiter
    def leg(name, fn):
        """the extra legs must never cost the headline line"""
        try:
            out[name] = fn()
        except Exception as e:                                   # pragma: no cover
            import traceback
            out[name] = {"error": "%s: %s" % (type(e).__name__, e), "trace": traceback.format_exc()[-600:]}

    if world == 1 and not args.no_configs:
        leg("graph_revision_incremental", lambda: bench_incremental_revision(sc, st))
    del st
    torch.cuda.empty_cache()
    if world == 1 and not args.no_configs:
        leg("configs", lambda: bench_configs(args, dev))
        leg("frame_loop", lambda: bench_frame_loop(args, dev))
    if not args.no_gn:
        out["gn"] = bench_gn(args, dev, rank, world, comm)
        leg("gn_depth_frame", lambda: bench_gn_depth_frame(args, dev, rank, world, comm))
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(sc, grid, budget_s=args.cpu_seconds)
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), t.cpu().numpy())
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def measured_traffic(kernel_name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed ncu --set full summary of
    THIS round's kernels (profiles/r2_ncu_full_summary.md, same 512^3 N=1 workload); None when no capture of that kernel is committed."""
    import re
    path = os.path.join(ROOT, "profiles", "r2_ncu_full_summary.md")
    if not os.path.isfile(path):
        return None
    base = kernel_name.split("<")[0]
    # the summary may hold several captures of the kernel (the full grid and one rank's slab): the longest launch is the full grid
    best, cur = None, None
    for line in open(path):
        if line.startswith("## "):
            cur = {"ms": 0.0} if base in line else None
            if cur is not None and (best is None or best.get("rd") is None):
                best = best or cur
        elif cur is not None:
            m = re.match(r"- gpu__time_duration\.sum = ([0-9.]+) (\w+)", line)
            if m:
                cur["ms"] = float(m.group(1)) * {"ms": 1.0, "us": 1e-3, "ns": 1e-6, "s": 1e3}.get(m.group(2), 1.0)
            m = re.match(r"- dram__bytes_(read|write)\.sum = ([0-9.]+) (\w+)", line)
            if m:
                mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(m.group(3), 1.0)
                cur["rd" if m.group(1) == "read" else "wr"] = float(m.group(2)) * mult
                if "rd" in cur and "wr" in cur and (best is None or "rd" not in best or cur["ms"] > best["ms"]):
                    best = cur
    rd, wr = (best or {}).get("rd"), (best or {}).get("wr")
    return None if rd is None or wr is None else int(rd + wr)


def parity_check(args, sc, st, parts, comm, rank, world, dev):
    """Three frames on the sharded volume (through the timed path: graph launches + NCCL broadcasts) against the same three
    frames on a single res^3 volume held by rank 0; slabs are gathered over NCCL (dfb_comm_sendrecv).  SURVEY 8e: weights and values
    must be equal bit for bit."""
    import torch
    from dynamicfusion_body_b200 import engine
    res = args.res
    vol, wf = st.vol, st.wf
    st.reset()
    st.prime(st.frames["depth_dev"])
    n_chk = 3
    for i in range(n_chk):
        st.step_resident(i)
    st.stream.synchronize()
    torch.cuda.synchronize()
    result = None
    if rank == 0:
        full_t = torch.empty((res, res, res), dtype=torch.float32, device=dev)
        full_w = torch.empty_like(full_t)
        full_t[parts[0][0]:parts[0][1]] = vol.tsdf
        full_w[parts[0][0]:parts[0][1]] = vol.weight
        for r in range(1, world):
            a, b = parts[r]
            comm.sendrecv(recv=full_t[a:b], recv_peer=r)
            comm.sendrecv(recv=full_w[a:b], recv_peer=r)
        torch.cuda.synchronize()
        # the same frames on one volume
        wf1 = engine.DeviceWarpField(args.k, dev)
        wf1.set_nodes(sc.node_pos, sc.node_dq, np.float32(sc.node_w))
        vol1 = engine.DeviceVolume((res, res, res), device=dev, fill=sc.tdist)
        for i in range(n_chk):
            wf1.set_dq(st.frames["dq_dev"][i])
            engine.update_projective(vol1, wf1, sc.lw, st.frames["depth_dev"], sc.K, sc.Kinv, sc.extrinsics, sc.tdist)
        torch.cuda.synchronize()
        w_equal = bool(torch.equal(full_w, vol1.weight))
        v_equal = bool(torch.equal(full_t, vol1.tsdf))
        max_diff = float((full_t - vol1.tsdf).abs().max().item())
        updated = int((vol1.weight > 0).sum().item())
        result = {"tsdf": "ok" if (w_equal and v_equal) else "MISMATCH", "frames": n_chk, "weights_bit_equal": w_equal, "values_bit_equal": v_equal,
                  "max_abs_value_diff": max_diff, "updated_voxels": updated,
                  "how": "slabs gathered on rank 0 over NCCL vs the same frames on one %d^3 volume" % res}
        del full_t, full_w, vol1, wf1
        torch.cuda.empty_cache()
    else:
        comm.sendrecv(send=vol.tsdf, send_peer=0)
        comm.sendrecv(send=vol.weight, send_peer=0)
        torch.cuda.synchronize()
    return result


def _event_ms(fn, reps, warm=2):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def bench_incremental_revision(sc, st):
    """A graph revision that appends 1 % new nodes (what update_graph does): incremental update of the kNN table + brick / region
    sets against the full rebuild.  The new nodes are surface points between existing nodes."""
    import torch
    from dynamicfusion_body_b200 import engine
    rng = np.random.default_rng(7)
    m = max(1, sc.n_nodes // 100)
    warm = engine.DeviceWarpField(st.wf.k, st.dev)                     # load the revision kernels on a throw-away field first
    warm.set_nodes(sc.node_pos[:-m], sc.node_dq[:-m], np.float32(sc.node_w))
    warm.brick_nodes((64, 64, 64), 0, 64)
    warm.append_nodes(sc.node_pos[-m:], sc.node_dq[-m:], np.float32(sc.node_w))
    del warm
    sel = rng.choice(len(sc.vertices), m, replace=False)
    new_pos = sc.vertices[sel].astype(np.float32)
    new_dq = np.tile(np.array([1, 0, 0, 0, 0, 0, 0, 0], np.float32), (m, 1))
    wf = st.wf
    res, x0, x1 = st.vol.res, st.vol.x0, st.vol.x1
    torch.cuda.synchronize()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    e[0].record()
    wf.append_nodes(new_pos, new_dq, np.float32(sc.node_w))
    e[1].record()
    torch.cuda.synchronize()
    dirty = float(wf.last_dirty.float().mean().item())
    ref = engine.DeviceWarpField(wf.k, st.dev)
    ref.set_nodes(wf.node_pos, wf.node_dq, wf.node_w)
    same = bool(torch.equal(ref.knn_table(res, x0, x1), wf.knn_table(res, x0, x1)))
    del ref
    return {"new_nodes": m, "ms": e[0].elapsed_time(e[1]), "dirty_8cube_bricks_fraction": dirty, "knn_table_equals_full_rebuild": same,
            "full_rebuild_ms": st.graph_revision_ms}


def bench_configs(args, dev):
    """The other BASELINE configs on one GPU (the driver only runs the default command).  256^3 volumes are 134 MB of (v, w): four
    volumes are rotated so that a frame never finds its volume in the 126 MB L2 (SURVEY 7 'honest HBM numbers')."""
    import torch
    from dynamicfusion_body_b200 import engine, synth
    peak, _ = measured_peaks()
    out = {}
    R = 256
    nvox = R ** 3
    n_rot = 4

    def line(ms, views=1, extra=None):
        d = {"ms_per_frame": ms, "voxels_per_s": nvox / (ms * 1e-3), "voxel_updates_per_s": views * nvox / (ms * 1e-3),
             "roofline_frac_16B_per_voxel": ALG_BYTES_PER_VOXEL * nvox / (ms * 1e-3) / 1e9 / peak, "rotating_volumes": n_rot}
        d.update(extra or {})
        return d

    # configs[1]: 256^3, 1 view per frame, ~1k nodes, k=4, 15-frame sequence
    sc = synth.make_scene(res=R, k=4, n_nodes=1000, seed=0, background=True)
    dqs = [torch.from_numpy(d).to(dev) for d in frame_dqs(sc, 15)]
    wf = engine.DeviceWarpField(4, dev)
    wf.set_nodes(sc.node_pos, sc.node_dq, np.float32(sc.node_w))
    vols = [engine.DeviceVolume((R, R, R), device=dev, fill=sc.tdist) for _ in range(n_rot)]
    depth = torch.from_numpy(sc.depths).to(dev)
    views = engine.make_views(depth, sc.K, sc.Kinv, sc.extrinsics)
    wf.brick_nodes((R, R, R), 0, R)
    it = {"i": 0}

    def a3():
        i = it["i"]; it["i"] += 1
        wf.set_dq(dqs[i % 15])
        engine.update_projective(vols[i % n_rot], wf, sc.lw, depth, sc.K, sc.Kinv, sc.extrinsics, sc.tdist, views=views)
    ms = _event_ms(a3, 30, 8)
    stt = vols[0].workspace.stats()
    out["c2_a3_256"] = line(ms, extra={"path": "Fusion.fuseFrame (a3: warp + projective update), %d nodes k=4, 1 view" % sc.n_nodes,
                                       "deferred_fraction": stt["deferred"] / nvox, "bricks_mixed_fraction": stt["bricks_mixed"] / stt["bricks"]})
    # the same frame with the camera along x and y: every other scene looks along z, the long axis of the 4x4x32 bricks (VERDICT r1)
    axes = {"z": {"ms_per_frame": ms, "bricks_mixed_fraction": stt["bricks_mixed"] / stt["bricks"], "deferred_fraction": stt["deferred"] / nvox}}
    for ax in ("x", "y"):
        sa = synth.make_scene(res=R, k=4, n_nodes=1000, seed=0, background=True, view_axis=ax)
        da = torch.from_numpy(sa.depths).to(dev)
        va = engine.make_views(da, sa.K, sa.Kinv, sa.extrinsics)

        def a3x():
            i = it["i"]; it["i"] += 1
            wf.set_dq(dqs[i % 15])
            engine.update_projective(vols[i % n_rot], wf, sa.lw, da, sa.K, sa.Kinv, sa.extrinsics, sa.tdist, views=va)
        msa = _event_ms(a3x, 30, 8)
        sta = vols[0].workspace.stats()
        axes[ax] = {"ms_per_frame": msa, "bricks_mixed_fraction": sta["bricks_mixed"] / sta["bricks"], "deferred_fraction": sta["deferred"] / nvox}
    out["c2_a3_256"]["view_axes"] = axes
    # configs[1] as profiled by the reference (profiles/updateTSDF_*): Fusion.updateTSDF against a live TSDF VOLUME (a1)
    nw = np.full(sc.n_nodes, np.float32(sc.node_w))
    wv = synth.blend_warp(sc.vertices, sc.node_pos, sc.node_dq, nw, sc.vert_knn, lw=None)
    t0 = time.time()
    sdf = synth.mesh_sdf_volume((R, R, R), wv, sc.normals)             # untruncated, as test.py:105-110 loads it
    sdf_s = time.time() - t0
    live_raw = torch.from_numpy(sdf).to(dev)
    # a live volume as FusionDM / fuseFrame leave it: the band around the surface, +tdist (the initial value) everywhere else --
    # such volumes never hold -tdist (voxels behind the band are simply not updated, core/fusion_dm.py:203)
    live_trunc = torch.from_numpy(np.where(sdf < -sc.tdist, np.float32(sc.tdist), np.minimum(sdf, np.float32(sc.tdist))).astype(np.float32)).to(dev)
    for name, live, td, what in (("c2_a1_256_reference_usage", live_raw, float(sdf.max()),
                                  "Fusion.updateTSDF, untruncated live SDF with trunc_distance = volume.max() (test.py:110): every voxel lies inside the "
                                  "band and takes the reference-exact float64 tier"),
                                 ("c2_a1_256_truncated", live_trunc, sc.tdist,
                                  "Fusion.updateTSDF, live TSDF as FusionDM / fuseFrame volumes hold it (band around the surface, +tdist elsewhere)")):
        vs = [engine.DeviceVolume((R, R, R), device=dev, fill=td) for _ in range(n_rot)]
        it["i"] = 0

        def a1():
            i = it["i"]; it["i"] += 1
            wf.set_dq(dqs[i % 15])
            engine.update_volume(vs[i % n_rot], wf, None, live, td)
        ms = _event_ms(a1, 8, 3)
        stt = vs[0].workspace.stats()
        out[name] = line(ms, extra={"path": what, "deferred_fraction": stt["deferred"] / nvox})
        del vs
    out["c2_a1_256_reference_usage"]["live_sdf_synthesis_s"] = sdf_s
    del vols, wf, live_raw, live_trunc
    torch.cuda.empty_cache()
    # configs[3]: 8 synthetic depth views per frame fused into a 256^3 TSDF with k=8 DQB
    sc8 = synth.make_scene(res=R, k=8, n_nodes=1000, seed=0, background=True, n_views=8)
    dqs8 = [torch.from_numpy(d).to(dev) for d in frame_dqs(sc8, 15)]
    wf8 = engine.DeviceWarpField(8, dev)
    wf8.set_nodes(sc8.node_pos, sc8.node_dq, np.float32(sc8.node_w))
    vols8 = [engine.DeviceVolume((R, R, R), device=dev, fill=sc8.tdist) for _ in range(n_rot)]
    depth8 = torch.from_numpy(sc8.depths).to(dev)
    views8 = engine.make_views(depth8, sc8.K, sc8.Kinv, sc8.extrinsics)
    wf8.brick_nodes((R, R, R), 0, R)
    it["i"] = 0

    def a3v8():
        i = it["i"]; it["i"] += 1
        wf8.set_dq(dqs8[i % 15])
        engine.update_projective(vols8[i % n_rot], wf8, sc8.lw, depth8, sc8.K, sc8.Kinv, sc8.extrinsics, sc8.tdist, views=views8)
    ms = _event_ms(a3v8, 20, 6)
    stt = vols8[0].workspace.stats()
    out["c4_8view_k8_256"] = line(ms, views=8, extra={"path": "Fusion.fuseFrame, 8 views (ring of cameras) fused in ONE pass, %d nodes k=8" % sc8.n_nodes,
                                                      "deferred_fraction": stt["deferred"] / nvox,
                                                      "bricks_mixed_fraction": stt["bricks_mixed"] / stt["bricks"]})
    del vols8, wf8
    torch.cuda.empty_cache()
    return out


def bench_frame_loop(args, dev):
    """The reference's frame loop (test.py:125-131: setupCorrespondences -> solve -> TSDF update -> update_graph) through the drop-in
    Fusion object at 256^3 / ~1k nodes: wall time per stage, host work and synchronisations included."""
    import torch
    from dynamicfusion_body_b200 import synth
    from dynamicfusion_body_b200.fusion import Fusion
    R = 256
    sc = synth.make_scene(res=R, k=4, n_nodes=1000, seed=0, background=True)
    fus = Fusion(sc.tdist, knn=4, device=dev, use_cnn=False, write_warpfield=False)
    fus.InitializeCanonicalSpace(tsdf_shape=(R, R, R), K=sc.K, vertices=sc.vertices, normals=sc.normals, faces=sc.faces,
                                 nodes=sc.nodes_as_reference_tuples(), radius=sc.radius)
    fus._lw = sc.lw
    live = sc.warped_vertices.astype(np.float32)
    depth = torch.from_numpy(sc.depths).to(dev)
    fus.build_knn()
    fus.fuseFrame(depth, extrinsics=sc.extrinsics)                     # a first frame so that the volume holds a surface
    torch.cuda.synchronize()
    stages = {}

    def timed(name, fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        stages.setdefault(name, []).append(1e3 * (time.perf_counter() - t0))

    n = 5
    for it in range(n + 1):
        if it == 1:
            stages = {}                                                # the first pass is a warm-up (module loads, allocator growth)
        timed("setupCorrespondences_ms", lambda: fus.setupCorrespondences(None, method='clpts', prune_result=False, live_vertices=live))
        timed("solve_ms", lambda: fus.solve(regularization_weight=0.5, method='cnn', precompute_lw=False, gn_iterations=5))
        timed("fuseFrame_ms", lambda: fus.fuseFrame(depth, extrinsics=sc.extrinsics))
        timed("update_graph_ms", lambda: fus.update_graph())
    stages = {k: float(np.median(v)) for k, v in stages.items()}      # wall-clock stages: the median of 5 passes (one host hiccup is not the loop)
    stages["total_ms"] = float(sum(stages.values()))
    stages["config"] = ("256^3, %d nodes -> %d after update_graph, %d canonical vertices, 5 Gauss-Newton iterations per solve, surface "
                        "extraction (step 3) + node re-sampling + incremental kNN revision inside update_graph" % (sc.n_nodes, fus._wf.n_nodes, len(fus._vertices)))
    return stages


def bench_gn(args, dev, rank, world, comm=None):
    """Second half of the BASELINE metric: Gauss-Newton ms/iteration (config 3: ~1k nodes, k=4, ~300k data residuals of
    one 640x480 frame, 15 iterations).  N>1: data residuals sharded over ranks, normal equations all-reduced (NCCL)."""
    import torch
    from dynamicfusion_body_b200 import dist as ddist
    from dynamicfusion_body_b200 import engine, gn, synth
    sc = synth.make_scene(res=256, k=4, n_nodes=args.gn_nodes, seed=0, background=True)
    pd = synth.make_gn_problem(sc, args.gn_points, seed=0)
    wf = engine.DeviceWarpField(4, dev)
    wf.set_nodes(sc.node_pos, sc.node_dq, np.float32(sc.node_w))
    shard = ddist.residual_partition(len(pd.vertices), world)[rank]
    prob = gn.Problem(wf, pd.vertices, pd.normals, pd.corr, pd.vert_knn, pd.node_vertex_idx, shard=shard, reg_owner=(rank == 0))
    x = torch.from_numpy(pd.x0).to(dev)
    allreduce = (lambda H, g, c: ddist.allreduce_normal_equations(H, g, c, comm=comm)) if world > 1 else None
    prob.pattern()
    bcast = (lambda t: comm.broadcast(t)) if (world > 1 and comm is not None) else None
    res = prob.gauss_newton(x, sc.lw, 0.05, max_iter=2, huber=True, allreduce=allreduce, broadcast=bcast)         # warm-up
    torch.cuda.synchronize()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    e[0].record()
    res = prob.gauss_newton(x, sc.lw, 0.05, max_iter=args.gn_iters, huber=True, ftol=0.0, allreduce=allreduce, broadcast=bcast)
    e[1].record()
    torch.cuda.synchronize()
    total_ms = ddist.max_over_ranks(e[0].elapsed_time(e[1]), dev)
    # breakdown of one iteration
    H, g, c = prob.normal_equations(x, sc.lw, 0.05, huber=True)
    torch.cuda.synchronize()
    t = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    t[0].record()
    H, g, c = prob.normal_equations(x, sc.lw, 0.05, huber=True)
    t[1].record()
    if allreduce:
        allreduce(H, g, c)
    t[2].record()
    x_new, delta, info = prob.solve_step(H, g, x, 1e-3, 400, 1e-9)
    t[3].record()
    torch.cuda.synchronize()
    row_ptr, col_idx, nnzb = prob.pattern()
    # the step in front of every solve (SURVEY 8f rank 1): closest-point correspondences of all canonical points against a
    # live surface of the same size -- warp, search-grid build, exact 4-NN, best point-to-plane candidate
    live = torch.from_numpy(pd.corr.astype(np.float32)).to(dev)
    loc = torch.from_numpy(pd.vert_knn.astype(np.int32)).to(dev)

    def corr_step():
        wv, wn = engine.warp_points(wf, sc.lw, pd.vertices, pd.normals, idx=loc, k=4)
        nn = engine.PointGrid(live, device=dev).knn(wv, 4)
        return engine.corr_select(wv, wn, live, nn)

    corr_step()
    torch.cuda.synchronize()
    c = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    c[0].record()
    for _ in range(3):
        best, cost = corr_step()
    c[1].record()
    torch.cuda.synchronize()
    corr_ms = c[0].elapsed_time(c[1]) / 3
    return {"metric": "gn_solve_ms_per_iter", "value": total_ms / max(1, res.iterations), "unit": "ms", "iterations": res.iterations,
            "accepted": res.accepted, "cost0": res.cost0, "cost": res.cost,
            "config": {"workload": "warp-field Gauss-Newton, %d nodes, k=4, %d data + %d regularisation residuals, %d unknowns, %d 8x8 blocks"
                                   % (sc.n_nodes, len(pd.vertices), 3 * 4 * sc.n_nodes, 8 * sc.n_nodes, nnzb)},
            "breakdown_ms": {"normal_equations": t[0].elapsed_time(t[1]), "allreduce": t[1].elapsed_time(t[2]),
                             "pcg_solve_and_update": t[2].elapsed_time(t[3]), "pcg_iterations": int(info[6].item())},
            "correspondences": {"ms": corr_ms, "canonical_points": len(pd.vertices), "live_points": int(live.shape[0]), "k": 4,
                                "matched_within_0.2": float((cost <= 0.2).float().mean().item()),
                                "note": "setupCorrespondences body (core/fusion.py:258-276) incl. host->device upload of the "
                                        "canonical points and the search-grid build"},
            "reference_published_ms_per_iter": 70100.0}


def bench_gn_depth_frame(args, dev, rank, world, comm=None):
    """BASELINE configs[2] as worded: the data residuals of ONE 640x480 depth frame.  Canonical surface samples = the valid pixels of a
    depth frame rendered from the canonical mesh, back-projected; live points = the back-projected pixels of the live depth frame;
    correspondences through the drop-in Fusion.setupCorrespondences (closest live point, best-of-k point-to-plane); then 15
    Gauss-Newton iterations from perturbed node transforms."""
    import torch
    from scipy.spatial import cKDTree
    from dynamicfusion_body_b200 import dist as ddist
    from dynamicfusion_body_b200 import gn, synth
    from dynamicfusion_body_b200.fusion import Fusion
    R = 256
    sc = synth.make_scene(res=R, k=4, n_nodes=args.gn_nodes, seed=0, background=False, focal=775.0)
    K, Kinv = sc.K, sc.Kinv
    E = np.zeros((3, 4))
    A = np.zeros(12)
    # the global rigid dq of a one-view scene is the camera extrinsic
    E = np.stack([synth.dq_apply(sc.lw[None, :].astype(np.float64), e[None, :])[0] for e in np.eye(3)], 1)
    t = synth.dq_apply(sc.lw[None, :].astype(np.float64), np.zeros((1, 3)))[0]
    Rm = E - t[:, None]

    def backproject(dm):
        v, u = np.nonzero(dm < 0)
        z = -dm[v, u].astype(np.float64)
        return (Kinv @ np.stack([u * z, v * z, z])).T

    canon_cam = backproject(synth.render_depth(sc.vertices.astype(np.float64) @ Rm.T + t, sc.faces, K, sc.rows, sc.cols))
    canon = ((canon_cam - t) @ Rm).astype(np.float32)                 # back into canonical (grid) coordinates
    _, nn = cKDTree(sc.vertices.astype(np.float64)).query(canon.astype(np.float64))
    normals = sc.normals[nn]
    live = backproject(sc.depths[0]).astype(np.float32)
    fus = Fusion(sc.tdist, knn=4, device=dev, use_cnn=False, write_warpfield=False)
    rng = np.random.default_rng(0)
    _, nvi = cKDTree(canon.astype(np.float64)).query(sc.node_pos.astype(np.float64))
    nodes = [(int(nvi[i]),) + n[1:] for i, n in enumerate(sc.nodes_as_reference_tuples())]
    fus.InitializeCanonicalSpace(tsdf_shape=(8, 8, 8), K=K, vertices=canon, normals=normals, nodes=nodes)
    fus._lw = sc.lw
    x0 = (sc.node_dq.reshape(-1).astype(np.float64) + rng.normal(size=8 * sc.n_nodes) * 2e-3)
    fus.set_node_dqs(x0.reshape(-1, 8).astype(np.float32))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fus.setupCorrespondences(None, method='clpts', prune_result=False, live_vertices=live)
    torch.cuda.synchronize()
    corr_ms = 1e3 * (time.perf_counter() - t0)
    shard = ddist.residual_partition(len(canon), world)[rank]
    prob = gn.Problem(fus._wf, fus._vertices, fus._normals, np.asarray(fus._correspondences, dtype=np.float64), np.asarray(fus._neighbor_look_up),
                      fus._node_vertex_idx, shard=shard, reg_owner=(rank == 0))
    allreduce = (lambda H, g, c: ddist.allreduce_normal_equations(H, g, c, comm=comm)) if world > 1 else None
    x = torch.from_numpy(x0).to(dev)
    prob.pattern()
    bcast = (lambda t: comm.broadcast(t)) if (world > 1 and comm is not None) else None
    prob.gauss_newton(x, sc.lw, 0.05, max_iter=2, huber=True, allreduce=allreduce, broadcast=bcast)
    torch.cuda.synchronize()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    e[0].record()
    res = prob.gauss_newton(x, sc.lw, 0.05, max_iter=args.gn_iters, huber=True, ftol=0.0, allreduce=allreduce, broadcast=bcast)
    e[1].record()
    torch.cuda.synchronize()
    total_ms = ddist.max_over_ranks(e[0].elapsed_time(e[1]), dev)
    return {"metric": "gn_solve_ms_per_iter", "value": total_ms / max(1, res.iterations), "unit": "ms", "iterations": res.iterations, "accepted": res.accepted,
            "cost0": res.cost0, "cost": res.cost, "data_residuals": int(len(canon)), "live_points": int(len(live)), "nodes": sc.n_nodes,
            "setupCorrespondences_ms": corr_ms, "pcg_iterations": [h["pcg_iterations"] for h in res.history],
            "config": {"workload": "valid pixels of one 640x480 depth frame (focal 775: the body fills the frame) as canonical samples, closest-point "
                                   "correspondences against the live frame's pixels via Fusion.setupCorrespondences, %d nodes k=4, 15 iterations" % sc.n_nodes}}


def raw_reference_rate(sc):
    """The UNMODIFIED reference's own loop (Fusion.updateTSDF, core/fusion.py:153-198: KD-tree query + warp + trilinear sample per
    voxel) on a 16^3 brick of the same node graph, one core -- only where /root/reference exists (the authoring container; the GPU
    box does not have it: there the figure probed for BASELINE.md section 2 on this container's host is quoted)."""
    try:
        from oracle import refload
        if not refload.available():
            raise RuntimeError("absent")
        R = 16
        rng = np.random.default_rng(0)
        nodes = sc.nodes_as_reference_tuples()
        centre = sc.node_pos.mean(0) - R / 2                           # a brick in the middle of the body
        nodes = [(n[0], (n[1] - centre).astype(np.float32), n[2], n[3]) for n in nodes]
        f = refload.make_fusion(nodes, np.zeros((R, R, R)), np.zeros((R, R, R)), sc.tdist, sc.k, np.array([1, 0, 0, 0, 0, 0, 0, 0], np.float32))
        curr = rng.normal(size=(R, R, R))
        t0 = time.perf_counter()
        with refload.quiet():
            f.updateTSDF(curr)
        dt = time.perf_counter() - t0
        return {"voxels_per_s_per_core": R ** 3 / dt, "how": "unmodified reference Fusion.updateTSDF on a 16^3 brick, %d nodes, k=%d, %.1f s, measured in this run" % (len(nodes), sc.k, dt)}
    except Exception:
        return {"voxels_per_s_per_core": 4651.0, "how": "unmodified reference Fusion.updateTSDF (N=1000, k=4), probed for BASELINE.md section 2 in the authoring "
                                                       "container (numpy 2.3.5, scipy 1.18.1, one Xeon core); the reference does not travel to the GPU box"}


def cpu_baseline(sc, res, budget_s=12.0):
    from oracle import driver
    sd = driver.scene_dict(sc)
    vps, n, dt = driver.time_projective(sd, res, 100_000)
    n_sample = int(min(4_000_000, max(100_000, vps * budget_s)))
    vps, n, dt = driver.time_projective(sd, res, n_sample, seed=1)
    return {"value": vps, "unit": "voxels/s", "cores": 1, "kind": "port",
            "sample": "%d random voxels of the same %dx%dx%d workload, numpy oracle (oracle/tsdf.py) incl. KD-tree kNN, %.1f s" % (n, res[0], res[1], res[2], dt),
            "raw_reference": raw_reference_rate(sc)}


def run_reference(args):
    """The reference path on the host cores.  The reference is pure Python and does not exist on the GPU box, so
    this times its numpy restatement (oracle/, kind="port") on a bounded voxel sample per step, all cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import driver
    res = args.res
    sc = build_scene(res, args.nodes, args.k, args.views)
    sd = driver.scene_dict(sc)
    cores = os.cpu_count() or 1
    per_step = args.ref_sample
    for _ in range(min(1, args.warmup)):
        driver.time_projective_parallel(sd, (res, res, res), max(cores * 20000, per_step // 4), cores)
    t0 = time.perf_counter()
    nvox = 0
    rates = []
    for _ in range(args.steps):
        r, n, wall = driver.time_projective_parallel(sd, (res, res, res), per_step, cores)
        nvox += n
        rates.append(n / wall)
    wall = time.perf_counter() - t0
    value = nvox / wall
    out = {"impl": "reference", "metric": "warped_tsdf_voxels_per_sec", "value": value, "unit": "voxels/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3, "higher_is_better": True,
           "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": "%d^3 voxels total, warped projective TSDF update (a3), k=%d DQB, %d nodes, %d view(s) 640x480; each step = a "
                                  "bounded sample of %d voxels, per-voxel KD-tree kNN included (the GPU arm's `value_amortised` accounts "
                                  "for its kNN table)" % (res, args.k, sc.n_nodes, args.views, per_step)},
           "cpu_baseline": {"value": value, "unit": "voxels/s", "cores": cores, "kind": "port",
                            "sample": "%d random voxels per step over %d worker processes (numpy oracle incl. KD-tree kNN)" % (per_step, cores)},
           "e2e": {"value": value, "unit": "voxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--res", type=int, default=512, help="per-GPU cube edge (voxels per GPU = res^3)")
    ap.add_argument("--nodes", type=int, default=4000)
    ap.add_argument("--k", type=int, default=4)
    ap.add_argument("--views", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gn", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the extra BASELINE configs / frame loop legs")
    ap.add_argument("--equal-slabs", action="store_true", help="N>1: keep the equal x-slabs (no cost-balanced boundaries)")
    ap.add_argument("--gn-nodes", type=int, default=1000)
    ap.add_argument("--gn-points", type=int, default=300000)
    ap.add_argument("--gn-iters", type=int, default=15)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--ref-sample", type=int, default=1_600_000)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the TSDF volume of the last timed step as DIR/tsdf.npy "
                                                          "and DIR/weight.npy (float32; a fixed seeded sample of %d voxels of a larger "
                                                          "volume, see dump_sample)" % DUMP_VOXELS)
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
