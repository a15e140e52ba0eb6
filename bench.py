#!/usr/bin/env python
"""bench.py -- frames/s of the BundleFusion hot path built so far (hashed-voxel TSDF integrate / re-integrate / GC per
frame + local and global sparse bundle adjustment per 10-frame chunk) on synthetic 640x480 RGB-D.

    python bench.py --gpus N --steps K --warmup W            # this implementation (libbundlefusion_b200.so)
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the oracle port on the host cores (rank 0 only)

A "step" is one frame of the reference's frame loop (FL/DepthSensing/DepthSensing.cpp:966-1129):
    reintegrate(): up to s_maxFrameFixes = 10 x { deIntegrate(old pose); integrate(new pose) }, garbageCollect()
    integrate(current frame)
and, on the last frame of every 10-frame chunk (FL/OnlineBundler.cpp:410-416), one local BA (11 frames, 2 GN x 100 PCG) and
one global BA over the keyframes (3 GN x 150 PCG).  One JSON line is printed by rank 0 (contract: see the task statement).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

W, H = 640, 480
LOOP_WORKLOAD = {
    "workload": "configs[1]: synthetic 640x480 RGB-D stream through the whole frame loop (one bfFrameLoopStep per frame: ingest, SIFT detect, dense "
                "cache, descriptor match + Kabsch / surface-area / dense-verify filters against the chunk, SIFT pose, <= 10 re-integrations + GC, "
                "integrate; per 10-frame chunk local BA 11 frames sparse + dense 2 GN x 100 PCG with verification, fuse to keyframe, match against "
                "all keyframes, global BA 3 GN x 150 PCG, trajectory update feeding the re-integration queue); hashed TSDF 1 cm voxels, 4M-block "
                "heap, 4M buckets; the timed steps continue a stream of `preroll_frames` frames",
    "frame": [W, H], "voxel_m": 0.010, "sdf_blocks": 4000000, "hash_buckets": 4000000, "reintegrations_per_frame": 10, "chunk": 10,
    "texture": "world-anchored 4-octave value noise (synth.rich_texture): ~180 SIFT features per frame; camera on the Lissajous path of SURVEY 8d",
    "l2_policy": "inputs larger than L2: every step reads a new 2.46 MB frame and re-integrates 10 stored frames (24.6 MB) against a voxel working set of several hundred MB; no explicit flush",
}
WORKLOAD = {
    "workload": "configs[1]: 640x480 RGB-D stream, hashed TSDF (1 cm voxels, 4M-block heap, 4M buckets), per frame 1 integrate + 10 "
                "re-integrations (de-integrate + integrate) + GC; per 10-frame chunk 1 local BA (11 frames, 2 GN x 100 PCG) + 1 global BA "
                "(500 keyframes, 187k correspondences, 3 GN x 150 PCG, sparse); local BA = sparse + dense depth term (80x60 caches); frame ingest, dense-cache build, SIFT detection / matching / match filters exist in the library (rows a17-a21) but are not part of this metric's step",
    "frame": [W, H], "voxel_m": 0.010, "sdf_blocks": 4000000, "hash_buckets": 4000000, "reintegrations_per_frame": 10,
    "chunk": 10, "global_keyframes": 500, "global_degree": 15, "frame_bank": 128,
    "streams": "reconstruction (TSDF) and bundling (BA) on two CUDA streams of one GPU, as the reference's two threads/devices",
    "l2_policy": "inputs larger than L2: the frame bank (315 MB) and the voxel working set are cycled; no explicit flush",
}
METRIC = "frames/sec (TSDF integrate + global BA solve) on synthetic 640x480 RGB-D"


# ------------------------------------------------------------------------------------------------------------------------
def clocks_sampler(stop_evt, out, gpu_index):
    q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    try:
        p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "10", "-i", str(gpu_index)],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except Exception:
        return
    def reader():
        for line in p.stdout:
            out.append(line.strip())
    t = threading.Thread(target=reader, daemon=True)
    t.start()
    stop_evt.wait()
    p.terminate()


def summarize_clocks(lines):
    sm, smax, reasons = [], 0, set()
    for ln in lines:
        f = [x.strip() for x in ln.split(",")]
        if len(f) < 6:
            continue
        try:
            sm.append(float(f[0])); smax = max(smax, float(f[1]))
        except ValueError:
            continue
        for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
            if v.lower().startswith("active"):
                reasons.add(name)
    if not sm:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
    return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback"


# ------------------------------------------------------------------------------------------------------------------------
class Workload:
    """Frame schedule shared by the GPU arm and the CPU arm: which frame is integrated, which are re-integrated at which poses."""

    def __init__(self, bank_poses, seed=99):
        self.poses_cur = [p.copy() for p in bank_poses]          # pose each bank frame is currently integrated with
        self.B = len(bank_poses)
        self.rng = np.random.Generator(np.random.MT19937(seed))

    def perturb(self, T):
        from bundlefusion_b200 import synth
        d = synth.se3_exp(self.rng.standard_normal(3) * 0.002, self.rng.standard_normal(3) * 0.003)
        return (d @ T.astype(np.float64)).astype(np.float32)

    def step_ops(self, f, n_reint):
        """ops of frame f: [(kind, bank index, pose)], kinds 0 integrate / 1 de-integrate / 2 GC (DepthSensing.cpp:854-902,1049)."""
        ops = []
        cur = f % self.B
        # re-integration targets: the most recent frames (TrajectoryManager's top-N by pose change, here all changed)
        for k in range(1, n_reint + 1):
            r = (cur - k) % self.B
            old = self.poses_cur[r]
            new = self.perturb(old)
            ops.append((1, r, old)); ops.append((0, r, new))
            self.poses_cur[r] = new
        ops.append((2, 0, None))
        # the incoming frame replaces what the slot held in the stream one bank-cycle ago (that observation stays integrated)
        ops.append((0, cur, self.poses_cur[cur]))
        return ops


def make_ba_problems(global_keyframes=None, global_degree=None):
    from bundlefusion_b200 import synth
    loc = synth.make_dense_ba_problem(11, stride=3, start=100, corr_per_pair=25, noise=0.002, seed=31)    # sparse + dense 80x60 caches
    glo = synth.make_ba_problem(global_keyframes or WORKLOAD["global_keyframes"], degree=global_degree or WORKLOAD["global_degree"], corr_per_pair=25, noise=0.002, seed=32, stride=10)
    return loc, glo


# ------------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    from bundlefusion_b200 import _capi as capi
    from bundlefusion_b200 import synth_gpu
    from bundlefusion_b200.scene_rep import CUDASceneRepHashSDF, camera_params, default_hash_params
    from bundlefusion_b200.solver import CUDASolverBundling

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = capi.lib()
    cam = camera_params(W, H)
    hp = default_hash_params(num_buckets=WORKLOAD["hash_buckets"], num_sdf_blocks=WORKLOAD["sdf_blocks"], voxel_size=WORKLOAD["voxel_m"])
    if world > 1:
        hp.m_dummy = (world << 32) | rank            # spatial shard of the voxel hash: this rank owns blocks with owner(pos) == rank
    scene = CUDASceneRepHashSDF(hp, dev, arithmetic=os.environ.get("BF_TSDF_ARITH", "fast"))       # "exact": the bit-identical kernels, for A/B runs

    B = WORKLOAD["frame_bank"]
    idx = [8 * i for i in range(B)]
    depth, color, poses = synth_gpu.make_frames(idx, W, H, device=str(dev))
    dlist, clist = [depth[i] for i in range(B)], [color[i] for i in range(B)]
    # host copies for the e2e leg (pinned), plus a device landing slot per bank frame
    h_depth = depth.cpu().pin_memory(); h_color = color.cpu().pin_memory()
    wl = Workload(list(poses))
    n_re = WORKLOAD["reintegrations_per_frame"]
    # the whole op schedule is prepared up front (poses come from the schedule, not from the timed loop)
    total_steps = args.warmup + 2 * args.steps
    packed_ops = [scene.packOps(wl.step_ops(f, n_re)) for f in range(total_steps)]
    packed_frames = scene.packFrames(dlist, clist)

    loc, glo = make_ba_problems()
    def upload(prob):
        return (torch.from_numpy(prob["corr"].view(np.uint8).reshape(-1).copy()).to(dev), torch.from_numpy(prob["init_rot"]).to(dev),
                torch.from_numpy(prob["init_trans"]).to(dev), torch.ones(len(prob["init_rot"]), dtype=torch.int32, device=dev))
    lc, lr0, lt0, lv = upload(loc); gc_, gr0, gt0, gv = upload(glo)
    lrot, ltrans, grot, gtrans = lr0.clone(), lt0.clone(), gr0.clone(), gt0.clone()
    from bundlefusion_b200.solver import DeviceCache
    loc_cache = DeviceCache(loc["caches"], loc["intrinsics"], dev)
    sol_l = CUDASolverBundling(11, 11 * 1000, dev); sol_g = CUDASolverBundling(len(glo["init_rot"]), max(len(glo["corr"]), 1000 * len(glo["init_rot"])), dev)
    h_grot = torch.empty_like(grot, device="cpu").pin_memory(); h_gtrans = torch.empty_like(gtrans, device="cpu").pin_memory()
    h_heap = torch.empty(1, dtype=torch.int32).pin_memory()

    # warm model: every bank frame integrated once
    scene.runOps([(0, i, poses[i]) for i in range(B)], dlist, clist, cam)
    torch.cuda.synchronize()

    # Bundling runs on its own stream, concurrently with the reconstruction stream -- the reference runs them on separate
    # threads / devices (FL/FriedLiver.cpp:118-182, FL/DualGPU.h:108-134); poses are consumed when the solve has finished.
    ba_stream = torch.cuda.Stream(device=dev)

    # Multi-GPU: chunks are independent units of bundling work -- chunk c's local + global solve runs on rank c % world, which then
    # broadcasts the 6N global pose update over NVLink (its own communicator, so the per-frame image broadcasts never queue behind a
    # solve); every rank ends up with the same poses (north_star: "the per-chunk local BA shards across the GPUs").
    ba_group = dist.new_group() if world > 1 else None

    def ba(e2e, chunk=0):
        owner = chunk % world
        ba_stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(ba_stream):
            if rank == owner:
                lrot.copy_(lr0); ltrans.copy_(lt0); grot.copy_(gr0); gtrans.copy_(gt0)
                # local BA as FL/SBA.cpp:28-31, 64-75: sparse weight 1, dense depth weights 1, 2, colour 0
                sol_l.solve(lc, len(loc["corr"]), lv, 11, 2, 100, [1.0, 1.0], [1.0, 2.0], [0.0, 0.0], d_rotationAnglesUnknowns=lrot, d_translationUnknowns=ltrans, cudaCache=loc_cache)
                sol_g.solve(gc_, len(glo["corr"]), gv, len(glo["init_rot"]), 3, 150, [1.0, 1.0, 1.0], d_rotationAnglesUnknowns=grot, d_translationUnknowns=gtrans)
            if world > 1:
                dist.broadcast(grot, owner, group=ba_group); dist.broadcast(gtrans, owner, group=ba_group)
            if e2e:
                h_grot.copy_(grot, non_blocking=True); h_gtrans.copy_(gtrans, non_blocking=True)

    skip_ba = [args.no_ba]

    # The incoming frame reaches its device slot one frame ahead of the fusion, on a side stream: frame f+1 crosses PCIe (e2e leg: the
    # sensor hands HOST pinned buffers to rank 0 every step, as FL/CUDAImageManager.cpp:22-158 uploads on arrival) and, with several
    # GPUs, NVLink (the sensor frame lives on rank 0: one NCCL broadcast of depth + colour per step, every rank fuses its own shard)
    # while frame f is being fused.  The slot it lands in was last read > 100 steps ago.
    pre_stream = torch.cuda.Stream(device=dev)
    pre_done = {}

    def prefetch_frame(f, e2e):
        cur = f % B
        with torch.cuda.stream(pre_stream):
            if e2e and rank == 0:
                dlist[cur].copy_(h_depth[cur], non_blocking=True); clist[cur].copy_(h_color[cur], non_blocking=True)
            if world > 1:
                dist.broadcast(dlist[cur], 0); dist.broadcast(clist[cur], 0)
            ev = torch.cuda.Event(); ev.record(pre_stream)
        pre_done[f] = ev

    def step(f, e2e):
        if e2e or world > 1:
            if f not in pre_done:
                prefetch_frame(f, e2e)
            torch.cuda.current_stream(dev).wait_event(pre_done.pop(f))
        scene.runPackedOps(packed_ops[f], packed_frames, cam)
        if (e2e or world > 1) and f + 1 < len(packed_ops):
            prefetch_frame(f + 1, e2e)
        if f % WORKLOAD["chunk"] == WORKLOAD["chunk"] - 1 and not skip_ba[0]:
            ba(e2e, f // WORKLOAD["chunk"])
        if e2e:
            h_heap.copy_(scene.d_heapCounter, non_blocking=True)

    def timed(n_steps, f0, e2e, profile):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        pre_done.clear()               # a frame prefetched at the end of the previous pass is fetched again by this pass's rules
        if profile:
            L.bfTsdfSetProfiling(1)
        l0 = L.bfGetLaunchCount()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for f in range(f0, f0 + n_steps):
            step(f, e2e)
        torch.cuda.current_stream(dev).wait_stream(ba_stream)     # the timed region ends when BOTH streams are done
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
        if world > 1:
            t = torch.tensor([ms], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item()); dist.barrier()
        return ms, L.bfGetLaunchCount() - l0

    K, Wm = args.steps, args.warmup
    if not args.no_ba:            # first-call costs of the bundling path (workspace allocation, cooperative-launch set-up) belong to warm-up
        for c in range(world):        # every rank's solver gets its first call here
            ba(False, c)
        torch.cuda.synchronize()
    timed(Wm, 0, False, False)
    clk_lines, stop_evt = [], threading.Event()
    th = threading.Thread(target=clocks_sampler, args=(stop_evt, clk_lines, local), daemon=True); th.start()
    ms, launches = timed(K, Wm, False, False)
    stop_evt.set()
    # separate pass with CUDA events around every stencil launch (the events cost a little, so it is not the headline run)
    total_needed = Wm + 3 * K
    while len(packed_ops) < total_needed:
        packed_ops.append(scene.packOps(wl.step_ops(len(packed_ops), n_re)))
    skip_ba[0] = True        # the stencil is timed alone (no bundling kernel, no front-lane kernel sharing the SMs): the burst HBM peak is its roof
    prev_lanes = L.bfTsdfSetLanes(0)
    timed(K, Wm + 2 * K, False, True)
    L.bfTsdfSetLanes(prev_lanes)
    skip_ba[0] = args.no_ba
    prof = (ctypes.c_ulonglong * 16)()
    capi.check(L.bfTsdfGetProfileEx(ctypes.byref(scene.m_hashData), prof), "bfTsdfGetProfileEx")
    L.bfTsdfSetProfiling(0)
    ms_e2e, _ = timed(K, Wm + K, True, False)
    stats = scene.getLastFrameStats()
    heap_free = scene.getHeapFreeCount()
    sg = sol_g.getStats() if not args.no_ba else {"pcg": 0, "gn": 0}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks, peak_kind = measured_peaks()
    n_launch, n_timed, ns, U, E, n_img = int(prof[0]), int(prof[1]), int(prof[2]), int(prof[3]), int(prof[4]), max(int(prof[5]), int(prof[0]))
    all_launches = {"launches": n_launch, "avg_launch_us": round(ns / max(1, n_timed) / 1e3, 2)}
    if int(prof[9]) > 0:          # the dominant kernel is the batch pass (one launch per frame's re-integrations): its own launches, bytes and time
        n_launch = n_timed = int(prof[9]); ns, U, E, n_img = int(prof[10]), int(prof[11]), int(prof[12]), int(prof[13])
    # SURVEY 8d: 24 B x U + 20 B x E + 2 x W x H x 4 B per frame image read (one per launch; a batch launch reads one per re-integration pair)
    alg_bytes = 24.0 * U + 20.0 * E + n_img * 2.0 * W * H * 4.0
    ach = (alg_bytes * (n_timed / max(1, n_launch))) / max(1e-9, ns * 1e-9) / 1e9 if n_timed else 0.0
    roof = {"kernel": "TSDF stencil (stencil_multi_kernel: a frame's re-integration batch in one pass; stencil_fast_kernel: single integrate)" if scene.arithmetic == "fast" else "integrate_kernel / reintegrate_kernel (bit-exact TSDF stencil)", "bound": "hbm", "achieved": round(ach, 1), "peak": peaks["hbm_gbs"],
            "peak_kind": f"{peak_kind} (MEASURED_PEAKS.json hbm_gbs, burst copy)", "unit": "GB/s", "frac": round(ach / peaks["hbm_gbs"], 4),
            "traffic": None, "launches": n_launch, "avg_launch_us": round(ns / max(1, n_timed) / 1e3, 2),
            "algorithmic_bytes_per_launch": round(alg_bytes / max(1, n_launch)), "U_per_launch": round(U / max(1, n_launch)), "E_per_launch": round(E / max(1, n_launch)),
            "frames_per_launch": round(n_img / max(1, n_launch), 2), "all_stencil_launches": all_launches}
    # DRAM traffic of the dominant kernel from the committed `ncu --set full` capture of this command (profiles/), per launch
    tpath = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r1_stencil_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        roof["traffic"] = tj.get("dram_bytes_per_launch")
        roof["traffic_note"] = tj.get("note")
    bytes_in = (W * H * 4 * 2)
    bytes_out = 4 + (6 * 4 * len(glo["init_rot"])) / WORKLOAD["chunk"]
    out = {
        "metric": METRIC, "value": round(K / (ms / 1e3), 2), "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": round(ms / K, 4), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(WORKLOAD, parallelism=("single GPU" if world == 1 else f"voxel hash sharded over {world} GPUs by block owner; frame broadcast (NCCL) per step; chunk c's bundle adjustment on rank c % {world}, 6N pose update broadcast"),
                       active_blocks=int(WORKLOAD["sdf_blocks"] - heap_free), in_frustum_blocks_last=int(stats["E"]), global_pcg_iters=int(sg["pcg"]), global_gn_iters=int(sg["gn"])),
        "e2e": {"value": round(K / (ms_e2e / 1e3), 2), "unit": "frames/s", "h2d_bytes_per_step": bytes_in, "d2h_bytes_per_step": int(bytes_out),
                "note": "incoming frame copied from pinned host memory every step on an upload stream, one frame ahead of the fusion; re-integrated frames come from the device-resident frame store"},
        "gpu_launches": int(launches), "roofline": roof, "tsdf_arithmetic": scene.arithmetic, "clocks": summarize_clocks(clk_lines),
    }
    if args.no_ba:
        out["diagnostic"] = "--no-ba: bundle adjustment left out, not a bench value"
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_arm(1, 0, quiet=True, n_reint=2)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()



# ------------------------------------------------------------------------------------------------------------------------
def run_loop(args):
    """headline workload: the frame loop, one bfFrameLoopStep per frame"""
    import torch
    import torch.distributed as dist

    from bundlefusion_b200 import _capi as capi
    from bundlefusion_b200 import synth_gpu
    from bundlefusion_b200.frame_loop import FrameLoop, default_params

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = capi.lib()
    K, Wm, pre = args.steps, args.warmup, args.preroll
    total = pre + Wm + 3 * K                       # pre-roll, warm-up, timed pass, profiled pass, end-to-end pass: one continuous stream
    P = default_params(W, H)
    P.maxNumFrames = total + 8
    P.maxNumImages = total // 10 + 8
    P.maxGlobalResiduals = 25 * P.maxNumImages * 48
    P.hash.m_hashNumBuckets = LOOP_WORKLOAD["hash_buckets"]; P.hash.m_numSDFBlocks = LOOP_WORKLOAD["sdf_blocks"]
    if world > 1:
        P.hash.m_dummy = (world << 32) | rank                   # spatial shard of the voxel hash: this rank integrates the blocks it owns
    clk_lines, stop_evt = [], threading.Event()
    if rank == 0:                                              # the line is rank 0's: one nvidia-smi loop per box, not one per rank (NVML queries contend with the ranks' launches)
        th = threading.Thread(target=clocks_sampler, args=(stop_evt, clk_lines, local), daemon=True); th.start()
    loop = FrameLoop(P, dev)
    overlap = os.environ.get("BF_LOOP_OVERLAP", "1") != "0"
    loop.set_overlap(overlap)
    # frame bank on the device, generated in slices (input generation, never timed); the stream advances 2 frames of the Lissajous path per step
    depth = torch.empty(total, H, W, dtype=torch.float32, device=dev); color = torch.empty(total, H, W, 4, dtype=torch.uint8, device=dev)
    for s0 in range(0, total, 64):
        idx = [args.stride * i for i in range(s0, min(total, s0 + 64))]
        d, c, _ = synth_gpu.make_frames(idx, W, H, device=str(dev), texture="rich")
        depth[s0:s0 + len(idx)] = d; color[s0:s0 + len(idx)] = c
    torch.cuda.synchronize()
    f_e2e0 = pre + Wm + 2 * K
    ahead = os.environ.get("BF_LOOP_AHEAD", "1") != "0"      # bfFrameLoopStepAhead: frame k + 1 of a pass is announced while frame k is stepped
    h_depth = depth[f_e2e0:f_e2e0 + K].cpu().pin_memory(); h_color = color[f_e2e0:f_e2e0 + K].cpu().pin_memory()
    stats = {"valid": 0, "local": 0, "local_valid": 0, "global": 0, "reint": 0, "kp": 0, "n": 0}
    last = {}                                              # status block of the most recent step

    trace = []

    def note(st):
        if args.trace:
            trace.append((int(st.frame), int(st.validTransform), int(st.numKeyPoints), int(st.lastMatchedFrame), int(st.numLocalCorrespondences), int(st.numReintegrated),
                          int(st.localSolved), int(st.localValid), int(st.numKeyframes), int(st.numGlobalCorrespondences), int(st.globalSolved), int(st.globalRemoved), int(st.globalTrackingLost)))
        stats["n"] += 1; stats["valid"] += st.validTransform; stats["reint"] += st.numReintegrated; stats["kp"] += st.numKeyPoints
        stats["local"] += 1 if st.localSolved >= 0 else 0; stats["local_valid"] += st.localValid; stats["global"] += st.globalSolved

    for f in range(pre):                                   # pre-roll: the state a long stream is in (keyframes, trajectory, populated hash)
        st = loop.step(depth[f], color[f], *((depth[f + 1], color[f + 1]) if ahead and f + 1 < pre else (None, None)))
        if args.trace:
            note(st)
    torch.cuda.synchronize()

    def timed(f0, n, e2e, profile):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if profile:
            L.bfTsdfSetProfiling(1)
        l0 = L.bfGetLaunchCount()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        steptimes = [] if (os.environ.get("BF_LOOP_STEPTIMES") and not profile) else None
        for k in range(n):
            t_step0 = time.perf_counter() if steptimes is not None else 0.0
            la = ahead and not profile and k + 1 < n       # look-ahead stays inside the pass: its first frame is never prefetched, its last announces nothing
            if e2e:
                st = loop.step(h_depth[k], h_color[k], *((h_depth[k + 1], h_color[k + 1]) if la else (None, None)))
            else:
                st = loop.step(depth[f0 + k], color[f0 + k], *((depth[f0 + k + 1], color[f0 + k + 1]) if la else (None, None)))
            last["st"] = st
            if not profile:
                note(st)
            if steptimes is not None:
                steptimes.append((int(st.frame), round((time.perf_counter() - t_step0) * 1e3, 3), int(st.localSolved), int(st.globalSolved), int(st.globalRemoved), int(st.numKeyframes)))
        if steptimes is not None and rank == 0:             # diagnostic: host wall time of every step call of this pass
            with open(os.environ["BF_LOOP_STEPTIMES"], "a") as fp:
                fp.write(f"# pass f0={f0} n={n} e2e={e2e}\n" + "".join(" ".join(str(v) for v in t) + "\n" for t in steptimes))
        loop.join()                                        # the timed region covers the reconstruction stream's work of its last frame
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
        if world > 1:
            t = torch.tensor([ms], device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item()); dist.barrier()
        return ms, L.bfGetLaunchCount() - l0

    timed(pre, Wm, False, False)
    for k in stats: stats[k] = 0
    clk_mark0 = len(clk_lines)
    if args.cuda_profiler:
        torch.cuda.profiler.start()
    ms, launches = timed(pre + Wm, K, False, False)
    if args.cuda_profiler:
        torch.cuda.profiler.stop()
    clk_mark1 = len(clk_lines)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, L, loop, last["st"], pre + Wm + K)
    c_before = loop.counters()
    prev_lanes = L.bfTsdfSetLanes(0)                       # the stencil is timed alone on its stream: the burst HBM peak is its roof
    loop.set_profiling(True)
    timed(pre + Wm + K, K, False, True)
    stages = loop.stage_times()
    loop.set_profiling(False)
    L.bfTsdfSetLanes(prev_lanes)
    prof = (ctypes.c_ulonglong * 16)()
    capi.check(L.bfTsdfGetProfileEx(L.bfFrameLoopGetHashData(loop._h), prof), "bfTsdfGetProfileEx")
    L.bfTsdfSetProfiling(0)
    clk_mark2 = len(clk_lines)
    stats_timed = dict(stats)
    ms_e2e, _ = timed(f_e2e0, K, True, False)
    stats_e2e = {k: stats[k] - stats_timed[k] for k in stats}
    stats = stats_timed
    stop_evt.set()
    if args.trace and rank == 0:
        os.makedirs(os.path.dirname(os.path.abspath(args.trace)), exist_ok=True)
        with open(args.trace, "w") as fp:
            fp.write("frame valid keypoints lastMatched localCorr reint localSolved localValid keyframes globalCorr globalSolved globalRemoved trackingLost\n")
            for t in trace:
                fp.write(" ".join(str(v) for v in t) + "\n")
    heap_free = loop.heap_free()
    cnt = loop.counters()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks, peak_kind = measured_peaks()
    use_batch = int(prof[9]) > 0
    n_launch, n_timed, ns, U, E, n_img = (int(prof[9]), int(prof[9]), int(prof[10]), int(prof[11]), int(prof[12]), int(prof[13])) if use_batch else \
                                         (int(prof[0]), int(prof[1]), int(prof[2]), int(prof[3]), int(prof[4]), max(int(prof[5]), int(prof[0])))
    alg_bytes = 24.0 * U + 20.0 * E + n_img * 2.0 * W * H * 4.0        # SURVEY 8d: 24 B x U + 20 B x E + 2 x W x H x 4 B per frame image read
    ach = (alg_bytes * (n_timed / max(1, n_launch))) / max(1e-9, ns * 1e-9) / 1e9 if n_timed else 0.0
    roof = {"kernel": "stencil_multi_kernel (TSDF stencil: a frame's re-integration batch, every voxel of the union list read and written once)" if use_batch else "stencil_fast_kernel",
            "bound": "hbm", "achieved": round(ach, 1), "peak": peaks["hbm_gbs"], "peak_kind": f"{peak_kind} (MEASURED_PEAKS.json hbm_gbs, burst copy)", "unit": "GB/s",
            "frac": round(ach / peaks["hbm_gbs"], 4), "traffic": None, "launches": n_launch, "avg_launch_us": round(ns / max(1, n_timed) / 1e3, 2),
            "algorithmic_bytes_per_launch": round(alg_bytes / max(1, n_launch)), "U_per_launch": round(U / max(1, n_launch)), "E_per_launch": round(E / max(1, n_launch)),
            "frames_per_launch": round(n_img / max(1, n_launch), 2),
            "avg_launch_us_device_timer": round(int(prof[14]) / max(1, n_timed) / 1e3, 2) if use_batch and int(prof[14]) else None,
            "all_stencil_launches": {"launches": int(prof[0]), "avg_launch_us": round(int(prof[2]) / max(1, int(prof[1])) / 1e3, 2)},
            "mvoxels_per_s": round(512.0 * E / max(1e-9, ns * 1e-9) / 1e6, 1),
            "block_pose_entries_culled_per_launch": round(int(prof[15]) / max(1, n_launch)) if use_batch else None}
    tpath = os.path.join(ROOT, "profiles", "r2_stencil_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath)); roof["traffic"] = tj.get("dram_bytes_per_launch"); roof["traffic_note"] = tj.get("note")
    steps_meas = max(1, stats["n"])
    out = {
        "metric": METRIC, "value": round(K / (ms / 1e3), 2), "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": round(ms / K, 4), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(LOOP_WORKLOAD, preroll_frames=pre, frame_stride=args.stride,
                       parallelism=("single GPU" if world == 1 else f"voxel hash sharded over {world} GPUs by block owner (each rank integrates its blocks); SIFT / bundling replicated per rank (deterministic inputs, no exchange)"),
                       active_blocks=int(LOOP_WORKLOAD["sdf_blocks"] - heap_free), keyframes=cnt["keyframes"], global_pcg_iters_last_solve=cnt["global_pcg_iters"],
                       in_timed_steps={"frames_with_pose": stats["valid"], "reintegrations_per_frame": round(stats["reint"] / steps_meas, 2), "keypoints_per_frame": round(stats["kp"] / steps_meas, 1),
                                       "local_solves": stats["local"], "local_solves_accepted": stats["local_valid"], "global_solves": stats["global"]},
                       host_syncs_per_frame=round((cnt["host_syncs"]) / max(1, cnt["frames"]), 2)),
        "e2e": {"value": round(K / (ms_e2e / 1e3), 2), "unit": "frames/s", "h2d_bytes_per_step": W * H * 8, "d2h_bytes_per_step": 120 + 64 + 8,
                "frames_with_pose": stats_e2e["valid"], "local_solves": stats_e2e["local"], "global_solves": stats_e2e["global"],
                "note": "bfFrameLoopStep with HOST (pinned) depth + colour pointers: the upload happens inside the call, as CUDAImageManager::process uploads on arrival; read back per step: the status block (pose of the frame), the SIFT pose and the match verdict"},
        "gpu_launches": int(launches), "roofline": roof, "tsdf_arithmetic": "fast",
        "streams": ("three" if ahead and overlap else "two" if ahead or overlap else "one") + " (bundling on the library stream" + ("; reconstruction on the loop's second stream" if overlap else "") +
                   ("; the NEXT frame's upload / ingest / SIFT detection / dense cache on the loop's feature stream (bfFrameLoopStepAhead, frames announced inside a pass only)" if ahead else "") +
                   "; events keep the single-threaded order's dependencies, results identical: tests/test_frame_loop_gpu.py)",
        "stages_ms_per_step": dict(stages, note="profiled pass (--steps steps, serial on one stream, one extra host synchronisation per step, TSDF lanes off): device time line between stage boundaries, mean per step"),
        "clocks": summarize_clocks(clk_lines[clk_mark0:clk_mark1]), "clocks_profile_pass": summarize_clocks(clk_lines[clk_mark1:clk_mark2]),
    }
    if world == 1 and os.environ.get("BF_BENCH_MESH", "1") != "0":
        out["mesh"] = mesh_leg(L, loop, P, dev, int(LOOP_WORKLOAD["sdf_blocks"] - heap_free))
    if world == 1 and not args.no_cpu_baseline:
        try:                                                       # the legs below explain the headline; a failure in one is reported in its entry and the line still prints
            loop.close(); del loop, depth, color
            torch.cuda.empty_cache()
            out["reference_cuda"] = reference_cuda_leg(dev)
            if isinstance(out["reference_cuda"], dict) and "pcg" in out["reference_cuda"]:
                out["pcg"] = out["reference_cuda"].pop("pcg")       # BASELINE's "ms/PCG-iter vs HBM roofline": the 500-keyframe solve of the reference_cuda leg
        except Exception as e:                                     # noqa: BLE001
            out["reference_cuda"] = {"error": repr(e)[:300]}
        out["cpu_baseline"] = cpu_arm(1, 0, quiet=True, n_reint=2)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()

# ------------------------------------------------------------------------------------------------------------------------
def run_sweep(args):
    """configs[3] of BASELINE.json: integrate / de-integrate throughput against the number of active voxels, the voxel hash sharded over the ranks by block
    owner (each rank allocates and fuses the blocks it owns; the frame and the pose pair come from rank 0 over NCCL every step).  One re-integration
    (de-integrate at the old pose + integrate at the new one, fused pass) per step.  Strong scaling: the same frames and voxel sizes at every N."""
    import torch
    import torch.distributed as dist

    from bundlefusion_b200 import _capi as capi
    from bundlefusion_b200 import synth_gpu
    from bundlefusion_b200.scene_rep import CUDASceneRepHashSDF, camera_params, default_hash_params

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = capi.lib()
    cam = camera_params(W, H)
    K, Wm, B = args.steps, args.warmup, 24
    idx = [8 * i for i in range(B)]
    depth, color, poses = synth_gpu.make_frames(idx, W, H, device=str(dev))           # the same bank on every rank (deterministic); the timed steps use rank 0's copy
    rng = np.random.Generator(np.random.MT19937(5))
    rows = []
    for vs in (0.04, 0.02, 0.01, 0.006, 0.004, 0.003, 0.002):
        hp = default_hash_params(num_buckets=4_000_000, num_sdf_blocks=3_000_000, voxel_size=vs)
        if world > 1:
            hp.m_dummy = (world << 32) | rank
        scene = CUDASceneRepHashSDF(hp, dev)
        cur = [np.array(p, np.float32) for p in poses]
        for i in range(B):
            scene.integrate(cur[i], depth[i], color[i], cam)
        # the exchange of step k + 1 (frame + pose pair: ONE packed NCCL broadcast from rank 0 on a communication stream) runs while step k is fused
        nbytes_d, nbytes_c = depth[0].numel() * 4, color[0].numel()
        slots = [torch.empty(nbytes_d + nbytes_c + 128, dtype=torch.uint8, device=dev) for _ in range(2)]
        h_pose = [torch.empty(32, dtype=torch.float32).pin_memory() for _ in range(2)]
        ev_ready = [torch.cuda.Event() for _ in range(2)]; ev_free = [torch.cuda.Event() for _ in range(2)]
        comm = torch.cuda.Stream(device=dev)
        deltas = []
        for k in range(Wm + K + 1):
            d = np.eye(4, dtype=np.float32); d[:3, 3] = rng.standard_normal(3).astype(np.float32) * 0.004
            deltas.append(d)
        pending = {}

        def exchange(k):                                    # queue the broadcast of step k's inputs into slot k & 1
            f = k % B; sl = slots[k & 1]
            new = (deltas[k] @ cur[f]).astype(np.float32)
            with torch.cuda.stream(comm):
                comm.wait_event(ev_free[k & 1])                                  # the fusion that last read this slot has finished
                if rank == 0:
                    sl[:nbytes_d].view(torch.float32).view(H, W).copy_(depth[f], non_blocking=True)
                    sl[nbytes_d:nbytes_d + nbytes_c].view(H, W, 4).copy_(color[f], non_blocking=True)
                    sl[nbytes_d + nbytes_c:].view(torch.float32).copy_(torch.from_numpy(np.concatenate([cur[f].reshape(-1), new.reshape(-1)])), non_blocking=True)
                dist.broadcast(sl, 0)
                h_pose[k & 1].copy_(sl[nbytes_d + nbytes_c:].view(torch.float32), non_blocking=True)
                ev_ready[k & 1].record(comm)
            cur[f] = new
            pending[k] = f

        def step(k):
            f = k % B
            if world > 1:
                if k not in pending:
                    exchange(k)
                ev_ready[k & 1].synchronize()                                    # pose pair on the host (the copy finished while the previous step ran)
                pp = h_pose[k & 1].numpy().copy(); old_p, new_p = pp[:16].reshape(4, 4), pp[16:].reshape(4, 4)
                sl = slots[k & 1]
                torch.cuda.current_stream().wait_event(ev_ready[k & 1])
                exchange(k + 1)                                                   # next step's inputs travel while this step is fused
                scene.runOps([(1, 0, old_p), (0, 0, new_p)], [sl[:nbytes_d].view(torch.float32).view(H, W)], [sl[nbytes_d:nbytes_d + nbytes_c].view(H, W, 4)], cam)
                ev_free[k & 1].record(torch.cuda.current_stream())
                del pending[k]
            else:
                new = (deltas[k] @ cur[f]).astype(np.float32)
                scene.runOps([(1, f, cur[f]), (0, f, new)], [depth[i] for i in range(B)], [color[i] for i in range(B)], cam)
                cur[f] = new

        for e in ev_free:
            e.record(torch.cuda.current_stream())
        for k in range(Wm):
            step(k)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        L.bfTsdfSetProfiling(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for k in range(Wm, Wm + K):
            step(k)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
        prof = (ctypes.c_ulonglong * 16)()
        hd = scene.getHashData()
        capi.check(L.bfTsdfGetProfileEx(ctypes.byref(hd), prof), "bfTsdfGetProfileEx")
        L.bfTsdfSetProfiling(0)
        t = torch.tensor([ms, float(prof[3]), float(prof[4]), float(prof[2]) / max(1, int(prof[1]))], device=dev, dtype=torch.float64)
        if world > 1:
            mx = t.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX); sm = t.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
            ms, U, E, st_ns = float(mx[0]), float(sm[1]), float(sm[2]), float(mx[3])
        else:
            ms, U, E, st_ns = float(t[0]), float(t[1]), float(t[2]), float(t[3])
        occupied = scene.getNumOccupiedBlocks()
        rows.append({"voxel_m": vs, "active_voxels_per_op_M": round(512.0 * E / (2 * K) / 1e6, 2), "ms_per_reintegration": round(ms / K, 4),
                     "mvoxels_per_s": round(512.0 * E / (ms * 1e-3) / 1e6, 1), "updates_per_s_M": round(U / (ms * 1e-3) / 1e6, 1),
                     "stencil_us_max_rank": round(st_ns / 1e3, 2), "occupied_blocks_this_rank": int(occupied)})
        scene.close()
        del scene
        torch.cuda.empty_cache()
    if rank == 0:
        print(json.dumps({"metric": "Mvoxels/s, TSDF de-integrate + integrate (BASELINE configs[3] sweep)", "unit": "Mvoxels/s", "n_gpus": world, "steps": K, "warmup": Wm,
                          "value": rows[-1]["mvoxels_per_s"], "higher_is_better": True, "scaling": "strong", "data": "synthetic", "dtype": "f32",
                          "config": {"workload": "one re-integration per step of a 24-frame bank at voxel sizes 4 cm ... 2 mm; Mvoxels = 512 x in-frustum blocks (both ops), summed over the ranks; time = max over ranks",
                                     "parallelism": "single GPU" if world == 1 else f"voxel hash sharded over {world} GPUs by block owner; frame + pose pair broadcast from rank 0 every step (one packed NCCL broadcast, one step ahead on a communication stream)"},
                          "sweep": rows}))
    if world > 1:
        dist.destroy_process_group()

# ------------------------------------------------------------------------------------------------------------------------
DUMP_BLOCKS = 2048               # voxel blocks of the fused model written by --dump-outputs (2048 x 512 voxels x 24 B = 25 MB)


def dump_outputs(out_dir, L, loop, st, n_frames):
    """--dump-outputs: what the timed pass computed in its last step, as a caller of bfFrameLoopStep receives it -- the status block (the frame's
    pose and counters), the trajectory of every frame so far, and the fused model: the voxel words (sdf, weight, colour) of a fixed sample of its
    blocks, in the order of their block coordinates (which hash slot a block occupies depends on scheduling; the block set and its voxels do not).
    A block is sampled by a hash of its own coordinates, so two runs whose block sets differ by a few blocks still sample the same blocks elsewhere."""
    from bundlefusion_b200 import _capi as capi
    os.makedirs(out_dir, exist_ok=True)
    save = lambda name, a: np.save(os.path.join(out_dir, name + ".npy"), a)
    loop.join()
    d = st.as_dict()
    save("pose", d.pop("transform"))
    for k, v in d.items():
        save("status_" + k, np.array([v], np.float64))
    save("trajectory", loop.trajectory(n_frames))
    rt = ctypes.CDLL("libcudart.so.12")                    # the runtime the library is linked against (loaded with it)
    rt.cudaMemcpy.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
    hd, hp = L.bfFrameLoopGetHashData(loop._h).contents, L.bfFrameLoopGetHashParams(loop._h).contents
    ent = np.empty((int(hp.m_hashNumBuckets) * capi.BF_HASH_BUCKET_SIZE, 8), np.int32)
    capi.check(rt.cudaMemcpy(ent.ctypes.data, hd.d_hash, ent.nbytes, 2), "cudaMemcpy")
    ent = ent[ent[:, 3] != -2]                                                          # allocated entries: (x, y, z, voxel offset, ...)
    ent = ent[np.lexsort((ent[:, 2], ent[:, 1], ent[:, 0]))]
    x, y, z = (ent[:, k].astype(np.int64) for k in range(3))
    h = ((x * 73856093) ^ (y * 19349669) ^ (z * 83492791)) & 0xFFFFFFFF
    pick = np.sort(np.argsort(h, kind="stable")[:DUMP_BLOCKS])
    vox = np.empty((len(pick), capi.BF_SDF_BLOCK_VOXELS, 3), np.int32)
    for i, e in enumerate(ent[pick]):
        capi.check(rt.cudaMemcpy(vox[i].ctypes.data, hd.d_SDFBlocks + int(e[3]) * 12, vox[i].nbytes, 2), "cudaMemcpy")
    save("tsdf_block_coords", ent[pick, :3].astype(np.float64))
    save("tsdf_sdf", np.ascontiguousarray(vox[..., 0]).view(np.float32))
    save("tsdf_weight", np.ascontiguousarray(vox[..., 1]).view(np.float32))
    save("tsdf_color", np.ascontiguousarray(vox[..., 2]).view(np.uint8).reshape(len(pick), -1, 4).astype(np.float32))


def mesh_leg(L, loop, P, dev, active_blocks):
    """Row N4: the iso-surface of the model the loop just built (bfMarchingCubesExtract on the loop's hash), timed with CUDA events on the library's stream -- the
    kernel's first hardware timing comes from this leg.  Runs after every other measurement of the line; a failure is reported in the entry, not raised."""
    try:
        import ctypes as C
        import torch
        from bundlefusion_b200.marching_cubes import _bind, marching_cubes_params
        _bind(L)
        hp = L.bfFrameLoopGetHashParams(loop._h).contents           # the loop's own copy (table size, voxel size)
        cap = 6_000_000                                               # 72 B each
        mp = marching_cubes_params(int(hp.m_hashNumBuckets), float(hp.m_virtualVoxelSize), cap)
        tri = torch.empty(cap * 18, dtype=torch.float32, device=dev)
        n = torch.zeros(1, dtype=torch.int32, device=dev)
        loop.join()
        loop._bind_stream()
        hd = L.bfFrameLoopGetHashData(loop._h)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        times = []
        for _ in range(6):
            torch.cuda.synchronize(dev)
            ev[0].record()
            rc = L.bfMarchingCubesExtract(hd, C.byref(hp), C.byref(mp), C.c_void_p(tri.data_ptr()), C.c_void_p(n.data_ptr()))
            ev[1].record()
            torch.cuda.synchronize(dev)
            if rc:
                return {"error": f"bfMarchingCubesExtract returned {rc}"}
            times.append(ev[0].elapsed_time(ev[1]))
        ms = sorted(times[1:])[len(times[1:]) // 2]
        ntri = int(n.item())
        slots = int(hp.m_hashNumBuckets) * 4
        alg = 32.0 * slots + active_blocks * (512 * 12.0) + 72.0 * ntri  # table scan + every block's voxels once + triangles written (DESIGN 4i; the one-voxel shells are L2 hits)
        peaks, kind = measured_peaks()
        return {"kernel": "mc_extract_kernel (iso-surface of the loop's model; staged 10^3-voxel tile per block)", "ms": round(ms, 4), "triangles": ntri, "capacity": cap,
                "blocks": int(active_blocks), "hash_slots_scanned": slots, "algorithmic_bytes": round(alg), "achieved_gbs": round(alg / (ms * 1e-3) / 1e9, 1),
                "frac_of_hbm_peak": round(alg / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"], 4), "mtriangles_per_s": round(ntri / (ms * 1e-3) / 1e6, 1),
                "note": "median of 5 launches after one warm-up, CUDA events; not part of the step"}
    except Exception as e:                                            # noqa: BLE001 -- the headline must not depend on this leg
        return {"error": repr(e)[:300]}


def reference_cuda_leg(dev, n_frames=12):
    """The reference's OWN CUDA for the TSDF + bundle-adjustment share of a step -- its kernels and host loops (oracle/_ref: the reference sources
    compiled for sm_100a with --use_fast_math, as it ships), driven exactly like this library on the same inputs, same box, same run: per frame
    1 integrate + 10 x (de-integrate + integrate) + garbage collection; per 10 frames one local BA (11 frames, sparse + dense, 2 x 100) and one global BA
    (500 keyframes, sparse, 3 x 150).  Wall clock with a device synchronise on both sides (the reference's host loops synchronise internally).
    A reported baseline like cpu_baseline: bounded sample, rank 0, N = 1."""
    import torch
    try:
        from oracle import ref_solver, ref_tsdf
        if not (ref_tsdf.available(True) and ref_solver.available(True)):
            return {"unavailable": "oracle/_ref libraries not built (they need /root/reference at build time)"}
    except Exception as e:                                  # noqa: BLE001
        return {"unavailable": f"{type(e).__name__}: {e}"}
    from bundlefusion_b200 import synth, synth_gpu
    from bundlefusion_b200.scene_rep import CUDASceneRepHashSDF, camera_params, default_hash_params
    from bundlefusion_b200.solver import CUDASolverBundling, DeviceCache

    def wall(fn, reps):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / reps * 1e3

    cam = camera_params(W, H)
    hp = default_hash_params(num_buckets=1 << 21, num_sdf_blocks=1 << 20, voxel_size=0.01)
    B = 24
    depth, color, poses = synth_gpu.make_frames([8 * i for i in range(B)], W, H, device=str(dev))
    rng = np.random.Generator(np.random.MT19937(3))
    out = {}
    pcg_info = {"unavailable": "global solve not reached"}
    for name in ("reference_cuda", "this_repo"):
        s = ref_tsdf.ReferenceSceneRepHashSDF(hp, dev, fast_math=True) if name == "reference_cuda" else CUDASceneRepHashSDF(hp, dev)
        s.reset()
        cur = [np.array(p, np.float32) for p in poses]
        for i in range(B):
            s.integrate(cur[i], depth[i], color[i], cam)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for f in range(n_frames):
            ops = []
            for k in range(10):
                i = (7 * f + k) % B
                d = np.eye(4, dtype=np.float32); d[:3, 3] = rng.standard_normal(3).astype(np.float32) * 0.004
                new = (d @ cur[i]).astype(np.float32)
                ops += [(1, i, cur[i]), (0, i, new)]
                cur[i] = new
            ops.append((2, 0, None))
            ops.append((0, f % B, cur[f % B]))
            if name == "this_repo":
                s.runOps(ops, [depth[i] for i in range(B)], [color[i] for i in range(B)], cam)
            else:
                for kind, i, T in ops:                      # the reference's loop: one host-synchronising call per operation
                    if kind == 2: s.garbageCollect()
                    elif kind == 1: s.deIntegrate(T, depth[i], color[i], cam)
                    else: s.integrate(T, depth[i], color[i], cam)
        torch.cuda.synchronize()
        out[name] = {"tsdf_ms_per_frame": (time.perf_counter() - t0) / n_frames * 1e3}
        del s
    # bundle adjustment: the local chunk and the global problem of the ops workload
    loc = synth.make_dense_ba_problem(11, stride=3, W=320, H=240)
    glo = synth.make_ba_problem(WORKLOAD["global_keyframes"], degree=WORKLOAD["global_degree"], corr_per_pair=25, noise=0.002, seed=32, stride=10)
    cache = DeviceCache(loc["caches"], loc["intrinsics"], dev)
    for tag, prob, gn, pcg, wS, wD, wC, ch in (("local_ba_ms", loc, 2, 100, [1.0, 1.0], [1.0, 2.0], [0.0, 0.0], cache), ("global_ba_ms", glo, 3, 150, [1.0] * 3, None, None, None)):
        N = len(prob["init_rot"]); nC = len(prob["corr"])
        corr = torch.from_numpy(prob["corr"].view(np.uint8).reshape(-1).copy()).to(dev)
        r0 = torch.from_numpy(prob["init_rot"]).to(dev); t0_ = torch.from_numpy(prob["init_trans"]).to(dev)
        valid = torch.ones(N, dtype=torch.int32, device=dev)
        rot, trans = r0.clone(), t0_.clone()
        ours = CUDASolverBundling(N, max(nC, 1000 * N), dev)
        ref = ref_solver.ReferenceSolverBundling(N, max(nC, 1000 * N), dev, fast_math=True)
        c2 = corr.clone()

        def run_ours():
            rot.copy_(r0); trans.copy_(t0_)
            ours.solve(corr, nC, valid, N, gn, pcg, wS, wD, wC, d_rotationAnglesUnknowns=rot, d_translationUnknowns=trans, cudaCache=ch)

        def run_ref():
            rot.copy_(r0); trans.copy_(t0_)
            ref.solve(c2, nC, valid, N, gn, pcg, wS, wD, wC, d_rot=rot, d_trans=trans, cudaCache=ch)

        run_ours(); run_ref()
        out["this_repo"][tag] = wall(run_ours, 3); out["reference_cuda"][tag] = wall(run_ref, 3)
        if tag == "global_ba_ms":                           # ms / PCG iteration of the keyframe solve, with the byte count SURVEY 8d attaches to it (140 B per correspondence and iteration)
            try:
                st = ours.getStats()
                it = max(1, int(st["pcg"]))
                t_it = out["this_repo"][tag] / it
                peaks, _ = measured_peaks()
                gbs = 140.0 * nC / (t_it * 1e-3) / 1e9
                pcg_info = {"ms_per_pcg_iter": round(t_it, 5), "pcg_iterations": it, "gn_iterations": int(st["gn"]), "images": N, "correspondences": nC,
                            "algorithmic_bytes_per_iter": 140 * nC, "achieved": round(gbs, 1), "unit": "GB/s", "peak": peaks["hbm_gbs"], "frac": round(gbs / peaks["hbm_gbs"], 4),
                            "bound": "hbm by the survey's accounting; the working set (block-sparse J^T J: 144 B x 2 x image pairs) is L2-resident and the iteration is bound by its chain of dependent L2 accesses and two grid barriers",
                            "host_round_trips_per_iter": 0, "includes": "prep + 3 Gauss-Newton set-ups in the per-iteration figure (whole solve / iterations)"}
            except Exception as e:                          # noqa: BLE001
                pcg_info = {"unavailable": f"{type(e).__name__}: {e}"}
    for name in out:
        o = out[name]
        o["ms_per_frame"] = o["tsdf_ms_per_frame"] + (o["local_ba_ms"] + o["global_ba_ms"]) / 10.0
        o["frames_per_s"] = 1e3 / o["ms_per_frame"]
        for k in list(o):
            o[k] = round(o[k], 3)
    return {"value": out["reference_cuda"]["frames_per_s"], "unit": "frames/s", "this_repo_same_sample": out["this_repo"]["frames_per_s"],
            "speedup": round(out["this_repo"]["frames_per_s"] / out["reference_cuda"]["frames_per_s"], 2), "parts": out, "pcg": pcg_info,
            "kind": "the reference's CUDA kernels and host loops (oracle/_ref: its sources built for sm_100a with --use_fast_math) on this box, TSDF + bundle-adjustment share of a step (the stages the reference's stub surface covers), serial on one stream, wall clock",
            "sample": f"{n_frames} frames of 1 integrate + 10 re-integrations + GC at 1 cm voxels; 3 repetitions of the local (11 frames, sparse + dense) and global (500 keyframes) solves"}

# ------------------------------------------------------------------------------------------------------------------------
LOOP_KEYFRAMES_CPU = 40          # keyframes of the CPU arm's global solve: the middle of what the loop's timed stretches hold (25 .. 55 after a 250-frame pre-roll)


def cpu_arm(steps, warmup, quiet=False, n_reint=None):
    """The reference's algorithm on the host cores: oracle port (liboracle_fast.so: -O3 -march=native, OpenMP over blocks for the
    integrate stencil; alloc / compactify / solver single-threaded as restated).  The heap is sized for the sample (400k blocks)
    instead of 4M to keep host memory modest; work per step is unchanged."""
    from bundlefusion_b200 import synth
    from bundlefusion_b200.scene_rep import camera_params, default_hash_params
    from oracle import oracle as orc
    orc.build()
    cam = camera_params(W, H)
    hp = default_hash_params(num_buckets=WORKLOAD["hash_buckets"], num_sdf_blocks=400000, voxel_size=WORKLOAD["voxel_m"])
    n_re = WORKLOAD["reintegrations_per_frame"] if n_reint is None else n_reint
    B = 12
    frames = [synth.make_frame(8 * i, W, H) for i in range(B)]
    scene = orc.OracleSceneRepHashSDF(hp, fast=True)
    for d, c, T in frames:
        scene.integrate(T, d, c, cam)
    wl = Workload([f[2] for f in frames])
    loc, glo = make_ba_problems(LOOP_KEYFRAMES_CPU, 10)
    def ba():
        orc.solve(loc["corr"], loc["init_rot"], loc["init_trans"], 2, 100, [1.0, 1.0], [1.0, 2.0], [0.0, 0.0], loc["caches"], loc["intrinsics"], fast=True)
        orc.solve_sparse(glo["corr"], glo["init_rot"], glo["init_trans"], 3, 150, fast=True)
    def step(f, with_ba):
        for kind, r, pose in wl.step_ops(f, n_re):
            if kind == 2: scene.garbageCollect()
            elif kind == 1: scene.deIntegrate(pose, frames[r][0], frames[r][1], cam)
            else: scene.integrate(pose, frames[r][0], frames[r][1], cam)
        if with_ba:
            ba()
    for f in range(warmup):
        step(f, False)
    t0 = time.perf_counter()
    for f in range(warmup, warmup + steps):
        step(f, False)
    t_tsdf = (time.perf_counter() - t0) / steps
    t0 = time.perf_counter(); ba(); t_ba = time.perf_counter() - t0
    t_feat, t_chunk_feat, n_keys = cpu_feature_share(orc, synth)
    # scale the TSDF part to the full 10 re-integrations per frame if a reduced sample was timed
    passes_timed, passes_full = 2 * n_re + 1, 2 * WORKLOAD["reintegrations_per_frame"] + 1
    per_frame = t_tsdf * passes_full / passes_timed + t_ba / WORKLOAD["chunk"] + t_feat + t_chunk_feat / WORKLOAD["chunk"]
    cores = os.cpu_count() or 1
    return {"value": round(1.0 / per_frame, 4), "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": f"{steps} frame(s) x ({n_re} re-integrations + 1 integrate + GC) at 640x480 scaled to {WORKLOAD['reintegrations_per_frame']} re-integrations, "
                      f"+ 1 local (11 frames, sparse + dense) and 1 global ({LOOP_KEYFRAMES_CPU} keyframes, {len(glo['corr'])} correspondences) BA solve / {WORKLOAD['chunk']} frames; TSDF {t_tsdf:.2f} s per sampled frame, BA {t_ba:.2f} s per chunk; "
                      f"feature share of a frame (ingest, SIFT detection: {n_keys} key points, dense cache, descriptor match against 5 frames of the chunk) {t_feat:.2f} s on 2 sampled frames, "
                      f"keyframe matching against 30 keyframes {t_chunk_feat:.2f} s per chunk (match filters left out: < 1 ms per frame on one core); "
                      f"OpenMP threads = {cores} on the integrate stencil and the alloc ray walk; hash insertions, compactify, GC, the bundle adjustment and the feature stages single-threaded as restated"}


def cpu_feature_share(orc, synth):
    """seconds per frame of the frame's feature stages on the host (oracle port, one core), and seconds per chunk of the keyframe matching"""
    fr = [synth.make_frame(2 * i, W, H, texture="rich") for i in range(3)]
    K = np.eye(4, dtype=np.float32); K[0, 0] = K[1, 1] = 525.0 * W / 640.0; K[0, 2] = (W - 1) / 2.0; K[1, 2] = (H - 1) / 2.0
    des, n_keys = [], 0
    t0 = time.perf_counter()
    for d, c, T in fr[:2]:
        dd, cc = orc.ingest_frame(d, c, W, H)                                                      # CUDAImageManager::process
        inten = ((0.299 * c[..., 0].astype(np.float32) + 0.587 * c[..., 1].astype(np.float32) + 0.114 * c[..., 2].astype(np.float32)) / 255.0).astype(np.float32)
        kp, de, _ = orc.sift_detect(inten, dd, depthMin=0.1, depthMax=4.0)                         # Bundler::detectFeatures
        orc.cache_store_frame(d, c, K, 80, 60)                                                     # CUDACache::storeFrame
        des.append(de); n_keys = len(de)
    t_front = (time.perf_counter() - t0) / 2
    t0 = time.perf_counter()
    for _ in range(5):                                                                             # a chunk's frame meets 1 .. 10 earlier frames: 5.5 on average
        orc.sift_match(des[0], des[1], fast=True)
    t_match = time.perf_counter() - t0
    t0 = time.perf_counter()
    for _ in range(30):                                                                            # a keyframe against the keyframes so far (25 .. 55 on the bench stream)
        orc.sift_match(des[0], des[1], fast=True)
    return t_front + t_match, time.perf_counter() - t0, n_keys


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    K, Wm = max(1, min(args.steps, 6)), min(args.warmup, 1)
    t0 = time.perf_counter()
    base = cpu_arm(K, Wm, n_reint=WORKLOAD["reintegrations_per_frame"])
    wall = time.perf_counter() - t0
    out = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": "frames/s", "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
           "steps": K, "warmup": Wm, "ms_per_step": round(1e3 / base["value"], 2), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic", "config": dict(LOOP_WORKLOAD, note="CPU arm: oracle port of the reference algorithm on the host cores (the reference ships no CPU path of its own; its CUDA path, rebuilt for sm_100a, is timed in the default arm's `reference_cuda` entry).  It times the stages of the default arm's step by bounded samples -- per frame 1 integrate + 10 re-integrations + GC, ingest, SIFT detection, dense cache, descriptor matching against the chunk; per 10 frames one local and one global solve and the keyframe matching -- and adds them up; the match filters (sub-millisecond per frame on one core) and the host sequencing are left out"),
           "cpu_baseline": base, "e2e": {"value": base["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "wall_s": round(wall, 1)}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ba", action="store_true", help="diagnostic: leave the bundle-adjustment solves out (the JSON line is then NOT a bench value)")
    ap.add_argument("--workload", default="loop", choices=["loop", "ops", "sweep"], help="loop: the whole frame loop (headline); ops: TSDF op replay + synthetic BA problems (round-1 bench, kept for A/B)")
    ap.add_argument("--cuda-profiler", action="store_true", help="bracket the timed pass with cudaProfilerStart/Stop (for `ncu --profile-from-start off`)")
    ap.add_argument("--preroll", type=int, default=250, help="frames streamed through the loop before warm-up (state of a long stream)")
    ap.add_argument("--trace", default=None, help="diagnostic: write the per-frame status of every step (pre-roll included) to this file")
    ap.add_argument("--stride", type=int, default=2, help="Lissajous path frames per step")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR", help="write what the timed pass computed in its last step to DIR/<name>.npy (frame-loop workload)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload != "loop"):
        ap.error("--dump-outputs writes the outputs of the frame-loop workload (--impl ours --workload loop)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "ops":
        run_ours(args)
    elif args.workload == "sweep":
        run_sweep(args)
    else:
        run_loop(args)


if __name__ == "__main__":
    main()
