#!/usr/bin/env python
"""bench.py -- RGB-D frames/s of the Co-Fusion per-frame hot path on B200.

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank/GPU)
  python bench.py --impl reference --gpus N --steps K ...  (CPU port of the reference path, rank 0 only)

A "step" is one CoFusion::processFrame of one 640x480 synthetic RGB-D frame (BASELINE.json configs[1]:
single model, synthetic room sequence): H2D upload, bilateral filter + depth pyramid, model/frame
pyramids, SO(3) + 19-iteration ICP+RGB Gauss-Newton tracking, predict, index map, fuse, index map,
clean, predict + fill-in.  `value` is measured with the frames already resident in HBM, `e2e` through
the same C-ABI call with pinned HOST buffers (H2D of the frame and D2H of the pose inside the timed
region).  One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

W, H = 640, 480
METRIC = "RGB-D frames/s @640x480 (per-model ICP+fuse)"
# SURVEY.md 8(d): algorithmic bytes of the tracker's Gauss-Newton loop per model per frame at 640x480
# = sum over the 10/5/4 iterations of (48 P + 116) ICP + 30 P RGB residual + (32 P + 116) RGB step
GN_ITERS = ((0, 10), (1, 5), (2, 4))


def gn_algorithmic_bytes(w, h):
    total = 0
    for lvl, it in GN_ITERS:
        P = (w >> lvl) * (h >> lvl)
        total += it * ((48 * P + 116) + 30 * P + (32 * P + 116))
    return total


WORKLOAD = ("configs[1]: single model, 640x480 synthetic room sequence, full processFrame (bilateral, pyramids, SO3 + "
            "10/5/4-iteration ICP+RGB tracking, index map, fuse, index map, clean, predict + fill-in; predictBeforeFuse=0: the "
            "prediction of CoFusion.cpp:347 that only the out-of-scope loop closure reads is not rendered)")


def base_config(world=1):
    """the `config` object both arms print (the driver compares them)"""
    return {"workload": WORKLOAD, "width": W, "height": H, "models_per_rank": 1, "scene_models": max(1, world),
            "predictBeforeFuse": 0, "sequence": "synth.room_sequence(seed=1234, noise=True), ping-pong over the rendered frames"}


def make_frames(n):
    from cofusion_b200 import synth
    return [(rgb, d) for _, rgb, d, _, _ in synth.room_sequence(n, W, H, synth.K_DEFAULT, noise=True, seed=1234)]


def frame_index(step, n):
    """ping-pong over the rendered frames so that camera motion stays continuous for any step count"""
    period = 2 * (n - 1)
    k = step % period
    return k if k < n else period - k


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self.stop_flag = False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 9:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(s[1]) for s in self.samples)
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for k, nm in enumerate(names):
                if s[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][2]), "reasons": sorted(reasons),
                "samples": len(sm)}


def dump_outputs(cf, out_dir, max_rows=1 << 18):
    """What a caller of processFrame reads back after the last timed step, as DIR/<name>.npy: every model's pose
    and tracking statistics, and the camera model's surfel map (a fixed, seeded sample of max_rows rows when it
    is larger, so that the files stay small)."""
    os.makedirs(out_dir, exist_ok=True)
    n = cf.num_models
    stats = [cf.last_stats(i) for i in range(n)]
    surfels = cf.model(0).download_map()
    count = len(surfels)
    if count > max_rows:
        surfels = surfels[np.sort(np.random.default_rng(0).choice(count, max_rows, replace=False))]
    out = {"poses": np.stack([cf.pose(i) for i in range(n)]).astype(np.float32),
           "track_stats": np.array([[s.lastICPError, s.lastICPCount, s.lastRGBError, s.lastRGBCount, s.lastSO3Error,
                                     s.lastSO3Count] for s in stats], np.float64),
           "surfel_count": np.array([count], np.float64),
           "surfels": surfels.astype(np.float32)}
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def cpu_port_fps(frames, n_frames, warm=2):
    """The CPU restatement of the same per-frame path (oracle/, single thread) on a bounded sample."""
    from orc_pipeline import OraclePipeline
    from cofusion_b200 import synth
    op = OraclePipeline(W, H, synth.K_DEFAULT, 1 << 21, predict_before_fuse=False)
    for t in range(warm):
        op.process_frame(*frames[frame_index(t, len(frames))])
    t0 = time.perf_counter()
    for t in range(warm, warm + n_frames):
        op.process_frame(*frames[frame_index(t, len(frames))])
    dt = time.perf_counter() - t0
    return n_frames / dt, dt


def cpu_segmentation_ms(frames, reps=3, n_models=1):
    """The part of the path that is CPU code in the reference (SLIC + dense CRF + components,
    Core/Segmentation): oracle/segment.c on one host core, n models + the "new" label, 640x480."""
    import orc
    rgb, d = frames[3]
    icp = [np.full((H, W), 0.002 * (m + 1), np.float32) for m in range(n_models)]
    vcs = []
    for m in range(n_models):
        vc = np.zeros((H, W, 4), np.float32)
        vc[..., 3] = 10.0 if m == 0 else 1.0
        vcs.append(vc)
    t0 = time.perf_counter()
    for _ in range(reps):
        orc.segment_crf(rgb, d, list(range(n_models)), icp, vcs, n_models, True)
    return 1e3 * (time.perf_counter() - t0) / reps


def reference_cuda_tracker():
    """SURVEY.md 8(d) "reference timed beside it" (1): the reference's OWN tracker kernels (oracle/_ref =
    Core/Cuda/reduce.cu + cudafuncs.cu compiled as they are for sm_100a) driven through the call sequence of
    RGBDOdometry::getIncrementalTransformation on one 640x480 frame pair of the same sequence, on this GPU.
    Timed inside the reference driver around the step calls only (no pyramid building).  Part of the
    cpu_baseline / reference leg: never on the product path."""
    try:
        import orc
        import scenes
        if orc.ref() is None:
            return None
        case = scenes.room_pair(W, H)
        best, steps = None, 0
        for _ in range(3):
            oo, _ = scenes.oracle_odometry(case)
            _, _, _, extra = oo.track(case["T0"], use_ref=True)
            best = extra["step_ms"] if best is None else min(best, extra["step_ms"])
            steps = extra["steps"]
        return {"tracker_ms_per_frame": best, "launch_sync_steps": steps, "kind": "reference",
                "what": "icpStep / computeRgbResidual / rgbStep / so3Step of the reference, reference launch "
                        "configuration and per-step synchronisation; compare with roofline.avg_launch_ms"}
    except Exception as e:  # the reference kernels are optional evidence, never a reason to fail the bench
        return {"unavailable": repr(e)[:200]}


def run_reference(args, budget_s=120.0):
    """--impl reference: the CPU port of the same per-frame path (oracle/ C restatement of the reference's
    CPU-visible algorithm; the reference's own host loops are single-threaded), one host core.  A step is
    one processFrame of the same 640x480 sequence; the CPU needs ~0.7 s per step, so the run is bounded:
    at most `budget_s` seconds of timed work, i.e. the first n <= K steps are timed and reported."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    frames = make_frames(24)
    from orc_pipeline import OraclePipeline
    from cofusion_b200 import synth
    op = OraclePipeline(W, H, synth.K_DEFAULT, 1 << 21, predict_before_fuse=False)
    warm = max(2, min(args.warmup, 3))  # frame 1 only initialises the map: at least one tracked frame of warm-up
    t0 = time.perf_counter()
    for t in range(warm):
        op.process_frame(*frames[frame_index(t, len(frames))])
    per_frame = (time.perf_counter() - t0) / warm
    n = max(1, min(args.steps, int(budget_s / max(per_frame, 1e-3))))
    t0 = time.perf_counter()
    for t in range(warm, warm + n):
        op.process_frame(*frames[frame_index(t, len(frames))])
    dt = time.perf_counter() - t0
    fps = n / dt
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / n,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": base_config(1), "reference_run": {"parallelism": "1 host thread", "steps_timed": n, "warmup_run": warm},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": 1, "kind": "port",
                             "sample": "%d of the %d requested steps timed (bounded to %.0f s of CPU work) after %d "
                                       "warm-up frames, oracle/ C restatement" % (n, args.steps, budget_s, warm)},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def objects4_bench(steps, warmup, local):
    """BASELINE.json configs[2] on this GPU: background + 4 moving boxes at 640x480 with the motion segmentation IN
    the loop (enableMultipleModels: tracking of every model -> SLIC + CRF -> spawn / lose models -> fuse / clean with
    the CRF's labels -> predict).  The number of live models is whatever the closed loop produces; it is reported."""
    import torch
    import cofusion_b200 as cfb
    from cofusion_b200 import synth
    n_render = 32
    seq = list(synth.room_sequence(n_render, W, H, synth.K_DEFAULT, noise=True, n_boxes=4, box_speed=1.0, seed=1234))
    dev = [(torch.from_numpy(np.ascontiguousarray(r)).cuda(), torch.from_numpy(np.ascontiguousarray(d)).cuda()) for _, r, d, _, _ in seq]
    p = cfb.CoFusionParams.default(1 << 21)
    p.enableMultipleModels = 1
    cf = cfb.CoFusion(W, H, synth.K_DEFAULT, p, device=local)
    ext = torch.cuda.ExternalStream(cf.ctx.stream)
    nm = []
    for t in range(warmup):
        cf.process_frame(*dev[frame_index(t, n_render)])
    cf.ctx.sync()
    cf.ctx.take_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ext)
    for t in range(warmup, warmup + steps):
        cf.process_frame(*dev[frame_index(t, n_render)])
        nm.append(cf.num_models)
    e1.record(ext)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    launches = cf.ctx.take_launch_count()
    out = {"workload": "configs[2]: 640x480 synthetic room + 4 moving boxes, motion-CRF segmentation in the loop, 1 GPU",
           "value": steps / (ms / 1e3), "unit": "frames/s", "ms_per_step": ms / steps, "steps": steps, "warmup": warmup,
           "models_mean": float(np.mean(nm)), "models_min": int(min(nm)), "models_max": int(max(nm)),
           "gpu_launches_per_step": launches / steps}
    del e0, e1, ext, dev
    cf.ctx.sync()
    return out, cf


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--impl", default="cofusion_b200")
    ap.add_argument("--cpu-frames", type=int, default=8, help="frames of the cpu_baseline sample (0 = skip)")
    ap.add_argument("--objects-steps", type=int, default=300, help="steps of the configs[2] leg at N = 1 (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        # the reference's path on the host cores: a bounded sample of the K requested steps (run_reference)
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import cofusion_b200 as cfb
    from cofusion_b200 import sharding, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    K = synth.K_DEFAULT
    n_render = 32
    n_models = sharding.scene_models(world)  # N ranks track ONE scene with N models: background + N - 1 moving boxes
    P = W * H
    # only the root renders / holds the frames: the other ranks receive them by the library's NCCL broadcast
    host, devf = [], []
    if rank == 0:
        for _, rgb, d, _, ids in synth.room_sequence(n_render, W, H, K, noise=True, seed=1234, n_boxes=n_models - 1, box_speed=0.5):
            trip = (torch.from_numpy(np.ascontiguousarray(rgb)).pin_memory(), torch.from_numpy(np.ascontiguousarray(d)).pin_memory(),
                    torch.from_numpy(np.ascontiguousarray(ids.astype(np.uint8))).pin_memory() if world > 1 else None)
            host.append(trip)
            devf.append(tuple(None if x is None else x.cuda() for x in trip))
    def build():
        params = cfb.CoFusionParams.default(1 << 21)
        cf = cfb.CoFusion(W, H, K, params, device=local)
        if world > 1:
            uid = [cfb.nccl_unique_id() if rank == 0 else None]  # one id per communicator
            dist.broadcast_object_list(uid, src=0)
            cf.shard_init(rank, world, uid[0])  # collective: the library's own NCCL communicator
        cfb.lib().cfb_model_odometry.restype = cfb.C.c_void_p
        return cf

    def step(cf, t, frames):
        if rank == 0:
            rgb, d, m = frames[frame_index(t, n_render)]
            cf.process_frame(rgb, d, m)
        else:
            cf.process_frame(None, None, None)
        if world > 1 and t == 1:
            # frame 1: every rank spawns the object model it owns from the renderer's labels (FrameData::mask path).
            # A new model starts at the camera pose (CoFusion.cpp:593), which only the camera model's rank tracks.
            cam = torch.from_numpy(cf.model(0).pose.reshape(16).copy()).cuda() if rank == 0 else torch.empty(16, device="cuda")
            dist.broadcast(cam, src=0)
            for mdl in sharding.models_of_rank(n_models, rank, world):
                if mdl > 0:
                    cf.spawn_object_model(mdl, cam.cpu().numpy())

    keep = []

    def timed(frames, sampler=None, dump_dir=None):
        cf = build()
        keep.append(cf)
        ext = torch.cuda.ExternalStream(cf.ctx.stream)  # only used to record / wait on events
        for t in range(args.warmup):
            step(cf, t, frames)
        cf.ctx.sync()
        cf.ctx.take_launch_count()
        mine = [m for m in sharding.models_of_rank(n_models, rank, world)]
        tracked = cf.model(0 if rank == 0 else cf.num_models - 1)
        odom = cfb.C.c_void_p(cfb.lib().cfb_model_odometry(tracked._h))
        cfb.check(cfb.lib().cfb_odom_enable_kernel_timing(odom, 1))
        sm, n = cfb.C.c_double(0), cfb.C.c_int(0)
        cfb.check(cfb.lib().cfb_odom_kernel_timing(odom, cfb.C.byref(sm), cfb.C.byref(n), 1))
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if sampler:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(ext)
        for t in range(args.warmup, args.warmup + args.steps):
            step(cf, t, frames)
        e1.record(ext)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1)
        if sampler:
            sampler.stop_flag = True
        launches = cf.ctx.take_launch_count()
        if dump_dir and rank == 0:
            dump_outputs(cf, dump_dir)
        # the tracker kernel is timed with CUDA events on its own stream: every launch of a short extra run (the
        # event pair is read back per launch, which would serialise the timed region above)
        ksum, kn = 0.0, 0
        for t in range(args.warmup + args.steps, args.warmup + args.steps + 50):
            step(cf, t, frames)
            cf.ctx.sync()
            cfb.check(cfb.lib().cfb_odom_kernel_timing(odom, cfb.C.byref(sm), cfb.C.byref(n), 1))
            ksum, kn = ksum + sm.value, kn + n.value
        t_ms = torch.tensor([ms], device="cuda")
        if world > 1:
            dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)  # max over ranks
        nsurf = tracked.last_count()
        del e0, e1, ext
        return float(t_ms.item()), launches, (ksum, kn), nsurf, mine

    sampler = ClockSampler(local) if rank == 0 else None
    ms, launches, (kms, kn), nsurf, mine = timed(devf, sampler, args.dump_outputs)
    ms_e2e, _, _, _, _ = timed(host)
    if rank != 0:
        # done: the reductions inside timed() were the last collectives.  Leave without a rank-by-rank tear-down of
        # the communicators (rank 0 still has its report to assemble and must not be waited for)
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)

    value = sharding.aggregate_value(n_models, args.steps, ms)
    e2e = sharding.aggregate_value(n_models, args.steps, ms_e2e)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
    alg = gn_algorithmic_bytes(W, H)
    k_avg_ms = kms / max(kn, 1)
    achieved = alg / (k_avg_ms * 1e-3) / 1e9 if kn else None
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))["gn_tiled_kernel"]["dram_bytes_per_launch"]
    except Exception:
        pass
    cpu = None
    frames_np = None
    if args.cpu_frames > 0 and world == 1:
        frames_np = make_frames(24)
        fps_cpu, dt = cpu_port_fps(frames_np, args.cpu_frames)
        cpu = {"value": fps_cpu, "unit": "frames/s", "cores": 1, "kind": "port",
               "sample": "%d frames of the same 640x480 room sequence through the oracle/ C restatement "
                         "(single thread, like the reference's CPU loops), %.1f s" % (args.cpu_frames, dt),
               "segmentation_ms_per_frame": cpu_segmentation_ms(frames_np),
               "segmentation_ms_per_frame_5_models": cpu_segmentation_ms(frames_np, reps=2, n_models=5)}
    cfg = base_config(world)
    cfg.update({"surfels": nsurf,
                "parallelism": ("object sharding: rank r owns model r of ONE %d-model scene (background + %d moving boxes, labels "
                                "from the renderer), one ncclBroadcast of the packed frame per step inside the library" %
                                (n_models, n_models - 1)) if world > 1 else "1 GPU",
                "l2": "inputs cycle over %d distinct frames (%.0f MB) + a %.0f MB surfel map; per-step working set is L2 resident "
                      "by nature of the workload, no flush" % (n_render, n_render * 7 * P / 1e6, nsurf * 96 / 1e6)})
    objects4 = None
    if world == 1 and args.objects_steps > 0:
        keep.clear()
        torch.cuda.synchronize()
        try:
            objects4, cf4 = objects4_bench(args.objects_steps, 60, local)
            keep.append(cf4)
        except Exception as e:  # the second workload must never take the headline line down
            objects4 = {"unavailable": repr(e)[:300]}
    cfg["objects4"] = objects4
    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": (8 if world > 1 else 7) * P, "d2h_bytes_per_step": 224 + 376,
                "ms_per_step": ms_e2e / args.steps,
                "note": "host RGB-D frame in pinned memory -> C-ABI processFrame -> pose block + tracker statistics copied back "
                        "every step (read by the host without stalling the pipeline)"},
        "gpu_launches": launches,
        "roofline": {"kernel": "gn_tiled_kernel (SO3 + 19 GN iterations of ICP/RGB reductions over shared-memory tiles, 1 launch/frame)",
                     "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                     "algorithmic_bytes_per_launch": alg, "avg_launch_ms": k_avg_ms, "launches_timed": kn,
                     "peak_source": peak_src,
                     "share_of_step": (k_avg_ms / (ms / args.steps)) if kn else None},
        "cpu_baseline": cpu,
        "reference_cuda": reference_cuda_tracker() if (world == 1 and args.cpu_frames > 0) else None,
        "clocks": sampler.summary() if sampler else None,
    }
    print(json.dumps(line), flush=True)
    torch.cuda.synchronize()
    if world > 1:
        # every rank has finished its timed loops (the max-over-ranks reductions above are collective): leave
        # without tearing communicators down rank by rank -- a rank that is slow to exit must not hold the others
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    keep.clear()


if __name__ == "__main__":
    main()
