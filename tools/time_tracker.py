"""Quick device timing of the tracker (CUDA events), ours vs the reference kernels. Scratch tool."""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch
import gpu_util as gu, orc, scenes
from test_tracker_gpu import _cuda_odometry

for (W, H) in ((640, 480), (1280, 960)):
    case = scenes.room_pair(W, H)
    co = _cuda_odometry(gu, case)
    torch.cuda.synchronize()
    for host_loop, name, N in ((False, "persistent cooperative kernel", 50), (True, "host_loop", 20)):
        for _ in range(4):
            co.track(case["T0"], force_host_loop=host_loop)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(N):
            p, st = co.track(case["T0"], force_host_loop=host_loop)
        e1.record(); torch.cuda.synchronize()
        print("%dx%d %s: %.3f ms/track" % (W, H, name, e0.elapsed_time(e1) / N), flush=True)
    if orc.ref() is not None and W == 640:
        oo, _ = scenes.oracle_odometry(case)
        for _ in range(2):
            oo2, _ = scenes.oracle_odometry(case)
            p, st, _, extra = oo2.track(case["T0"], use_ref=True)
        print("%dx%d reference CUDA kernels via reference call sequence: %.3f ms in %d steps" % (W, H, extra["step_ms"], extra["steps"]), flush=True)
