#!/usr/bin/env python
"""Cost of a frame's first-hit feature buffers (AOVs) and of denoising it when the frame is rendered on the GPUs of one box:
config 5N's scene (final_northstar, 1000x1000, 100 spp, bench.py's seed).

For G = 1, 2, 4, 8 devices (those the box has; the others are reported as "not measured"), each repetition runs, alternating:
  rtnw_render_multi                          the colour frame alone
  rtnw_render_aov_multi                      the colour frame and its AOVs
  rtnw_render_aov_multi with denoising       the same, denoised on device 0
and reports the medians of their total_ms (first launch to the end of the last host copy) and kernel_ms (the slowest device's
colour render).  For every G, also on device 0 alone: the kernel time of one rank's AOV share (rtnw_render_aov_device with
RTNW_F_ROTATE_SAMPLES, rank 0 of G), which is what the AOVs add to each device's stream in the multi-GPU frame.
On one GPU: rtnw_denoise (host buffers, with its copies: total_ms) against rtnw_denoise_device on the same inputs in device
memory (kernel_ms and the host time of the call), alternating.  Each measured call is warmed up first.  Prints one JSON
object, with the device name and power limit read in the same run."""
import argparse
import importlib
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
rtnw = importlib.import_module("peter-shirley-ray-tracing-the-next-week_b200")

SEED = 20181025  # bench.py's
ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=7)
ap.add_argument("--gpus", default="1,2,4,8")
a = ap.parse_args()

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
n_dev = rtnw.device_count()
hs = rtnw.HostScene("final_northstar")
nx, ny, ns = 1000, 1000, 100
cam = hs.camera(nx, ny)
params = hs.params(nx=nx, ny=ny, ns=ns, seed=SEED)
dp = rtnw.DenoiseParams(5, 4.0, 1.0, 7)
result = dict(device=gpu.stdout.strip().splitlines() if gpu.returncode == 0 else "unknown", devices_present=n_dev,
              workload=f"final_northstar {nx}x{ny}, {ns} spp, seed {SEED}", reps=a.reps, multi={}, aov_rank_share_kernel_ms={})


def med(xs):
    return statistics.median(xs)


# ---- the multi-GPU frame
for G in map(int, a.gpus.split(",")):
    if G > n_dev:
        result["multi"][str(G)] = "not measured"
        continue
    mc = rtnw.MultiContext(list(range(G)))
    ms = mc.upload(hs.desc_ptr)
    calls = dict(render=lambda: ms.render(cam, params)[1], render_aov=lambda: ms.render_aov(cam, params)[3],
                 render_aov_denoise=lambda: ms.render_aov(cam, params, dp)[3])
    for f in calls.values():  # warm-up
        f()
    total = {k: [] for k in calls}
    kernel = {k: [] for k in calls}
    for _ in range(a.reps):
        for k, f in calls.items():
            st = f()
            total[k].append(st.total_ms)
            kernel[k].append(st.kernel_ms)
    r = {f"{k}_total_ms_median": med(v) for k, v in total.items()}
    r.update({f"{k}_kernel_ms_median": med(v) for k, v in kernel.items()})
    r.update({f"{k}_total_ms": v for k, v in total.items()})
    r["aov_added_ms"] = r["render_aov_total_ms_median"] - r["render_total_ms_median"]
    r["denoise_added_ms"] = r["render_aov_denoise_total_ms_median"] - r["render_aov_total_ms_median"]
    r["render_mpaths_per_s"] = nx * ny * ns / r["render_total_ms_median"] / 1e3
    result["multi"][str(G)] = r
    ms.close()
    mc.close()

# ---- one rank's AOV share, and the denoiser with and without host copies, on device 0
ctx = rtnw.Context(0)
ds = ctx.upload(hs.desc_ptr)
planes = {k: torch.empty((ny, nx, 3) if k in ("albedo", "normal") else (ny, nx), dtype=torch.int32 if k in ("hits", "prim_id") else torch.float32,
                         device="cuda:0") for k in rtnw.AOV_KEYS}
ptrs = {k: v.data_ptr() for k, v in planes.items()}
for G in map(int, a.gpus.split(",")):
    share = hs.params(nx=nx, ny=ny, ns=ns, seed=SEED, sample_begin=0, sample_stride=G, flags_extra=rtnw.F_ROTATE_SAMPLES)
    ds.render_aov_device(cam, share, ptrs)  # warm-up
    v = [ds.render_aov_device(cam, share, ptrs).kernel_ms for _ in range(a.reps)]
    result["aov_rank_share_kernel_ms"][str(G)] = dict(median=med(v), all=v)

sums, _ = ds.render(cam, params)
aov = ds.render_aov(cam, params)
colour = torch.from_numpy(sums).cuda()
dev_aov = {k: torch.from_numpy(np.ascontiguousarray(aov[k])).cuda() for k in ("albedo", "normal", "depth", "hits")}
out = torch.empty_like(colour)
torch.cuda.synchronize()


def host_denoise():
    st = rtnw.Stats()
    ctx.denoise(sums, aov, ns, stats=st)
    return st


def device_denoise():
    t0 = time.perf_counter()
    st = ctx.denoise_device(colour.data_ptr(), {k: v.data_ptr() for k, v in dev_aov.items()}, nx, ny, ns, out.data_ptr())
    return st, (time.perf_counter() - t0) * 1e3


host_denoise(), device_denoise()  # warm-up
h_total, h_kernel, d_kernel, d_host = [], [], [], []
for _ in range(a.reps):
    st = host_denoise()
    h_total.append(st.total_ms)
    h_kernel.append(st.kernel_ms)
    st, wall = device_denoise()
    d_kernel.append(st.kernel_ms)
    d_host.append(wall)
same = out.cpu().numpy().tobytes() == ctx.denoise(sums, aov, ns).tobytes()
result["denoise_one_gpu"] = dict(denoise_total_ms_median=med(h_total), denoise_kernel_ms_median=med(h_kernel),
                                 denoise_device_kernel_ms_median=med(d_kernel), denoise_device_call_ms_median=med(d_host),
                                 denoise_total_ms=h_total, denoise_device_call_ms=d_host, same_bits=same)
print(json.dumps(result))
ds.close()
ctx.close()
