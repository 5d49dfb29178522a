#!/usr/bin/env python
"""Cost of the first-hit feature buffers (rtnw_render_aov) next to the frame they belong to: config 5N's scene
(final_northstar, 1000x1000, bench.py's seed), rtnw_render at 100 spp against rtnw_render_aov at 1, 4, 16 and 100 spp.
Device time of each call from CUDA events (stats.kernel_ms); after one warm-up call of each, REPS repetitions with the two calls
alternating.  Prints one JSON object, with the device name and power limit the numbers were measured at."""
import argparse
import importlib
import json
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
rtnw = importlib.import_module("peter-shirley-ray-tracing-the-next-week_b200")

SEED = 20181025  # bench.py's
ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--aov-spp", default="1,4,16,100")
a = ap.parse_args()

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
ctx = rtnw.Context(0)
hs = rtnw.HostScene("final_northstar")
ds = ctx.upload(hs.desc_ptr)
nx, ny, ns = 1000, 1000, 100
cam = hs.camera(nx, ny)
render_params = hs.params(nx=nx, ny=ny, ns=ns, seed=SEED)
result = dict(device=gpu.stdout.strip().splitlines()[ctx.device] if gpu.returncode == 0 else "unknown",
              workload=f"final_northstar {nx}x{ny}, seed {SEED}", reps=a.reps, render_spp=ns, aov={})


def render_ms():
    _, st = ds.render(cam, render_params)
    return st.kernel_ms


def aov_ms(spp):
    st = rtnw.Stats()
    ds.render_aov(cam, hs.params(nx=nx, ny=ny, ns=spp, seed=SEED), st)
    return st.kernel_ms


render_times = []
for spp in map(int, a.aov_spp.split(",")):
    render_ms(), aov_ms(spp)  # warm-up
    r, v = [], []
    for _ in range(a.reps):
        r.append(render_ms())
        v.append(aov_ms(spp))
    render_times += r
    result["aov"][str(spp)] = dict(aov_ms_median=statistics.median(v), aov_ms=v, render_ms_median=statistics.median(r),
                                   aov_over_render=statistics.median(v) / statistics.median(r),
                                   aov_mrays_per_s=nx * ny * spp / statistics.median(v) / 1e3)
result["render_ms_median"] = statistics.median(render_times)
result["render_mpaths_per_s"] = nx * ny * ns / result["render_ms_median"] / 1e3
print(json.dumps(result))
ds.close()
ctx.close()
