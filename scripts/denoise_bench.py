#!/usr/bin/env python
"""Cost of the denoiser (rtnw_denoise) next to the frame it cleans: config 5N's scene (final_northstar, 1000x1000, bench.py's
seed), the 100-spp rtnw_render and rtnw_render_aov against rtnw_denoise with the default parameters on 16- and 100-spp inputs.
Device time of each call from CUDA events (stats.kernel_ms) and, for the denoiser, with its host<->device copies
(stats.total_ms); after one warm-up call of each, REPS repetitions with the calls alternating, medians reported.  The
denoiser's 101 bytes per pixel fit the L2, so repeated calls read their inputs from there.  Prints one JSON object, with the
device name and power limit the numbers were measured at."""
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
ap.add_argument("--spp", default="16,100")
a = ap.parse_args()

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
ctx = rtnw.Context(0)
hs = rtnw.HostScene("final_northstar")
ds = ctx.upload(hs.desc_ptr)
nx, ny, render_ns = 1000, 1000, 100
cam = hs.camera(nx, ny)
result = dict(device=gpu.stdout.strip().splitlines()[ctx.device] if gpu.returncode == 0 else "unknown",
              workload=f"final_northstar {nx}x{ny}, seed {SEED}", reps=a.reps, denoise={})


def render_ms(spp):
    _, st = ds.render(cam, hs.params(nx=nx, ny=ny, ns=spp, seed=SEED))
    return st.kernel_ms


def aov_ms(spp):
    st = rtnw.Stats()
    ds.render_aov(cam, hs.params(nx=nx, ny=ny, ns=spp, seed=SEED), st)
    return st.kernel_ms


render_times = []
for spp in map(int, a.spp.split(",")):
    params = hs.params(nx=nx, ny=ny, ns=spp, seed=SEED)
    sums, _ = ds.render(cam, params)
    aov = ds.render_aov(cam, params)

    def denoise():
        st = rtnw.Stats()
        ctx.denoise(sums, aov, spp, stats=st)
        return st.kernel_ms, st.total_ms

    render_ms(render_ns), aov_ms(spp), denoise()  # warm-up
    r, v, k, t = [], [], [], []
    for _ in range(a.reps):
        r.append(render_ms(render_ns))
        v.append(aov_ms(spp))
        km, tm = denoise()
        k.append(km)
        t.append(tm)
    render_times += r
    result["denoise"][str(spp)] = dict(denoise_kernel_ms_median=statistics.median(k), denoise_total_ms_median=statistics.median(t),
                                       denoise_kernel_ms=k, aov_ms_median=statistics.median(v),
                                       denoise_kernel_over_render=statistics.median(k) / statistics.median(r))
result["render_spp"] = render_ns
result["render_ms_median"] = statistics.median(render_times)
print(json.dumps(result))
ds.close()
ctx.close()
