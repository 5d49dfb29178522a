#!/usr/bin/env python
"""What RTNW_F_LIGHT_SAMPLING and RTNW_F_NEXT_EVENT buy on the scenes lit by one small area light: BASELINE configs 3
(cornell_box), 4 (cornell_smoke) and 5N (final_northstar), each at its stated size and spp N, on one GPU.  --modes picks the
estimators from exact (no flag), lights (RTNW_F_LIGHT_SAMPLING) and nee (RTNW_F_NEXT_EVENT); exact is always measured.

Per config:
  speed     rtnw_render in each mode, alternating, after a warm-up of each; Mpaths/s from the kernel time (CUDA events,
            rtnw_stats.kernel_ms), and closest-hit queries (rtnw_stats.rays) per path, medians over --reps.
  error     RMSE of the per-pixel mean colour against a converged image: the mean of --conv exact-mode frames of N spp each
            (other seeds), i.e. --conv times N spp.  Measured for both modes at N and at N/4 spp, averaged over --seeds frames;
            the exponent of RMSE ~ spp^-e between the two spp values checks the 1/sqrt(spp) scaling the ratio below assumes.
            The converged image still has 1/conv of the exact mode's variance at N: it is included in every RMSE.
  ratio     equal-error time ratio of each flagged mode: the time the exact mode needs to reach the flagged mode's RMSE at N
            spp, N (rmse_exact / rmse_flag)^2 spp at the exact mode's rate, over the flagged mode's time for N spp.  > 1 means the
            flag reaches that error sooner.
Prints one JSON object, with the device name and power limit read in the same run, and writes it to --out when given."""
import argparse
import importlib
import json
import statistics
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
rtnw = importlib.import_module("peter-shirley-ray-tracing-the-next-week_b200")

CONFIGS = {"3": ("cornell_box", 500, 500, 1000), "4": ("cornell_smoke", 500, 500, 1000), "5N": ("final_northstar", 1000, 1000, 100)}
ap = argparse.ArgumentParser()
ap.add_argument("--configs", default="3,4,5N")
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--seeds", type=int, default=3)
ap.add_argument("--conv", type=int, default=16)
ap.add_argument("--modes", default="exact,lights")
ap.add_argument("--out")
a = ap.parse_args()

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
result = dict(device=gpu.stdout.strip().splitlines() if gpu.returncode == 0 else "unknown", reps=a.reps, seeds=a.seeds,
              converged_frames=a.conv, configs={})
ctx = rtnw.Context(0)

for cfg in a.configs.split(","):
    name, nx, ny, ns = CONFIGS[cfg]
    hs = rtnw.HostScene(name)
    ds = ctx.upload(hs.desc_ptr)
    cam = hs.camera(nx, ny)

    def render(spp, seed, flags):
        sums, st = ds.render(cam, hs.params(nx=nx, ny=ny, ns=spp, seed=seed, flags_extra=flags))
        return sums.astype(np.float64) / spp, st

    flags = {"exact": 0, "lights": rtnw.F_LIGHT_SAMPLING, "nee": rtnw.F_NEXT_EVENT}
    modes = {k: flags[k] for k in ["exact"] + [m for m in a.modes.split(",") if m != "exact"]}
    for f in modes.values():
        render(ns, 1, f)  # warm-up
    rate = {k: [] for k in modes}
    rays = {k: [] for k in modes}
    for r in range(a.reps):
        for k, f in modes.items():
            st = render(ns, 10 + r, f)[1]
            rate[k].append(st.paths / st.kernel_ms / 1e3)
            rays[k].append(st.rays / st.paths)
    conv = sum(render(ns, 5000 + r, 0)[0] for r in range(a.conv)) / a.conv
    rmse = {}
    for k, f in modes.items():
        for spp in (ns, ns // 4):
            mse = [np.mean((render(spp, 100 + s, f)[0] - conv) ** 2) for s in range(a.seeds)]
            rmse[f"{k}_{spp}"] = float(np.sqrt(np.mean(mse)))
    mp = {k: statistics.median(v) for k, v in rate.items()}
    exponent = {k: float(np.log(rmse[f"{k}_{ns // 4}"] / rmse[f"{k}_{ns}"]) / np.log(4.0)) for k in modes}
    flagged = [k for k in modes if k != "exact"]
    spp_eq = {k: ns * (rmse[f"exact_{ns}"] / rmse[f"{k}_{ns}"]) ** 2 for k in flagged}
    ratio = {k: (spp_eq[k] / mp["exact"]) / (ns / mp[k]) for k in flagged}
    if flagged == ["lights"]:  # the layout of the light-sampling run
        spp_eq, ratio = spp_eq["lights"], ratio["lights"]
    result["configs"][cfg] = dict(workload=f"{name} {nx}x{ny}, {ns} spp", mpaths_per_s_median=mp, mpaths_per_s=rate, rmse=rmse,
                                  rmse_spp_exponent=exponent, exact_spp_for_equal_rmse=spp_eq, equal_error_time_ratio=ratio)
    if "nee" in modes:
        result["configs"][cfg]["rays_per_path_median"] = {k: statistics.median(v) for k, v in rays.items()}
    print(json.dumps({cfg: result["configs"][cfg]}), flush=True)
    ds.close()
    hs.close()

ctx.close()
print(json.dumps(result))
if a.out:
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(result, indent=1) + "\n")
