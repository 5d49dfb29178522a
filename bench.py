#!/usr/bin/env python
"""bench.py — BASELINE.json's metric: Mpaths/s (and Mrays/s) of the path-tracing sample loop, on N B200s of one box, with
the reference's CPU renderer beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 5N] [--impl reference] [--dump-outputs DIR]

--config selects one of BASELINE.json's configs at its stated size and samples per pixel (SURVEY.md §8d):
    1       Ch01 motion-blur random scene, flat list as shipped, 200x100 x 100 spp
    2       two_perlin (checker ground + noise_texture(4) sphere), 400x200 x 256 spp
    3       cornell_box, 500x500 x 1000 spp
    4       cornell_smoke, 500x500 x 1000 spp
    5R      final() as shipped (flat list of 1108 objects), 1000x1000 x 100 spp
    5R+bvh  final() wrapped in one bvh_node, 1000x1000 x 100 spp
    5N      final_northstar (BVH floor + instanced BVH sphere cluster + media + perlin + image texture), 1000x1000 x 100 spp
The default, and the configuration BASELINE.json's metric is quoted on, is 5N.

One step = one full render of the workload: every (pixel, sample) path traced by ONE launch of k_render per GPU.
N > 1 (torchrun, one rank per GPU): rank g renders, for pixel p, the samples s = (g - p) mod N + k*N, then a single NCCL
reduce (sum) of the float accumulation buffer to rank 0 — strong scaling, the partition the north star names.
value  = paths per second with the scene resident in HBM (CUDA events around the step on the launching stream).
e2e    = the same through the host-buffer C-ABI: the scene's device image copied from pinned host memory, render,
         accumulation buffer copied back to pinned host memory, every step.
--dump-outputs DIR writes what the last timed step computed, DIR/accum.npy: the (ny, nx, 3) float32 per-pixel sums over
the ns samples (row 0 at the bottom, after the reduce on rank 0).  Scene, camera and seed are fixed, so two builds run with
the same arguments can be compared output for output.
"""
import argparse
import hashlib
import importlib
import json
import os
import statistics
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

SEED = 20181025
# name -> (scene, nx, ny, ns, workload string printed by BOTH arms, the scene the reference ships for this config (flat list))
CONFIGS = {
    "1": ("ch01_random", 200, 100, 100, "ch01_random 200x100x100spp (config 1: Ch01 motion-blur random scene, flat hitable_list as shipped)", "ch01_random"),
    "2": ("two_perlin", 400, 200, 256, "two_perlin 400x200x256spp (config 2: checker ground + noise_texture(4) sphere)", "two_perlin"),
    "3": ("cornell_box", 500, 500, 1000, "cornell_box 500x500x1000spp (config 3)", "cornell_box"),
    "4": ("cornell_smoke", 500, 500, 1000, "cornell_smoke 500x500x1000spp (config 4: two constant_medium boxes)", "cornell_smoke"),
    "5R": ("final", 1000, 1000, 100, "final 1000x1000x100spp (config 5R: final() as shipped, flat hitable_list of 1108 objects)", "final"),
    "5R+bvh": ("final+bvh", 1000, 1000, 100, "final+bvh 1000x1000x100spp (config 5R in one F2-patched bvh_node)", "final"),
    "5N": ("final_northstar", 1000, 1000, 100,
           "final_northstar 1000x1000x100spp (config 5N: BVH over 1024 floor boxes + translate(rotate_y(BVH over 1000 spheres)) + "
           "media + perlin + image texture)", "final"),
}
# Algorithmic FP32 operations per ray on the reference topology (SURVEY.md §8d): 18/aabb test, 25/sphere, 30/moving
# sphere, 10/rect, 60/medium, +100 shading (+800 per noise_texture hit, +60 per checker hit: not separable from the
# reference's counters, so the shading term is the 100 floor).
F_OPS = dict(aabb=18.0, sphere=25.0, moving_sphere=30.0, rect=10.0, medium=60.0, shade=100.0)
COUNT_KEYS = ("aabb", "sphere", "moving_sphere", "rect", "medium")


def flops_per_ray(c):
    return sum(F_OPS[k] * c[k] for k in COUNT_KEYS) + F_OPS["shade"]


def source_id():
    """identifies the kernel build a profiles/*_dram_traffic.json capture belongs to"""
    h = hashlib.sha256()
    for f in ("peter-shirley-ray-tracing-the-next-week_b200/csrc/rtnw_cuda.cu", "peter-shirley-ray-tracing-the-next-week_b200/csrc/rtnw_device.cuh",
              "include/rtnw.h"):
        h.update((ROOT / f).read_bytes())
    return h.hexdigest()[:16]


# ------------------------------------------------------------------------------------------------ reference arm
def _ref_worker(args):
    scene, nx, ny, ns, seed, begin = args
    import ref_oracle as ro
    rs = ro.RefScene(scene, tagged=False)
    _, st = rs.render(nx, ny, ns, seed=seed, rng_mode=0, sample_begin=begin)  # glibc drand48, as shipped
    return st


def run_reference(scene, nx, ny, ns_total, procs):
    """The reference's own CPU implementation (oracle/_ref/libref_oracle.so = its headers compiled unmodified, +F2 fix)
    on `procs` processes, each rendering ns_total/procs samples of every pixel with its own srand48 seed (the reference
    is single-threaded and drand48 is process-global, so processes are the only way to use more cores)."""
    import multiprocessing as mp
    per = max(1, ns_total // procs)
    jobs = [(scene, nx, ny, per, 1000 + k, k * per) for k in range(procs)]
    t0 = time.perf_counter()
    if procs == 1:
        stats = [_ref_worker(jobs[0])]
    else:
        with mp.get_context("fork").Pool(procs) as pool:
            stats = pool.map(_ref_worker, jobs)
    wall = time.perf_counter() - t0
    paths = sum(s["paths"] for s in stats)
    rays = sum(s["rays"] for s in stats)
    loop_s = max(s["seconds"] for s in stats)  # the render loops run concurrently; scene construction excluded
    counts = {k: sum(s[k] for s in stats) / rays for k in COUNT_KEYS}
    return dict(paths=paths, rays=rays, seconds=loop_s, wall=wall, counts=counts)


def reference_sample(scene, procs, seconds):
    """(nx, ny, spp per process): a bounded sample of the scene's own camera sized for about `seconds` of CPU work per core"""
    rate = {"ch01_random": 55e3, "two_perlin": 1.2e6, "cornell_box": 300e3, "cornell_smoke": 420e3, "final": 17e3,
            "final+bvh": 190e3, "final_northstar": 160e3}[scene]  # paths/s per core, survey probes (BASELINE.md §2)
    nx = ny = 200 if scene.startswith(("final", "cornell")) else 0
    if not nx:
        nx, ny = 200, 100
    spp = max(1, int(rate * seconds / (nx * ny)))
    return nx, ny, spp


def reference_main(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import ref_oracle as ro
    scene, _, _, _, workload, _ = CONFIGS[args.config]
    if not ro.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libref_oracle.so was not built"}))
        return 0
    procs = os.cpu_count() or 1
    nx, ny, spp = reference_sample(scene, procs, 6.0)  # about 6 s of CPU work per core and step
    times, paths, rays = [], 0, 0
    for it in range(args.warmup + args.steps):
        r = run_reference(scene, nx, ny, spp * procs, procs)
        if it >= args.warmup:
            times.append(r["seconds"])
            paths += r["paths"]
            rays += r["rays"]
    total = sum(times)
    v = paths / total / 1e6
    sample = f"{nx}x{ny} pixels x {spp * procs} spp of the same scene/camera per step, {procs} processes (the reference is single-threaded), glibc drand48"
    line = {
        "impl": "reference", "metric": "Mpaths/s", "value": v, "unit": "Mpaths/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "config": args.config, "sample": sample},
        "mrays_per_s": rays / total / 1e6,
        "cpu_baseline": {"value": v, "unit": "Mpaths/s", "cores": procs, "per_core": v / procs, "kind": "reference", "sample": sample},
        "e2e": {"value": v, "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.02)

    def result(self):
        self.stop_flag = True
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        top = sorted(self.samples)[len(self.samples) // 2:]  # upper half = samples taken under load
        return {"sm_mhz": statistics.median(top), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def measured_traffic(config, world):
    """dram__bytes_read.sum + dram__bytes_write.sum of one k_render launch of this config from the committed ncu capture
    (profiles/round2_dram_traffic.json, written by scripts/capture_traffic.py), or (None, why) when there is no capture of
    THIS kernel build / config / GPU count — never a stale constant."""
    try:
        t = json.loads((ROOT / "profiles" / "round2_dram_traffic.json").read_text())
    except Exception:
        return None, "no profiles/round2_dram_traffic.json"
    if t.get("source_id") != source_id():
        print(f"bench.py: profiles/round2_dram_traffic.json was captured from another kernel build ({t.get('source_id')} != "
              f"{source_id()}): roofline.traffic is null; re-run scripts/capture_traffic.py", file=sys.stderr)
        return None, "capture is from another kernel build (stale)"
    e = t.get("configs", {}).get(f"{config}@{world}")
    if e is None:
        return None, f"no capture for config {config} on {world} GPU(s)"
    return e, None


# ------------------------------------------------------------------------------------------------ our arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="rtnw", choices=["rtnw", "reference"])
    ap.add_argument("--config", default="5N", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--flags", type=int, default=0, help="extra RTNW_F_* render flags (4 = RTNW_F_FAST_BVH, the non-reference-exact fast traversal mode)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's accumulation buffer to DIR/accum.npy (not with --impl reference)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes this project's render; the reference arm keeps no image")
    if args.impl == "reference":
        return reference_main(args)

    import torch
    rtnw = importlib.import_module("peter-shirley-ray-tracing-the-next-week_b200")
    mg = importlib.import_module("peter-shirley-ray-tracing-the-next-week_b200.multi_gpu")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    scene, nx, ny, ns, workload, shipped_scene = CONFIGS[args.config]
    ctx = rtnw.Context(local)
    hs = rtnw.HostScene(scene)
    prepared = rtnw.PreparedScene(hs.desc_ptr)  # host-side: the scene's device image, built once (pinned memory)
    ds = ctx.upload(prepared)
    cam = hs.camera(nx, ny)
    plan = mg.partition_plan(ns, nx * ny, world, rank)  # one launch; even for any ns (RTNW_F_ROTATE_SAMPLES)

    def launch_params(launch):
        extra = args.flags | (rtnw.F_ROTATE_SAMPLES if launch["rotate"] else 0) | (rtnw.F_ACCUMULATE if launch["accumulate"] else 0)
        return hs.params(nx=nx, ny=ny, ns=launch["sample_count"], seed=SEED, sample_begin=launch["sample_begin"],
                         sample_stride=launch["sample_stride"], flags_extra=extra)
    params = launch_params(plan[0])  # world == 1: the whole frame in one launch
    accum = torch.empty(ny, nx, 3, dtype=torch.float32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    stream = torch.cuda.current_stream()  # the legacy default stream: rtnw_render_device is stream-ordered on it

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}

    def step(scene_dev):
        last["rays"], last["kernel_ms"], last["launches"] = 0, 0.0, 0

        def render(**launch):
            st = scene_dev.render_device(cam, launch_params(launch), accum.data_ptr(), stream.cuda_stream)
            last["rays"] += st.rays; last["kernel_ms"] += st.kernel_ms; last["launches"] += st.kernel_launches; last["ranges"] = st.sample_ranges
        mg.render_partitioned(render, accum, ns, dist=dist, dst=0)  # k_render launches of this rank, then one NCCL reduce(sum)
        return last

    for _ in range(args.warmup):
        step(ds)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    rays = 0
    kernel_ms = []
    for a, b in ev:
        flush.zero_()  # L2 flush between timed iterations (outside the timed events)
        barrier()
        a.record(stream)
        st = step(ds)
        b.record(stream)
        rays += st["rays"]
        kernel_ms.append(st["kernel_ms"])
        launches_per_step = st["launches"]
        sample_ranges = st["ranges"]
    barrier()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    clocks = sampler.result()
    if args.dump_outputs and rank == 0:  # before the e2e steps, which reuse `accum` when world > 1
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "accum.npy"), accum.cpu().numpy())
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    tot_rays = torch.tensor([float(rays)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot_rays, op=dist.ReduceOp.SUM)
    total_s = total_ms.item() / 1e3
    # per-rank kernel time and step time (diagnoses a slow GPU / a slow reduce when the max over ranks is off)
    mine = torch.tensor([sum(kernel_ms) / len(kernel_ms), sum(step_ms) / len(step_ms)], dtype=torch.float64, device=dev)
    per_rank = [torch.zeros_like(mine) for _ in range(world)]
    if dist is not None:
        dist.all_gather(per_rank, mine)
    else:
        per_rank = [mine]
    per_rank = [[round(float(x), 3) for x in t.tolist()] for t in per_rank]
    paths_per_step = nx * ny * ns
    value = paths_per_step * args.steps / total_s / 1e6
    mrays = tot_rays.item() / total_s / 1e6

    # ---- e2e: host buffers through the C-ABI, copies inside the timed region: every step copies the scene's device image
    # (rtnw_scene_upload_prepared, pinned -> HBM), renders, and brings the frame back to pinned host memory
    image_bytes = prepared.nbytes
    host_accum = torch.empty(ny, nx, 3, dtype=torch.float32).pin_memory()
    host_np = host_accum.numpy()
    e2e_kernel_ms = []

    def e2e_step():
        s2 = ctx.upload(prepared)  # H2D of every scene table
        if dist is None:
            _, st2 = s2.render(cam, params, out=host_np)  # render + D2H into pinned host memory
            e2e_kernel_ms.append(st2.kernel_ms)
        else:
            e2e_kernel_ms.append(step(s2)["kernel_ms"])
            if rank == 0:
                host_accum.copy_(accum, non_blocking=False)
        s2.close()

    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = paths_per_step * args.steps / e2e_s.item() / 1e6

    # ---- per-ray test counts of the reference topology (for flop_per_ray) and the CPU baseline, on rank 0
    counts, cpu = None, None
    if rank == 0:
        import ref_oracle as ro
        if ro.available():
            # live counters of the reference itself (oracle/ref_harness.cpp ref_cnt) on this scene: one process, a few seconds, any N
            cnx, cny, cspp = reference_sample(scene, 1, 1.5)
            counts = run_reference(scene, cnx, cny, cspp, 1)["counts"]
            if world == 1 and not args.no_cpu_baseline:
                procs = os.cpu_count() or 1
                bx, by, bspp = reference_sample(scene, procs, 14.0)  # ~14 s of CPU work per core
                r = run_reference(scene, bx, by, bspp * procs, procs)
                v = r["paths"] / r["seconds"] / 1e6
                cpu = {"value": v, "unit": "Mpaths/s", "cores": procs, "per_core": v / procs, "kind": "reference",
                       "mrays_per_s": r["rays"] / r["seconds"] / 1e6,
                       "sample": f"{bx}x{by} pixels x {bspp * procs} spp of the same scene/camera, {procs} processes "
                                 f"(the reference is single-threaded), glibc drand48; {r['seconds']:.1f} s"}
                # BASELINE.md §3(a): the reference AS SHIPPED — flat hitable_list, one thread
                sx, sy, sspp = reference_sample(shipped_scene, 1, 4.0)
                r1 = run_reference(shipped_scene, sx, sy, sspp, 1)
                cpu["as_shipped_single_thread"] = {"scene": f"{shipped_scene} (flat hitable_list, 1 thread)",
                                                   "value": r1["paths"] / r1["seconds"] / 1e6, "unit": "Mpaths/s",
                                                   "sample": f"{sx}x{sy} pixels x {sspp} spp; {r1['seconds']:.1f} s"}
    if rank == 0:
        peaks = {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except Exception:
            pass
        info = ctx.info()
        kernel_s = sum(kernel_ms) / 1e3 / len(kernel_ms)  # the k_render launch of one step on rank 0
        rays_per_launch = rays / args.steps
        f_ray = flops_per_ray(counts) if counts else None
        sm_mhz = clocks["sm_mhz"] or (info["clock_khz"] / 1e3)
        fp32_nominal = info["sm_count"] * 128 * 2 * sm_mhz * 1e6 / 1e12  # TFLOP/s at the clock seen under load (FMA = 2)
        fp32_peak = ctx.fp32_peak_tflops()  # measured on this device: independent FFMA chains (rtnw_measure_fp32_peak)
        achieved = rays_per_launch * f_ray / kernel_s / 1e12 if f_ray else None
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        # algorithmic HBM bytes of one launch: the scene image read once + the frame written once (+ the fixed-point plane of the
        # sample-range sums written and read back once when a pixel's samples are cut into ranges)
        hbm_bytes = image_bytes + nx * ny * 3 * 4 + (2 * nx * ny * 3 * 8 if sample_ranges > 1 else 0)
        traffic, traffic_note = measured_traffic(args.config, world) if not (args.flags & 4) else (None, "no capture of the fast-mode kernel")
        line = {
            "metric": "Mpaths/s", "value": value, "unit": "Mpaths/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * total_s / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "config": args.config,
                       "paths_per_step": paths_per_step, "partition": f"spp split over {world} GPU(s) (sample ownership rotates with the pixel index), 1 NCCL reduce; "
                                    f"{sample_ranges} sample ranges per pixel per launch",
                       "l2": "flushed between timed steps (256 MiB write)", "traversal": "fast (RTNW_F_FAST_BVH)" if args.flags & 4 else "reference-exact",
                       "seed": SEED},
            "mrays_per_s": mrays, "rays_per_path": tot_rays.item() / (paths_per_step * args.steps),
            "e2e": {"value": e2e_value, "unit": "Mpaths/s", "h2d_bytes_per_step": image_bytes * world,
                    "d2h_bytes_per_step": nx * ny * 3 * 4, "ms_per_step": 1e3 * e2e_s.item() / args.steps,
                    "kernel_ms_per_step": sum(e2e_kernel_ms[-args.steps:]) / args.steps},
            "gpu_launches": args.steps * launches_per_step,
            "per_rank_ms": {"kernel": [r[0] for r in per_rank], "step": [r[1] for r in per_rank]},
            "clocks": clocks,
            "roofline": {"bound": "fp32", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s",
                         "frac": achieved / fp32_peak if achieved else None,
                         "traffic": traffic["bytes"] if traffic else None,
                         "traffic_source": (f"profiles/round2_dram_traffic.json ({traffic['read']} read + {traffic['write']} written, ncu, this kernel build)"
                                            if traffic else traffic_note),
                         "kernel": "k_render", "kernel_ms": 1e3 * kernel_s, "flop_per_ray": f_ray,
                         "tests_per_ray": counts,
                         "counts_source": "the reference's own counters on this scene, this run" if counts else "reference not available",
                         "peak_source": f"measured FFMA microbenchmark on this GPU (nominal {fp32_nominal:.1f} = {info['sm_count']} SM x "
                                        f"128 lanes x 2 x {sm_mhz:.0f} MHz)",
                         "note": "FP32-issue bound, not HBM/tensor: the scene (<2 MB) lives in L1/L2; see the hbm sub-object",
                         "hbm": {"achieved": hbm_bytes / kernel_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": hbm_bytes / kernel_s / 1e9 / hbm_peak, "algorithmic_bytes": hbm_bytes,
                                 "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"}},
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    ds.close()
    prepared.close()
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
