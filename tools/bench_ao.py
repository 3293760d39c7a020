"""Throughput of the 'ao' integrator on one GPU.  Rewrites the (integrator ...) block of each scene in memory and prints one
JSON line: per workload the samples/s and occlusion rays/s (device events, median of --runs timed renders after one warm-up
render), the TRACE / SHADE split of a separate profiling render, and the rate of the CPU oracle on a crop.  The card's name and
power limit are read in the same run.

    python tools/bench_ao.py [--out FILE] [--runs 3] [--only WORKLOAD ...]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import pearray_b200 as prb  # noqa: E402
from test_ao import oracle_ao, scene_with_integrator  # noqa: E402

# name: (scene file, sample_count, spp, oracle crop, oracle spp)
WORKLOADS = {
    "c2_cornellbox_500x500_256spp": ("c2_cornellbox.prc", 10, 256, (218, 218, 282, 282), 16),
    "c4_boltsandgears_1000x1000_64spp": ("c4_boltsandgears.prc", 10, 64, (468, 468, 532, 532), 4),
    "c4c_complex_1920x1080_16spp": ("c4c_complex.prc", 10, 16, (928, 508, 992, 572), 2),
}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers stay valid; the card is then unnamed
        return {"name": "unknown (%s)" % e}


def run(name, path, n, spp, crop, ospp, runs):
    scene = scene_with_integrator(os.path.join(ROOT, "scenes", path), "(integrator :type 'ao' :sample_count %d)" % n)
    tiles = scene.tiles(8, 8)
    pixels = sum((t[2] - t[0]) * (t[3] - t[1]) for t in tiles)
    ctx = prb.Context(0)
    ctx.upload_scene(scene)
    rng = scene.rng_map()
    times, rays = [], []
    for r in range(runs + 1):  # the first render warms up (graph instantiation, module load)
        ctx.upload_rng(rng)
        ctx.reset_stats()
        ctx.render_tiles(tiles, 0, spp)
        if r:
            times.append(ctx.last_device_ms() / 1e3)
            rays.append(ctx.stats().shadow_ray_count)
    t = statistics.median(times)
    ctx.upload_rng(rng)
    ctx.set_profiling(True)
    ctx.render_tiles(tiles, 0, spp)
    st = ctx.stage_times()
    ctx.set_profiling(False)
    ctx.close()
    t0 = time.perf_counter()
    oracle_ao(scene, [crop], 0, ospp, n)
    ot = time.perf_counter() - t0
    return {"workload": name, "sample_count": n, "spp": spp, "pixels": pixels, "device_s_median": t, "device_s_runs": times,
            "samples_per_s": pixels * spp / t, "occlusion_rays_per_s": statistics.median(rays) / t,
            "trace_ms": st["trace"][0], "shade_ms": st["shade"][0],
            "oracle_samples_per_s": (crop[2] - crop[0]) * (crop[3] - crop[1]) * ospp / ot, "oracle_threads": os.cpu_count()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--only", nargs="*")
    args = ap.parse_args()
    res = {"card": card(), "workloads": [run(k, *v, args.runs) for k, v in WORKLOADS.items() if not args.only or k in args.only]}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
