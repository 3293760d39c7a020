"""Throughput of the 'visualfeedback' integrator on one GPU.  Rewrites the (integrator ...) block of each scene in memory and
prints one JSON line: per workload and mode the samples/s (device events, median of --runs timed renders after one warm-up
render) and the TRACE share of a separate profiling render (k_vf is the one kernel of an iteration), and per workload the rate of
the CPU oracle on a crop.  The card's name and power limit are read in the same run.

    python tools/bench_vf.py [--out FILE] [--runs 3] [--only WORKLOAD ...] [--modes MODE ...]"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import pearray_b200 as prb  # noqa: E402
from bench_ao import card  # noqa: E402
from test_ao import scene_with_integrator  # noqa: E402
from test_visualfeedback import oracle_vf  # noqa: E402

# name: (scene file, spp, oracle crop, oracle spp).  The spp give timed windows of tens of milliseconds or more per render.
WORKLOADS = {
    "c2_cornellbox_500x500_1024spp": ("c2_cornellbox.prc", 1024, (218, 218, 282, 282), 16),
    "c4_boltsandgears_1000x1000_256spp": ("c4_boltsandgears.prc", 256, (468, 468, 532, 532), 4),
    "c4c_complex_1920x1080_64spp": ("c4c_complex.prc", 64, (928, 508, 992, 572), 2),
}


def run(name, path, spp, crop, ospp, modes, runs):
    scene = scene_with_integrator(os.path.join(ROOT, "scenes", path), "(integrator :type 'visualfeedback')")
    tiles = scene.tiles(8, 8)
    pixels = sum((t[2] - t[0]) * (t[3] - t[1]) for t in tiles)
    ctx = prb.Context(0)
    ctx.upload_scene(scene)
    rng = scene.rng_map()
    per_mode = {}
    for mode in modes:
        ctx.set_integrator("visualfeedback", mode=mode)
        times = []
        for r in range(runs + 1):  # the first render warms up (graph instantiation, module load)
            ctx.upload_rng(rng)
            ctx.render_tiles(tiles, 0, spp)
            if r:
                times.append(ctx.last_device_ms() / 1e3)
        t = statistics.median(times)
        ctx.upload_rng(rng)
        ctx.set_profiling(True)
        ctx.render_tiles(tiles, 0, spp)
        st = ctx.stage_times()
        total_ms = ctx.last_device_ms()
        ctx.set_profiling(False)
        per_mode[mode] = {"device_s_median": t, "device_s_runs": times, "samples_per_s": pixels * spp / t, "trace_ms": st["trace"][0],
                          "profiled_render_ms": total_ms, "trace_share": st["trace"][0] / total_ms}
    ctx.close()
    t0 = time.perf_counter()
    oracle_vf(scene, [crop], 0, ospp, "colored_entity_id")
    ot = time.perf_counter() - t0
    return {"workload": name, "spp": spp, "pixels": pixels, "modes": per_mode,
            "oracle_samples_per_s": (crop[2] - crop[0]) * (crop[3] - crop[1]) * ospp / ot, "oracle_threads": os.cpu_count()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--only", nargs="*")
    ap.add_argument("--modes", nargs="*", default=list(prb.VF_MODES))
    args = ap.parse_args()
    res = {"card": card(), "workloads": [run(k, *v, args.modes, args.runs) for k, v in WORKLOADS.items() if not args.only or k in args.only]}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
