#!/usr/bin/env python3
"""bench.py -- spectral path samples/s of the 'direct' (unidirectional PT) hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scene c2|c1|c3|c4|c4b|c4c|c0|c5] [--spp S]
                  [--partition samples|tiles] [--no-extras] [--dump-outputs DIR]

Headline workload (BASELINE.json configs[1], SURVEY 8(d) C2): cornellbox.prc, 500x500, 'direct' integrator depth 6, mjitt
sampler, 1024 spp, diffuse materials + one area light.  One "step" = one complete render of that configuration
(500*500*1024 = 262 144 000 spectral path samples, 4 wavelengths each) through prb_render_tiles.

Our arm prints ONE JSON line:
  value   samples/s with the scene, RNG map and film resident in HBM (CUDA events via the C ABI, max over ranks)
  e2e     samples/s through the C ABI with HOST buffers: per step the RNG map is uploaded, the tiles rendered and the
          film (xyz + sample counts) downloaded inside the timed region
  roofline / cpu_baseline / clocks / gpu_launches as the contract asks (DESIGN.md section "Measurement")
  workloads   (default run only) the same kind of numbers for the two other workloads BASELINE.json names:
      complex   complex.prc as shipped (1920x1080, sky + sun, sobol; a bounded number of its 4096 spp per step)
      c5        synthetic 10 M-triangle soup: primary / shadow / incoherent ray streams (Mrays/s), hit ids checked against
                the oracle on a sample, e2e with host ray buffers in and hit buffers out
  strong_scaling   (N > 1) complex.prc partitioned by INTERLEAVED TILES (fixed total work, time-to-image falls with N);
                   the reduced film is checked bit-identical against a 1-GPU render outside the timed region
  embree      whether Embree 3 is on the box (the "vs CPU Embree" half of the metric needs it; absent in this image)
Multi-GPU (torchrun, one rank per GPU): scene replicated, films combined by prb_film_reduce_comm (NCCL over NVLink, inside
the C ABI) in the timed region.  Headline partition: sample ranges (rank r renders iterations [r spp, (r+1) spp) of ONE
N*spp-sample sequence from a decorrelated RNG map -> weak scaling); --partition tiles: interleaved tiles (strong scaling).

--dump-outputs DIR: after the timed steps of the headline workload, what its last step returned goes to DIR/<name>.npy --
film_xyz (H, W, 3) and sample_count (H, W) of the last render (float32); for c5 a fixed, seeded sample of 2^19 rays of every
class from the last timed pass (hit ids as float64, u / v / t and occlusion as float32).  The inputs depend on the arguments
only, so two builds run with the same arguments can be compared output for output.

--impl reference: the reference's own CPU implementation cannot be built here (Eigen/Embree/TBB/OIIO absent, SURVEY F4), so
the arm times oracle/ (the CPU restatement, std::thread x all host cores) on a bounded sample of the same workload.  This
file and tests/ are the only places that execute oracle/.
"""
import argparse
import glob
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SCENES = {
    "c1": ("c1_sphere.prc", "sphere.prc 1000x1000 direct sobol 64spp"),
    "c2": ("c2_cornellbox.prc", "cornellbox.prc 500x500 direct(depth 6) mjitt 1024spp"),
    "c3": ("c3_cornellbox_glassy.prc", "cornellbox_glassy.prc 256x256 direct(depth 16, power MIS) mjitt 128spp"),
    "c4": ("c4_boltsandgears.prc", "boltsandgears.prc 1000x1000 direct mjitt 256spp"),
    "c4b": ("c4b_complex_env.prc", "complex.prc 1920x1080 direct sobol 4096spp (sky+sun replaced by a D65 env light)"),
    "c4c": ("c4c_complex.prc", "complex.prc 1920x1080 direct sobol 4096spp (as shipped: Hosek-Wilkie sky + sun)"),
    "c0": ("c0_evaluation.prc", "evaluation/scene.prc 256x256 direct(depth 6) sobol 128spp"),
}


# ----------------------------------------------------------------------------------------------- helpers
class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self.proc = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self._stop.is_set():
                    break
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        self._stop.set()
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(scene_key, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, from the committed ncu --set full capture of this
    workload (profiles/traffic.json, copied from the profiles/*_ncu_*.txt summaries); None when no capture is on file"""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)[scene_key][kernel]["dram_bytes_per_launch"]
    except Exception:
        return None


def bvh_depth_bytes(n_tris):
    """minimal-path bytes of one closest-hit / any-hit ray, SURVEY 8(d): 32 + (24|4) + 80*ceil(log8(N/4)) + 4*48"""
    import math
    levels = max(1, math.ceil(math.log(max(n_tris / 4.0, 1.0001), 8)))
    return 32 + 24 + 80 * levels + 4 * 48, 32 + 4 + 80 * levels + 4 * 48


def embree_probe():
    """SURVEY 8(d) CPU-baseline option 2: is Embree 3 on this box?  (header for the optional oracle stage + the library)"""
    hdr = [p for pat in ("/usr/include/embree3/rtcore.h", "/usr/local/include/embree3/rtcore.h", "/opt/*/include/embree3/rtcore.h") for p in glob.glob(pat)]
    lib = [p for pat in ("/usr/lib/x86_64-linux-gnu/libembree3.so*", "/usr/lib/libembree3.so*", "/usr/local/lib/libembree3.so*", "/opt/*/lib/libembree3.so*")
           for p in glob.glob(pat)]
    if hdr and lib:
        return {"status": "present", "header": hdr[0], "library": lib[0],
                "note": "oracle/Makefile builds oracle/_ref/liboracle_embree.so when the header is found; hit-id cross-check in tests/test_embree_crosscheck.py"}
    return {"status": "absent", "note": "no embree3/rtcore.h or libembree3.so on this box: hit ids are pinned to the oracle's restatement of Embree's "
                                         "documented robust semantics, the 'vs CPU Embree' half of the metric is unmeasured (cpu_baseline.kind = port)"}


def load_scene(prb, key, aa_samples=None):
    """the .prc scene of a config; aa_samples overrides the sample count of the 'aa' sampler (sample-range partition: ONE
    sequence of world * spp samples whose index ranges are dealt to the ranks)"""
    fname, label = SCENES[key]
    path = os.path.join(ROOT, "scenes", fname)
    if aa_samples is None:
        return prb.Scene.from_file(path), fname, label
    src = open(path).read()
    pat = re.compile(r"(\(sampler\s+:slot\s+'aa'[^)]*?:sample_count\s+)(\d+)", re.S)
    assert pat.search(src), "no aa sampler with a sample_count in " + fname
    src = pat.sub(lambda m: m.group(1) + str(aa_samples), src, count=1)
    return prb.Scene.from_string(src, path), fname, label


# ----------------------------------------------------------------------------------------------- reference arm
def run_reference(args, rank, world):
    if rank != 0:
        return
    import numpy as np
    import pearray_b200 as prb
    from oracle_binding import OracleScene
    fname, label = SCENES[args.scene]
    scene = prb.Scene.from_file(os.path.join(ROOT, "scenes", fname))
    ora = OracleScene(scene)
    cores = os.cpu_count() or 1
    tiles = scene.tiles(8, 8)
    npix = scene.width * scene.height
    rng = scene.rng_map()
    # calibrate: 1 spp, then size a step to ~4 s of CPU work
    t0 = time.perf_counter()
    r = ora.render(tiles, 0, 1, rng=rng, threads=cores, aov=False)
    t1 = time.perf_counter() - t0
    spp = max(1, min(int(scene.settings.max_sample_count), int(round(4.0 / max(t1, 1e-3)))))
    film = np.zeros((scene.height, scene.width, 3), np.float32)
    cnt = np.zeros((scene.height, scene.width), np.uint32)
    for _ in range(args.warmup):
        ora.render(tiles, 0, 1, rng=rng, threads=cores, film=film, count=cnt, aov=False)
    t0 = time.perf_counter()
    rays = 0
    for k in range(args.steps):
        r = ora.render(tiles, k * spp, spp, rng=rng, threads=cores, film=film, count=cnt, aov=False)
        rays += r["stats"]["primary_ray_count"] + r["stats"]["bounce_ray_count"] + r["stats"]["shadow_ray_count"]
    dt = time.perf_counter() - t0
    value = npix * spp * args.steps / dt
    sample = "%d spp per step over the full %dx%d film (of %d spp; rate-normalised), %d threads" % (spp, scene.width, scene.height, scene.settings.max_sample_count, cores)
    line = {"impl": "reference", "metric": "spectral path samples/s", "value": value, "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "mrays_per_s": rays / dt / 1e6,
            "config": {"workload": label, "scene": fname, "note": "reference not buildable here (Eigen/Embree/TBB/OIIO absent): CPU oracle port (scalar C++17, own "
                                                                  "median-split BVH, no SIMD -- NOT Embree, NOT PearRay), bounded sample"},
            "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample},
            "embree": embree_probe(),
            "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ----------------------------------------------------------------------------------------------- distributed plumbing
class Job:
    """rank / world, the torch.distributed process group (rendezvous, barrier, max over ranks) and the NCCL communicator of the
    C ABI (prb_comm_init) that carries the film reduce"""

    def __init__(self, rank, world, local_rank):
        import torch
        self.torch = torch
        self.rank, self.world, self.local_rank = rank, world, local_rank
        self.dev = torch.device("cuda", local_rank)
        torch.cuda.set_device(self.dev)
        self.dist = None
        if world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist

    def barrier(self):
        self.torch.cuda.synchronize(self.dev)
        if self.dist:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, x):
        if not self.dist:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x):
        if not self.dist:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def gather_rows(self, row):
        if not self.dist:
            return [row]
        t = self.torch.tensor(row, dtype=self.torch.float64, device=self.dev)
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [[float(v) for v in x] for x in out]

    def join_communicator(self, ctx):
        """rank 0 creates the NCCL unique id through the C ABI, the 128 bytes travel over torch.distributed (out of band)"""
        if not self.dist:
            return
        import pearray_b200 as prb
        uid = self.torch.zeros(128, dtype=self.torch.uint8, device=self.dev)
        if self.rank == 0:
            uid.copy_(self.torch.from_numpy(prb.Context.comm_unique_id()))
        self.dist.broadcast(uid, src=0)
        ctx.comm_init(uid.cpu().numpy(), self.rank, self.world)

    def finish(self):
        if self.dist:
            self.dist.barrier()
            self.dist.destroy_process_group()


DUMP_LIMIT_BYTES = 64 << 20
DUMP_SAMPLE_RAYS = 1 << 19  # c5: rays of every class kept by --dump-outputs (a fixed, seeded sample of the 4 M-ray passes)


def dump_outputs(dump_dir, arrays):
    """--dump-outputs: the arrays the timed path returned in its last step, one DIR/<name>.npy each (float32 / float64), so that
    the outputs of two builds of the project can be compared on the same inputs"""
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, "dump of %d bytes exceeds %d" % (total, DUMP_LIMIT_BYTES)
    os.makedirs(dump_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dump_dir, name + ".npy"), np.ascontiguousarray(a))


def render_workload(job, prb, key, spp, steps, warmup, partition, want_e2e=True, want_profile=True, cpu_seconds=0.0, clock_sampler=None, dump_dir=None):
    """times `steps` renders of `spp` iterations of scene `key` on job.world GPUs; returns the dict of numbers of this workload
    (rank 0; None on the other ranks).  partition: 'samples' (weak) | 'tiles' (strong) | 'single'.  dump_dir: write the film of
    the last timed render (rank 0 holds the combined film) there."""
    import numpy as np
    torch = job.torch
    from pearray_b200 import multigpu
    rank, world = job.rank, job.world
    if world == 1:
        partition = "single"
    scene, fname, label = load_scene(prb, key, aa_samples=spp * world if partition == "samples" else None)
    W, H = scene.width, scene.height
    all_tiles = scene.tiles(8, 8)
    if partition == "tiles":
        # interleaved ownership over a FINE tile map (32 x 32 tiles, SURVEY 8(e)): per-pixel cost varies strongly over the image
        # (glass / metal regions), 64 coarse tiles left the two ranks of a 2-GPU run 10 % apart
        tiles, first_iter, scaling, seed_rank = multigpu.partition_tiles(scene.tiles(32, 32), rank, world), 0, "strong", 0
    elif partition == "samples":
        tiles, first_iter, scaling, seed_rank = all_tiles, rank * spp, "weak", rank
    else:
        tiles, first_iter, scaling, seed_rank = all_tiles, 0, "weak", 0
    npix_rank = sum((t[2] - t[0]) * (t[3] - t[1]) for t in tiles)
    scene.settings.seed = multigpu.rank_seed(scene.settings.seed, seed_rank)  # decorrelated per-rank RNG map in sample-range mode
    ctx = prb.Context(job.local_rank)
    ctx.upload_scene(scene)
    job.join_communicator(ctx)
    rng_host = scene.rng_map()
    rng_pinned = torch.empty(W * H, dtype=torch.int64).pin_memory()
    rng_pinned.numpy().view(np.uint64)[:] = rng_host
    film_pinned = torch.empty((H, W, 3), dtype=torch.float32).pin_memory()
    cnt_pinned = torch.empty((H, W), dtype=torch.int32).pin_memory()
    total_iters = spp * world if partition == "samples" else spp
    split_ms = [0.0, 0.0]  # render, film reduce (the reduce of a rank that finished early includes waiting for the slowest rank)

    def reduce_films():
        if world == 1:
            return 0.0
        ctx.film_reduce_comm("samples" if partition == "samples" else "tiles", total_iters, 0)  # export + ncclReduce + import on rank 0
        return ctx.last_reduce_ms()

    def step_resident():
        if world > 1:
            ctx.upload_rng(rng_host)  # the film of rank 0 was overwritten by the last reduce: every step is a render from scratch
        if tiles:
            ctx.render_tiles(tiles, first_iter, spp)  # returns when the wavefront retired every sample
        r = ctx.last_device_ms() if tiles else 0.0
        f = reduce_films()
        split_ms[0] += r
        split_ms[1] += f
        return r + f

    def step_e2e():
        t0 = time.perf_counter()
        ctx.upload_rng(rng_pinned.numpy().view(np.uint64))
        if tiles:
            ctx.render_tiles(tiles, first_iter, spp)
        reduce_films()
        if rank == 0:
            ctx.film(out=film_pinned.numpy(), count_out=cnt_pinned.numpy().view(np.uint32))
        return 1e3 * (time.perf_counter() - t0)

    ctx.upload_rng(rng_host)
    for _ in range(warmup):
        step_resident()
    ctx.reset_stats()
    split_ms[0] = split_ms[1] = 0.0
    if clock_sampler is not None and rank == 0:
        clock_sampler.start()
    # ---- timed: K steps, device time (CUDA events on the context stream inside the C ABI), max over ranks
    job.barrier()
    wall0 = time.perf_counter()
    dev_ms = 0.0
    for _ in range(steps):
        dev_ms += step_resident()
    job.barrier()
    wall_ms = 1e3 * (time.perf_counter() - wall0)
    if dump_dir is not None and rank == 0:
        xyz, cnt = ctx.film()
        dump_outputs(dump_dir, {"film_xyz": xyz, "sample_count": cnt.astype(np.float32)})
    dev_ms = job.max_over_ranks(dev_ms)
    rank_ms = None
    if world > 1:
        rank_ms = [{"render": x[0] / steps, "film_reduce": x[1] / steps} for x in job.gather_rows(split_ms)]
    st = ctx.stats()
    launches = int(st.kernel_launches)
    rays_all = job.sum_over_ranks(float(st.ray_count))
    # ---- e2e leg: host buffers through the C ABI
    e2e_ms = None
    if want_e2e:
        step_e2e()
        job.barrier()
        e2e_ms = 0.0
        for _ in range(steps):
            e2e_ms += step_e2e()
        job.barrier()
        e2e_ms = job.max_over_ranks(e2e_ms)
    if clock_sampler is not None and rank == 0:
        clock_sampler.stop()
    # ---- per-stage profile pass (rank 0): event pair around every kernel launch of one more render
    roofline = stage = None
    if want_profile and rank == 0 and tiles:
        ctx.upload_rng(rng_host)
        ctx.set_profiling(True)
        ctx.reset_stats()
        ctx.render_tiles(tiles, first_iter, min(spp, 64))
        stage = ctx.stage_times()
        pst = ctx.stats()
        ctx.set_profiling(False)
        total = sum(v[0] for v in stage.values()) or 1.0
        dom = max(stage, key=lambda k: stage[k][0])
        n_tris = int(scene.desc.contents.n_bvh_tris)
        b_closest, b_any = bvh_depth_bytes(n_tris)
        # algorithmic bytes per launch (DESIGN.md "Rooflines"): trace = B_ray per closest-hit ray + B_any per any-hit ray (SURVEY
        # 8(d)); shade = wavefront state read + written per path vertex (ray 2x32, hit 20, path state 5x16 r+w, RNG 16,
        # film/accumulator 32, shadow ray out 48)
        n_closest = int(pst.primary_ray_count + pst.bounce_ray_count)
        n_any = int(pst.shadow_ray_count)
        units = {"trace": n_closest + n_any, "shade": n_closest}
        bytes_total = {"trace": n_closest * b_closest + n_any * b_any, "shade": n_closest * (64 + 20 + 160 + 16 + 32 + 48)}
        ms_dom, n_dom = stage[dom]
        peak, peak_src = measured_peak_gbs()
        achieved = bytes_total[dom] / (ms_dom * 1e-3) / 1e9 if ms_dom > 0 else 0.0
        roofline = {"bound": "hbm", "kernel": "k_" + dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": ncu_traffic(key, "k_" + dom), "peak_source": peak_src, "avg_launch_us": 1e3 * ms_dom / max(n_dom, 1), "launches": n_dom,
                    "bytes_per_unit": bytes_total[dom] / max(units[dom], 1), "units_per_launch": units[dom] / max(n_dom, 1),
                    "slots": npix_rank, "stage_share": {k: v[0] / total for k, v in stage.items()},
                    "note": "scene is L2-resident (%d triangles): HBM is not the binding resource, see DESIGN.md" % n_tris}
    # ---- cpu baseline (rank 0, N=1 only): the oracle port on all host cores, bounded sample
    cpu = None
    if rank == 0 and world == 1 and cpu_seconds > 0:
        from oracle_binding import OracleScene
        ora = OracleScene(scene)
        cores = os.cpu_count() or 1
        t0 = time.perf_counter()
        ora.render(all_tiles, 0, 1, rng=rng_host, threads=cores, aov=False)
        t1 = time.perf_counter() - t0
        n = max(1, min(spp, int(round(cpu_seconds / max(t1, 1e-3)))))
        t0 = time.perf_counter()
        ora.render(all_tiles, 0, n, rng=rng_host, threads=cores, aov=False)
        dt = time.perf_counter() - t0
        cpu = {"value": W * H * n / dt, "unit": "samples/s", "cores": cores, "kind": "port",
               "sample": "%d of %d spp over the full %dx%d film (rate-normalised), oracle (scalar C++17 restatement, own BVH, std::thread x %d; not Embree)" % (n, spp, W, H, cores)}
    out = None
    if rank == 0:
        total_samples = npix_rank * spp * world * steps if scaling == "weak" else W * H * spp * steps
        out = {"value": total_samples / (dev_ms * 1e-3), "unit": "samples/s", "ms_per_step": dev_ms / steps, "wall_ms_per_step": wall_ms / steps, "scaling": scaling,
               "mrays_per_s": rays_all / (dev_ms * 1e-3) / 1e6,
               "config": {"workload": label, "scene": fname, "spp_per_step": spp, "spp_of_scene": int(scene.settings.max_sample_count) // (world if partition == "samples" else 1),
                          "film": [W, H], "partition": partition, "paths_in_flight_per_gpu": npix_rank,
                          "l2": "wavefront state (%d paths x ~250 B) and film are re-written every wavefront iteration; scene is L2-resident by nature" % npix_rank},
               "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu, "stage_ms": {k: v[0] for k, v in stage.items()} if stage else None,
               "rank_ms_per_step": rank_ms,
               "shading": {0: "single k_shade", 1: "staged (k_shade_geom + nee/scatter per material type)", -1: "undecided"}[ctx.shading_mode()]}
        if e2e_ms is not None:
            out["e2e"] = {"value": total_samples / (e2e_ms * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": W * H * 8 + len(tiles) * 16,
                          "d2h_bytes_per_step": W * H * 3 * 4 + W * H * 4, "ms_per_step": e2e_ms / steps}
    ctx.close()
    return out


def verify_tile_partition(job, prb, key, iters):
    """outside every timed region: the film reduced over job.world GPUs in tile mode must be bit-identical to a 1-GPU render"""
    import numpy as np
    from pearray_b200 import multigpu
    scene, _, _ = load_scene(prb, key)
    tiles = scene.tiles(8, 8)
    ctx = prb.Context(job.local_rank)
    ctx.upload_scene(scene)
    job.join_communicator(ctx)
    ctx.upload_rng(scene.rng_map())
    mine = multigpu.partition_tiles(scene.tiles(32, 32), job.rank, job.world)
    if mine:
        ctx.render_tiles(mine, 0, iters)
    ctx.film_reduce_comm("tiles", iters, 0)
    ok = None
    if job.rank == 0:
        xyz, cnt = ctx.film()
        single = prb.Context(job.local_rank)
        single.upload_scene(scene)
        single.upload_rng(scene.rng_map())
        single.render_tiles(tiles, 0, iters)
        sx, sc = single.film()
        ok = bool(np.array_equal(xyz.view(np.uint32), sx.view(np.uint32)) and np.array_equal(cnt, sc))
        single.close()
    ctx.close()
    job.barrier()
    return ok


# ----------------------------------------------------------------------------------------------- C5: triangle soup
def soup_workload(job, prb, args, steps, passes, want_cpu, clock_sampler=None, dump_dir=None):
    """SURVEY 8(d) C5: synthetic N-triangle soup (default 10 M), 2048x2048 pinhole, jittered passes; three ray classes timed
    separately through prb_trace_closest_device / prb_trace_any_device with the ray streams resident in HBM: primary (coherent
    closest hit), shadow (any hit towards a point light at (0,3,0), tfar = dist - 1e-3) and incoherent (cosine-hemisphere bounce
    from every primary hit, closest hit).  The only configuration that streams the BVH from HBM.  Weak scaling over ranks (every
    rank traces its own passes against the replicated scene).  dump_dir: write a fixed, seeded sample of the hit buffers of
    every ray class of rank 0's last timed pass there."""
    import numpy as np
    torch = job.torch
    rank, world, dev = job.rank, job.world, job.dev
    res = args.soup_film
    t0 = time.perf_counter()
    scene = prb.Scene.soup(args.triangles, seed=1234, film=(res, res))
    build_s = time.perf_counter() - t0
    d = scene.desc.contents
    ctx = prb.Context(job.local_rank)
    ctx.upload_scene(scene)
    ctx.upload_rng(scene.rng_map())
    verts = torch.from_numpy(np.ctypeslib.as_array(d.vertices, shape=(d.n_vertices, 3)).copy()).to(dev).view(-1, 3, 3)
    n = res * res
    f32 = dict(dtype=torch.float32, device=dev)
    ent = torch.empty(n, dtype=torch.int32, device=dev); prim = torch.empty_like(ent)
    u = torch.empty(n, **f32); v = torch.empty(n, **f32); t = torch.empty(n, **f32)
    occ = torch.empty(n, dtype=torch.uint8, device=dev)
    light = torch.tensor([0.0, 3.0, 0.0], **f32)

    def soa(x):  # (n,3) -> three contiguous columns
        return [x[:, i].contiguous() for i in range(3)]

    def ptrs(o, dd, tmin=None, tmax=None):
        return [c.data_ptr() for c in o] + [c.data_ptr() for c in dd] + [tmin.data_ptr() if tmin is not None else None, tmax.data_ptr() if tmax is not None else None]

    hitp = [ent.data_ptr(), prim.data_ptr(), u.data_ptr(), v.data_ptr(), t.data_ptr()]
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    ms = {"primary": 0.0, "shadow": 0.0, "incoherent": 0.0}
    rays = {"primary": 0, "shadow": 0, "incoherent": 0}
    hits = {"primary": 0, "shadow": 0, "incoherent": 0}
    keep = {}
    dumped = {}

    def dump_hits(cls, count, seed):
        """a fixed, seeded sample of the rays of one class: the hit columns (ids as float64) or the occlusion flags"""
        sel = np.sort(np.random.default_rng(seed).choice(count, min(count, DUMP_SAMPLE_RAYS), replace=False))
        idx = torch.from_numpy(sel).to(dev)
        if cls == "shadow":
            dumped["shadow_occluded"] = occ[idx].cpu().numpy().astype(np.float32)
            return
        for name, col in (("entity_id", ent), ("primitive_id", prim)):
            dumped["%s_%s" % (cls, name)] = col[idx].cpu().numpy().view(np.uint32).astype(np.float64)
        for name, col in (("u", u), ("v", v), ("t", t)):
            dumped["%s_%s" % (cls, name)] = col[idx].cpu().numpy()

    def one_pass(p, timed, capture=False):
        org, dr, _, _ = ctx.generate_camera_rays([(0, 0, res, res)], p)
        o = soa(torch.from_numpy(org).to(dev)); dd = soa(torch.from_numpy(dr).to(dev))
        torch.cuda.synchronize(dev)
        ctx.trace_closest_device(ptrs(o, dd), n, hitp)
        if timed:
            ms["primary"] += ctx.last_device_ms(); rays["primary"] += n
        if capture:  # the incoherent trace below reuses these hit buffers
            dump_hits("primary", n, 1)
        hit = ent != -1
        idx = hit.nonzero().squeeze(1)
        m = int(idx.numel())
        if timed:
            hits["primary"] += m
        O = torch.stack(o, 1)[idx]; D = torch.stack(dd, 1)[idx]
        P = O + D * t[idx, None]
        tri = verts[prim[idx].long()]
        N = torch.linalg.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
        N = N / N.norm(dim=1, keepdim=True).clamp_min(1e-30)
        N = torch.where((N * D).sum(1, keepdim=True) > 0, -N, N)  # face the incoming ray
        # shadow rays (Scene::traceShadowRay semantics: tnear 1e-4, tfar = distance - 1e-3)
        L = light - P
        dist_l = L.norm(dim=1)
        L = L / dist_l[:, None]
        so = soa(P); sd = soa(L)
        tmin = torch.full((m,), 1e-4, **f32); tmax = (dist_l - 1e-3).contiguous()
        torch.cuda.synchronize(dev)
        ctx.trace_any_device(ptrs(so, sd, tmin, tmax), m, occ.data_ptr())
        if timed:
            ms["shadow"] += ctx.last_device_ms(); rays["shadow"] += m; hits["shadow"] += int(occ[:m].sum())
        # incoherent: cosine-hemisphere bounce around N
        r1 = torch.rand(m, generator=gen, **f32); r2 = torch.rand(m, generator=gen, **f32)
        ct = r1.sqrt(); st_ = (1 - r1).clamp_min(0).sqrt(); ph = 2 * np.pi * r2
        a = torch.where(N[:, 0:1].abs() > 0.9, torch.tensor([0.0, 1.0, 0.0], **f32), torch.tensor([1.0, 0.0, 0.0], **f32)).expand(m, 3)
        T = torch.linalg.cross(N, a); T = T / T.norm(dim=1, keepdim=True); B = torch.linalg.cross(N, T)
        Wd = T * (st_ * ph.cos())[:, None] + B * (st_ * ph.sin())[:, None] + N * ct[:, None]
        bo = soa(P); bd = soa(Wd)
        torch.cuda.synchronize(dev)
        ctx.trace_closest_device(ptrs(bo, bd, tmin, None), m, hitp)
        if timed:
            ms["incoherent"] += ctx.last_device_ms(); rays["incoherent"] += m; hits["incoherent"] += int((ent[:m] != -1).sum())
        if capture:
            dump_hits("shadow", m, 2)
            dump_hits("incoherent", m, 3)
        if not keep:  # one sample of every class, with the device results, for the oracle cross-check and the e2e / cpu legs
            # a contiguous block of the pass, in ray order: the host-buffer leg traces rays as coherent as the resident leg does (a random
            # subset would time the traversal of shuffled rays, 2-3x slower, instead of the copies around it)
            sel = torch.arange(min(m, 1 << 20), device=dev) + max(0, (m - (1 << 20)) // 2)
            keep.update(org=org[:1 << 20].copy(), dr=dr[:1 << 20].copy(), P=P[sel].cpu().numpy(), L=L[sel].cpu().numpy(), tmax=tmax[sel].cpu().numpy(),
                        W=Wd[sel].cpu().numpy(), occ=occ[:m][sel].cpu().numpy(), ent2=ent[:m][sel].cpu().numpy().view(np.uint32),
                        prim2=prim[:m][sel].cpu().numpy().view(np.uint32), t2=t[:m][sel].cpu().numpy())

    for w in range(max(args.warmup, 1)):
        one_pass(1000 + w, False)
    keep.clear()
    ctx.reset_stats()
    if clock_sampler is not None and rank == 0:
        clock_sampler.start()
    job.barrier()
    wall0 = time.perf_counter()
    for s in range(steps):
        for p in range(passes):
            one_pass(rank * passes + p, True, capture=dump_dir is not None and rank == 0 and s == steps - 1 and p == passes - 1)
    torch.cuda.synchronize(dev)
    wall = time.perf_counter() - wall0
    if dumped:
        dump_outputs(dump_dir, dumped)
    if clock_sampler is not None and rank == 0:
        clock_sampler.stop()
    tot_ms_max = job.max_over_ranks(sum(ms.values()))
    all_rays = job.sum_over_ranks(float(sum(rays.values())))
    out = None
    if rank == 0:
        n_tris = int(d.n_bvh_tris)
        b_closest, b_any = bvh_depth_bytes(n_tris)
        peak, peak_src = measured_peak_gbs()
        per_class = {}
        for k in ms:
            bpr = b_any if k == "shadow" else b_closest
            per_class[k] = {"mrays_per_s": rays[k] / (ms[k] * 1e-3) / 1e6, "hit_fraction": hits[k] / max(rays[k], 1), "ms": ms[k],
                            "achieved_gbs": rays[k] * bpr / (ms[k] * 1e-3) / 1e9, "frac": rays[k] * bpr / (ms[k] * 1e-3) / 1e9 / peak, "bytes_per_ray": bpr}
        dom = max(ms, key=lambda k: ms[k])
        launches = steps * passes
        roofline = {"bound": "hbm", "kernel": "k_trace_any" if dom == "shadow" else "k_trace_closest (%s rays)" % dom, "achieved": per_class[dom]["achieved_gbs"],
                    "peak": peak, "unit": "GB/s", "frac": per_class[dom]["frac"], "traffic": ncu_traffic("c5", "k_trace_any" if dom == "shadow" else "k_trace_closest"),
                    "peak_source": peak_src, "avg_launch_us": 1e3 * ms[dom] / launches, "launches": launches, "bytes_per_unit": per_class[dom]["bytes_per_ray"],
                    "units_per_launch": rays[dom] / launches}
        # ---- e2e: HOST ray buffers in, hit buffers out through prb_trace_closest / prb_trace_any (copies inside the timed region)
        k = keep
        ne = len(k["org"])
        npl = len(k["P"])

        def pinned(a):  # a page-locked copy of a host array (the ray / hit columns a caller of the C ABI would own)
            t_ = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
            return t_.numpy()

        def cols(o, d_, tmin_, tmax_):
            return [pinned(o[:, i]) for i in range(3)] + [pinned(d_[:, i]) for i in range(3)] + [None if tmin_ is None else pinned(tmin_), None if tmax_ is None else pinned(tmax_)]

        def hit_cols(m_):
            return [pinned(np.empty(m_, np.uint32)), pinned(np.empty(m_, np.uint32)), pinned(np.empty(m_, np.float32)), pinned(np.empty(m_, np.float32)), pinned(np.empty(m_, np.float32))]

        tmin_h = np.full(npl, 1e-4, np.float32)
        rays1, rays2, rays3 = cols(k["org"], k["dr"], None, None), cols(k["P"], k["L"], tmin_h, k["tmax"]), cols(k["P"], k["W"], tmin_h, None)
        got1, got2, got_occ = hit_cols(ne), hit_cols(npl), pinned(np.empty(npl, np.uint8))
        ctx.trace_closest_soa(rays1, ne, got1)  # warm the scratch buffers
        t0 = time.perf_counter()
        reps = 4
        for _ in range(reps):
            ctx.trace_closest_soa(rays1, ne, got1)
            ctx.trace_any_soa(rays2, npl, got_occ)
            ctx.trace_closest_soa(rays3, npl, got2)
        e2e_dt = time.perf_counter() - t0
        e2e_rays = reps * (ne + 2 * npl)
        e2e = {"value": e2e_rays / e2e_dt, "unit": "rays/s", "h2d_bytes_per_step": (ne * 24 + npl * (32 + 28)), "d2h_bytes_per_step": ne * 20 + npl * 21,
               "sample": "%d primary + %d shadow + %d incoherent rays per step in page-locked host columns (copied in and out by prb_trace_*)" % (ne, npl, npl)}
        # the HBM-resident timed launches returned the same answers as the host-buffer calls
        consistent = bool(np.array_equal(got_occ, k["occ"]) and np.array_equal(got2[0], k["ent2"]) and np.array_equal(got2[1], k["prim2"]))
        cpu = parity = None
        if want_cpu:
            from oracle_binding import OracleScene
            t0 = time.perf_counter()
            ora = OracleScene(scene)
            accel_s = time.perf_counter() - t0
            cores = os.cpu_count() or 1
            nc = 65536  # bounded CPU sample: 64 k rays of every class, spread evenly over the host-buffer sample
            p1 = np.linspace(0, ne - 1, min(nc, ne)).astype(np.int64)
            p2 = np.linspace(0, npl - 1, min(nc, npl)).astype(np.int64)
            t0 = time.perf_counter()
            ref1 = ora.trace_closest(k["org"][p1], k["dr"][p1], threads=cores)
            ref_occ = ora.trace_any(k["P"][p2], k["L"][p2], tmin_h[p2], k["tmax"][p2], threads=cores)
            ref2 = ora.trace_closest(k["P"][p2], k["W"][p2], tmin_h[p2], threads=cores)
            dt = time.perf_counter() - t0
            nc, n2 = len(p1), len(p2)
            cpu = {"value": (nc + 2 * n2) / dt, "unit": "rays/s", "cores": cores, "kind": "port",
                   "sample": "%d primary + %d shadow + %d incoherent rays, oracle BVH (median split, scalar), std::thread x %d; accel build %.1f s" % (nc, n2, n2, cores, accel_s)}
            h1 = ref1[0] != 0xFFFFFFFF
            parity = {"rays_checked": int(nc + 2 * n2),
                      "primary_id_mismatches": int((got1[0][p1] != ref1[0]).sum() + (got1[1][p1] != ref1[1]).sum()),
                      "primary_t_mismatches": int((got1[4][p1][h1].view(np.uint32) != ref1[4][h1].view(np.uint32)).sum()),
                      "shadow_mismatches": int((got_occ[p2] != ref_occ).sum()),
                      "incoherent_id_mismatches": int((got2[0][p2] != ref2[0]).sum() + (got2[1][p2] != ref2[1]).sum())}
        out = {"metric": "rays/s (primary+shadow+incoherent)", "value": all_rays / (tot_ms_max * 1e-3), "unit": "rays/s", "ms_per_step": tot_ms_max / steps,
               "scaling": "weak", "n_gpus": world,
               "config": {"workload": "synthetic %d-triangle soup, %dx%d pinhole, %d passes/step, primary+shadow+1-bounce incoherent" % (n_tris, res, res, passes),
                          "bvh_nodes": int(d.n_bvh_nodes), "bvh_mbytes": (int(d.n_bvh_nodes) * 80 + n_tris * 48) / 1e6, "host_build_s": build_s,
                          "l2": "BVH + triangles (%.0f MB) exceed the 126 MB L2 for >= 2.4 M triangles" % ((int(d.n_bvh_nodes) * 80 + n_tris * 48) / 1e6)},
               "classes": per_class, "roofline": roofline, "gpu_launches": int(ctx.stats().kernel_launches), "e2e": e2e, "cpu_baseline": cpu,
               "parity_vs_oracle": parity, "resident_equals_host_path": consistent, "wall_s": wall}
    ctx.close()
    return out


# ----------------------------------------------------------------------------------------------- our arm
def run_ours(args, rank, world, local_rank):
    import torch
    import pearray_b200 as prb
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU fallback (use --impl reference for the CPU arm)")
    job = Job(rank, world, local_rank)
    sampler = ClockSampler(local_rank)
    line = None
    if args.scene == "c5":
        r = soup_workload(job, prb, args, args.steps, args.passes, want_cpu=(world == 1 and not args.no_cpu), clock_sampler=sampler, dump_dir=args.dump_outputs)
        if rank == 0:
            line = {"metric": r["metric"], "value": r["value"], "unit": r["unit"], "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
                    "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": r["config"], "classes": r["classes"],
                    "roofline": r["roofline"], "gpu_launches": r["gpu_launches"], "clocks": sampler.summary(), "e2e": r["e2e"], "cpu_baseline": r["cpu_baseline"],
                    "parity_vs_oracle": r["parity_vs_oracle"], "resident_equals_host_path": r["resident_equals_host_path"], "embree": embree_probe()}
    else:
        key = args.scene
        scene_spp = {"c1": 64, "c2": 1024, "c3": 128, "c4": 256, "c4b": 4096, "c4c": 4096, "c0": 128}[key]
        spp = scene_spp if args.spp is None else args.spp
        r = render_workload(job, prb, key, spp, args.steps, args.warmup, args.partition, cpu_seconds=0.0 if args.no_cpu else 12.0, clock_sampler=sampler,
                            dump_dir=args.dump_outputs)
        extras = {}
        if not args.no_extras and key == "c2" and args.spp is None:
            if world == 1:
                # the two other workloads BASELINE.json names, bounded so that the default run stays within a few minutes
                c = render_workload(job, prb, "c4c", 64, 2, 1, "single", cpu_seconds=0.0 if args.no_cpu else 8.0)
                extras["workloads"] = {"complex": c}
                s = soup_workload(job, prb, args, 1, 4, want_cpu=not args.no_cpu)
                extras["workloads"]["c5"] = s
            else:
                # strong scaling on the north star's target: complex.prc by interleaved tiles, fixed total work
                ss = render_workload(job, prb, "c4c", 64, 2, 1, "tiles", want_e2e=True, want_profile=False)
                ok = verify_tile_partition(job, prb, "c4c", 2)
                # the same fixed total work split by SAMPLE RANGES: every GPU keeps the whole film in flight (full occupancy) and
                # renders 64 / N iterations of one 64-sample sequence; statistically equivalent to the 1-GPU image, not bit-identical
                sr = render_workload(job, prb, "c4c", max(1, 64 // world), 2, 1, "samples", want_e2e=False, want_profile=False)
                if rank == 0:
                    ss["tile_film_bit_identical_to_1gpu"] = ok
                    ss["note"] = "fixed total work: 64 spp of the 1920x1080 film per step over %d GPUs (interleaved tiles of a 32x32 tile map), one prb_film_reduce_comm per step" % world
                    sr["scaling"] = "strong"
                    sr["note"] = "fixed total work: %d x %d = 64 spp of the 1920x1080 film per step, sample-range partition" % (world, max(1, 64 // world))
                    extras["strong_scaling"] = {"by_tiles": ss, "by_sample_ranges": sr}
                s = soup_workload(job, prb, args, 1, 4, want_cpu=False)
                if rank == 0:
                    extras["workloads"] = {"c5": s}
        if rank == 0:
            line = {"metric": "spectral path samples/s", "value": r["value"], "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                    "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": r["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                    "mrays_per_s": r["mrays_per_s"], "wall_ms_per_step": r["wall_ms_per_step"], "config": r["config"], "e2e": r.get("e2e"),
                    "gpu_launches": r["gpu_launches"], "clocks": sampler.summary(), "roofline": r["roofline"], "cpu_baseline": r["cpu_baseline"],
                    "stage_ms": r["stage_ms"], "rank_ms_per_step": r["rank_ms_per_step"], "embree": embree_probe()}
            line.update(extras)
    if rank == 0:
        emit(line)
    job.finish()


_JSON_FD = None


def emit(line):
    """the ONE JSON line goes to the real stdout; everything else (NCCL banners, library chatter) was moved to stderr"""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)  # NCCL prints its version banner on fd 1: keep stdout for the JSON line only
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scene", default="c2", choices=sorted(SCENES) + ["c5"])
    ap.add_argument("--triangles", type=int, default=10000000, help="c5: soup size")
    ap.add_argument("--soup-film", type=int, default=2048, help="c5: film resolution (square)")
    ap.add_argument("--passes", type=int, default=16, help="c5: jittered passes per step")
    ap.add_argument("--spp", type=int, default=None, help="iterations per step (default: the scene's sample count)")
    ap.add_argument("--partition", default="samples", choices=["samples", "tiles"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--no-extras", action="store_true", help="default run: skip the complex.prc / C5 / strong-scaling legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the headline workload returned in its last step as DIR/<name>.npy "
                         "(film + sample counts; c5: a fixed sample of the hit buffers)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    import __graft_entry__ as g
    if rank == 0 and not os.path.exists(os.path.join(ROOT, "pearray_b200", "libprb200.so")):
        g.build()
    if args.impl == "reference":
        if args.scene == "c5":
            run_reference_soup(args, rank)
        else:
            run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


def run_reference_soup(args, rank):
    """CPU arm of C5: the oracle's own BVH traced on all host cores over a bounded sample of the same three ray classes"""
    if rank != 0:
        return
    import numpy as np
    import pearray_b200 as prb
    from oracle_binding import OracleScene
    res = args.soup_film
    scene = prb.Scene.soup(args.triangles, seed=1234, film=(res, res))
    ora = OracleScene(scene)
    cores = os.cpu_count() or 1
    n = 262144
    rs = np.random.RandomState(3)
    # pinhole at (0,0,-3) looking +z, fov 40 degrees, jittered pixel positions
    px = rs.rand(n, 2).astype(np.float32) * 2 - 1
    half = np.float32(np.tan(np.radians(20.0)))
    dr = np.stack([px[:, 0] * half, px[:, 1] * half, np.ones(n, np.float32)], 1).astype(np.float32)
    dr /= np.linalg.norm(dr, axis=1, keepdims=True)
    org = np.tile(np.array([0, 0, -3], np.float32), (n, 1))
    ora.trace_closest(org[:4096], dr[:4096], threads=cores)
    t0 = time.perf_counter()
    rays = 0
    for _ in range(args.steps):
        ent, prim, u, v, t = ora.trace_closest(org, dr, threads=cores)
        hit = ent != 0xFFFFFFFF
        P = (org[hit] + dr[hit] * t[hit, None]).astype(np.float32)
        L = np.array([0, 3, 0], np.float32) - P
        dist = np.linalg.norm(L, axis=1).astype(np.float32)
        L = (L / dist[:, None]).astype(np.float32)
        tmin = np.full(len(P), 1e-4, np.float32)
        ora.trace_any(P, L, tmin, (dist - 1e-3).astype(np.float32), threads=cores)
        b = rs.normal(size=P.shape).astype(np.float32)
        b /= np.linalg.norm(b, axis=1, keepdims=True)
        ora.trace_closest(P, b, tmin, threads=cores)
        rays += n + 2 * len(P)
    dt = time.perf_counter() - t0
    value = rays / dt
    emit({"impl": "reference", "metric": "rays/s (primary+shadow+incoherent)", "value": value, "unit": "rays/s", "n_gpus": args.gpus, "steps": args.steps,
          "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
          "data": "synthetic", "config": {"workload": "synthetic %d-triangle soup, %d primary rays per step + their shadow and bounce rays" % (args.triangles, n)},
          "cpu_baseline": {"value": value, "unit": "rays/s", "cores": cores, "kind": "port", "sample": "%d primary rays per step, oracle BVH (scalar, median split), std::thread x %d" % (n, cores)},
          "embree": embree_probe(), "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


if __name__ == "__main__":
    main()
