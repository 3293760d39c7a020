"""bench.py contract checks: the reference arm (the CPU oracle timed on the host cores) prints one JSON line with the keys
the driver reads, and the product arm refuses to run without a CUDA device instead of falling back.  On a GPU,
--dump-outputs writes what the timed path returned in its last step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, env=e, capture_output=True, text=True, timeout=600)


def test_reference_arm_prints_the_contract_line():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--spp", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    assert d["metric"] == "spectral path samples/s" and d["unit"] == "samples/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert d["config"]["workload"].startswith("cornellbox.prc")
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    e2e = d["e2e"]
    assert e2e["value"] == d["value"] and e2e["unit"] == d["unit"]
    assert e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    assert d["vs_baseline"] is None  # BASELINE.json publishes no number for this metric


def test_reference_arm_other_ranks_exit_without_work():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"], env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0, r.stderr[-2000:]
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_product_arm_has_no_cpu_fallback():
    r = _run(["--steps", "1", "--warmup", "3"])
    assert r.returncode != 0
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert "no CUDA device" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_hold_the_film_of_the_last_timed_render(tmp_path):
    r = _run(["--scene", "c1", "--spp", "2", "--steps", "1", "--warmup", "0", "--no-cpu", "--dump-outputs", str(tmp_path)])
    assert r.returncode == 0, r.stderr[-2000:]
    assert sorted(p.name for p in tmp_path.iterdir()) == ["film_xyz.npy", "sample_count.npy"]
    xyz, cnt = np.load(tmp_path / "film_xyz.npy"), np.load(tmp_path / "sample_count.npy")
    assert xyz.dtype == np.float32 and cnt.dtype == np.float32
    # the one timed step renders the scene's first two iterations from its seeded RNG map: a plain render gives the same film
    import pearray_b200 as prb
    ctx, ref, ref_cnt = prb.render(prb.Scene.from_file(os.path.join(ROOT, "scenes", "c1_sphere.prc")), spp=2)
    ctx.close()
    assert np.array_equal(xyz.view(np.uint32), ref.view(np.uint32))
    assert np.array_equal(cnt, ref_cnt.astype(np.float32))


@pytest.mark.gpu
def test_dump_outputs_hold_the_hits_of_the_last_timed_pass(tmp_path):
    res, tris = 128, 200000
    r = _run(["--scene", "c5", "--triangles", str(tris), "--soup-film", str(res), "--passes", "2", "--steps", "2", "--warmup", "1", "--no-cpu",
              "--dump-outputs", str(tmp_path)])
    assert r.returncode == 0, r.stderr[-2000:]
    cols = ["entity_id", "primitive_id", "u", "v", "t"]
    want = sorted(["shadow_occluded.npy"] + ["%s_%s.npy" % (c, n) for c in ("primary", "incoherent") for n in cols])
    assert sorted(p.name for p in tmp_path.iterdir()) == want
    d = {p.name[:-4]: np.load(p) for p in tmp_path.iterdir()}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    # fewer rays than the sample size: every primary ray of the last pass (pass 1 of rank 0), in ray order
    import pearray_b200 as prb
    scene = prb.Scene.soup(tris, seed=1234, film=(res, res))
    ctx = prb.Context(0)
    ctx.upload_scene(scene)
    ctx.upload_rng(scene.rng_map())
    org, dr, _, _ = ctx.generate_camera_rays([(0, 0, res, res)], 1)
    ent, prim, u, v, t = ctx.trace_closest(org, dr)
    ctx.close()
    assert np.array_equal(d["primary_entity_id"], ent.astype(np.float64)) and np.array_equal(d["primary_primitive_id"], prim.astype(np.float64))
    hit = ent != prb.INVALID_ID
    for name, a in (("u", u), ("v", v), ("t", t)):
        assert np.array_equal(d["primary_" + name][hit].view(np.uint32), a[hit].view(np.uint32))
    assert len(d["shadow_occluded"]) == len(d["incoherent_t"]) == int(hit.sum())
