"""The ambient-occlusion integrator ('ao'): loader and C ABI on the CPU, known answers on the oracle (oracle_ao/) and on the
device, and the device bit-exact against the oracle (`-m gpu`).

Known answers hold for any correct cosine-weighted AO; the renders use a monotonic film (`:spectral_domain 520`), where a pixel's
value is the mean of its samples' 1 - occluded / N."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import pearray_b200 as prb
from conftest import ROOT, scene_path
from oracle_binding import OracleScene, _p
from test_golden_oracle import STAT_NAMES

_ao_lib = None


def ao_lib():
    global _ao_lib
    if _ao_lib is None:
        path = os.path.join(ROOT, "oracle_ao", "libao_oracle.so")
        if not os.path.exists(path):
            subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle_ao"), "-s"])
        lib = C.CDLL(path)
        lib.orc_scene_create.restype = C.c_void_p
        lib.orc_scene_create.argtypes = [C.POINTER(prb.SceneDesc)]
        lib.orc_scene_destroy.argtypes = [C.c_void_p]
        lib.orc_render_ao.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(prb.Tile), C.c_size_t, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]
        _ao_lib = lib
    return _ao_lib


def oracle_ao(scene, tiles, first, count, sample_count, rng=None, film=None, cnt=None, aov=None, aove=None, feedback=None, variance=None):
    """renders iterations [first, first + count) with the 'ao' oracle; the film buffers continue when given"""
    w, h = scene.width, scene.height
    rng = scene.rng_map() if rng is None else np.array(rng, dtype=np.uint64, copy=True)
    film = np.zeros((h, w, 3), np.float32) if film is None else film
    cnt = np.zeros((h, w), np.uint32) if cnt is None else cnt
    aov = np.zeros((h, w, 10), np.float32) if aov is None else aov
    aove = np.zeros((h, w, 11), np.float32) if aove is None else aove
    feedback = np.zeros((h, w), np.uint32) if feedback is None else feedback
    stats = np.zeros(11, np.uint64)
    vm, vv = variance if variance is not None else (None, None)
    lib = ao_lib()
    hdl = lib.orc_scene_create(scene.desc)
    try:
        lib.orc_render_ao(hdl, _p(rng), prb.make_tiles(tiles), len(tiles), first, count, _p(film), _p(cnt), _p(aov), _p(stats), os.cpu_count() or 1,
                          _p(feedback), None if vm is None else _p(vm), None if vv is None else _p(vv), None, _p(aove), sample_count)
    finally:
        lib.orc_scene_destroy(hdl)
    return dict(film=film, count=cnt, aov=aov, aov_ext=aove, feedback=feedback, rng=rng, online_mean=vm, online_variance=vv,
                stats=dict(zip(STAT_NAMES, (int(x) for x in stats))))


def scene_with_integrator(path, block, extra=""):
    """a scene file with its (integrator ...) block replaced (and `extra` appended inside the scene)"""
    src = open(path).read()
    i = src.index("(integrator")
    depth, j = 0, i
    while True:
        depth += {"(": 1, ")": -1}.get(src[j], 0)
        j += 1
        if depth == 0:
            break
    src = src[:i] + block + src[j:]
    k = src.rindex(")")
    return prb.Scene.from_string(src[:k] + extra + src[k:], path)


# a lone floor (plane, normal +z) seen from above; the pixels of the border miss it
LONE_FLOOR = """
(scene :name 'ao_floor' :render_width 32 :render_height 32 :camera 'Camera' :spectral_domain 520
 (integrator :type 'ao' :sample_count %(n)d)
 (sampler :slot 'aa' :type 'random' :sample_count 4)
 (filter :slot 'pixel' :type 'block' :radius 0)
 (camera :name 'Camera' :type 'orthographic' :width 4 :height 4 :local_direction [0,0,-1] :local_up [0,1,0] :local_right [1,0,0]
   :position [0,0,2])
 (material :name 'm' :type 'diffuse' :albedo 0.8)
 (entity :name 'floor' :type 'plane' :centering true :width 2 :height 2 :material 'm' :position [0,0,0])
)
"""

# a floor under a downward-facing square ceiling of half-size a at height h; an orthographic camera of tiny extent between the
# two looks down at the floor below the ceiling's centre
CEILING = """
(scene :name 'ao_ceiling' :render_width %(res)d :render_height %(res)d :camera 'Camera' :spectral_domain 520
 (integrator :type 'ao' :sample_count %(n)d)
 (sampler :slot 'aa' :type 'random' :sample_count %(spp)d)
 (filter :slot 'pixel' :type 'block' :radius 0)
 (camera :name 'Camera' :type 'orthographic' :width 0.001 :height 0.001 :local_direction [0,0,-1] :local_up [0,1,0]
   :local_right [1,0,0] :position [0,0,%(cam)g])
 (material :name 'm' :type 'diffuse' :albedo 0.8)
 (entity :name 'floor' :type 'plane' :centering true :width 8 :height 8 :material 'm' :position [0,0,0])
 (entity :name 'ceiling' :type 'plane' :centering true :width %(w)g :height %(w)g :material 'm'
   :transform [1,0,0,0, 0,-1,0,0, 0,0,-1,%(h)g, 0,0,0,1])
)
"""


def ceiling_scene(A=1.0, res=64, spp=16, n=16):
    h = 1.0
    return prb.Scene.from_string(CEILING % dict(res=res, spp=spp, n=n, w=2 * A * h, h=h, cam=0.5 * h))


def ceiling_expectation(A):
    """1 - 4 x the form factor of a differential area to the corner of a parallel A x A rectangle (unit height)"""
    s = A / math.sqrt(1 + A * A)
    return 1 - (4 / math.pi) * s * math.atan(s)


# ----------------------------------------------------------------------------- CPU: loader and ABI
def test_loader_yields_the_integrator_record():
    ao = prb.Scene.from_string(LONE_FLOOR % dict(n=7))
    rec = ao.integrator
    assert (rec.type, rec.sample_count) == (prb.INTEGRATOR["ao"], 7)
    default = prb.Scene.from_string((LONE_FLOOR % dict(n=7)).replace(":sample_count 7)", ")"))
    assert (default.integrator.type, default.integrator.sample_count) == (prb.INTEGRATOR["ao"], 10)
    direct = prb.Scene.from_file(scene_path("c2_cornellbox.prc"))
    assert direct.integrator.type == prb.INTEGRATOR["direct"]
    assert "ao" in {l.split(":")[0]: l.split(":")[1].split() for l in ao.plugins().strip().splitlines()}["integrator"]


def test_zero_sample_count_falls_back_to_one():
    assert prb.Scene.from_string(LONE_FLOOR % dict(n=0)).integrator.sample_count == 1


def test_integrator_mirror_and_null_arguments():
    host = prb.host_lib()
    assert host.prh_abi_sizeof(b"prb_integrator") == C.sizeof(prb.Integrator) == 8
    assert host.prh_scene_integrator(None, None) == -1  # PRB_ERR_INVALID_ARG
    dev = prb.device_lib()
    assert dev.prb_set_integrator(None, None) == -1
    assert dev.prb_get_integrator(None, None) == -1


# ----------------------------------------------------------------------------- CPU: known answers on the oracle
def test_oracle_lone_floor_is_unoccluded():
    scene = prb.Scene.from_string(LONE_FLOOR % dict(n=8))
    check_lone_floor(oracle_ao(scene, scene.full_tile(), 0, 1, 8), oracle_ao(scene, scene.full_tile(), 0, 4, 8), 8)


def check_lone_floor(one, four, n):
    """one sample: a pixel that hits is 1 and counts one sample, one that misses is 0 and counts none; four samples: the film is
    the fraction of samples that hit"""
    hit = one["count"] > 0
    assert hit.any() and (~hit).any() and one["count"].max() == 1
    assert np.abs(one["film"][hit] - 1.0).max() <= 1e-6 and np.all(one["film"][~hit] == 0)
    assert one["stats"]["shadow_ray_count"] == n * int(hit.sum()) and one["stats"]["background_hit_count"] == int((~hit).sum())
    assert np.abs(four["film"][..., 0] - four["count"] / np.float32(4)).max() <= 1e-6


def test_oracle_floor_under_square_ceiling_matches_form_factor():
    A, res, spp, n = 1.0, 64, 16, 16
    scene = ceiling_scene(A, res, spp, n)
    r = oracle_ao(scene, scene.full_tile(), 0, spp, n)
    assert np.all(r["count"] == spp)
    p = ceiling_expectation(A)
    sigma = math.sqrt(p * (1 - p) / (res * res * spp * n))
    assert abs(float(r["film"][..., 0].astype(np.float64).mean()) - p) < 5 * sigma


def test_oracle_one_sample_values_are_exact_fractions():
    n = 7
    scene = ceiling_scene(1.0, 32, 1, n)
    r = oracle_ao(scene, scene.full_tile(), 0, 1, n)
    allowed = {np.float32(1.0) - np.float32(k) / np.float32(n) for k in range(n + 1)}
    assert set(np.unique(r["film"][..., 0]).tolist()) <= {float(v) for v in allowed}


# ----------------------------------------------------------------------------- GPU
def device_render(scene, tiles, first, count, sample_count=None, ctx=None, rng=None):
    if ctx is None:
        ctx = prb.Context(0)
        ctx.upload_scene(scene)
        ctx.upload_rng(scene.rng_map() if rng is None else rng)
    if sample_count is not None:
        ctx.set_integrator("ao", sample_count)
    ctx.render_tiles(tiles, first, count)
    return ctx


def device_outputs(ctx, variance=False):
    xyz, cnt = ctx.film()
    out = dict(film=xyz, count=cnt, aov=ctx.film_aov(), feedback=ctx.film_feedback(), rng=ctx.download_rng(), stats=ctx.stats().as_dict())
    if ctx.scene.settings.want_aov_ext:
        out["aov_ext"] = ctx.film_aov_ext()
    if variance:
        out["online_mean"], out["online_variance"] = ctx.film_variance()
    return out


def assert_bit_exact(dev, ref):
    for k in ("film", "count", "aov", "feedback") + (("aov_ext",) if "aov_ext" in dev else ()) + (("online_mean", "online_variance") if "online_mean" in dev else ()):
        assert np.array_equal(dev[k].view(np.uint32), ref[k].view(np.uint32)), k
    assert np.array_equal(dev["rng"], ref["rng"]), "rng states"
    for n in STAT_NAMES:
        assert dev["stats"][n] == ref["stats"][n], n


# scene, tiles (crops: the oracle walks them on the CPU), iterations
GPU_CASES = {
    "c2": ("c2_cornellbox.prc", [(100, 100, 164, 164), (300, 250, 364, 314)], 4),
    "c1": ("c1_sphere.prc", [(468, 400, 532, 464), (200, 700, 264, 764)], 4),
    "c4": ("c4_boltsandgears.prc", [(400, 400, 464, 464), (600, 500, 664, 564)], 2),
    "c4c": ("c4c_complex.prc", [(900, 500, 964, 548)], 2),
}


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [None, "static", "persistent", "bvh"])
@pytest.mark.parametrize("n", [1, 7, 10, 33])
@pytest.mark.parametrize("name", list(GPU_CASES))
def test_gpu_ao_bit_exact_vs_oracle(name, n, mode, monkeypatch):
    if mode is not None:
        monkeypatch.setenv("PRB_TRACE_MODE", mode)
    else:
        monkeypatch.delenv("PRB_TRACE_MODE", raising=False)
    path, tiles, iters = GPU_CASES[name]
    scene = scene_with_integrator(scene_path(path), "(integrator :type 'ao' :sample_count %d)" % n)
    ctx = device_render(scene, tiles, 0, iters)  # upload_scene selects the scene's 'ao' record
    assert ctx.integrator == (prb.INTEGRATOR["ao"], n)
    dev = device_outputs(ctx)
    assert_bit_exact(dev, oracle_ao(scene, tiles, 0, iters, n))
    assert dev["stats"]["shadow_ray_count"] == n * int(dev["count"].sum())


@pytest.mark.gpu
def test_gpu_ao_tile_layouts_resume_and_variance():
    scene = scene_with_integrator(scene_path("c2_cornellbox.prc"), "(integrator :type 'ao' :sample_count 10)")
    whole = device_outputs(device_render(scene, scene.full_tile(), 0, 8))
    tiled = device_outputs(device_render(scene, scene.tiles(8, 8), 0, 8))
    for k in ("film", "count", "aov", "rng"):
        assert np.array_equal(whole[k], tiled[k]), k
    ctx = device_render(scene, scene.tiles(8, 8), 0, 4)
    ctx.render_tiles(scene.tiles(8, 8), 4, 4)
    resumed = device_outputs(ctx)
    for k in ("film", "count", "aov", "rng"):
        assert np.array_equal(whole[k], resumed[k]), k
    assert np.array_equal(whole["film"].view(np.uint32), oracle_ao(scene, scene.full_tile(), 0, 8, 10)["film"].view(np.uint32))


@pytest.mark.gpu
def test_gpu_ao_variance_and_extended_aovs_vs_oracle():
    scene = scene_with_integrator(scene_path("c1_sphere.prc"), "(integrator :type 'ao' :sample_count 5)",
                                  "(output :name 'v' (channel :type 'variance') (channel :type 'tangent'))")
    assert scene.settings.want_variance and scene.settings.want_aov_ext
    tiles = scene.full_tile()
    dev = device_outputs(device_render(scene, tiles, 0, 3), variance=True)
    w, h = scene.width, scene.height
    ref = oracle_ao(scene, tiles, 0, 3, 5, variance=(np.zeros((h, w, 3), np.float32), np.zeros((h, w, 3), np.float32)))
    assert_bit_exact(dev, ref)


@pytest.mark.gpu
def test_gpu_ao_known_answers():
    scene = prb.Scene.from_string(LONE_FLOOR % dict(n=8))
    check_lone_floor(device_outputs(device_render(scene, scene.full_tile(), 0, 1)), device_outputs(device_render(scene, scene.full_tile(), 0, 4)), 8)
    A, res, spp, n = 1.0, 64, 16, 16
    scene = ceiling_scene(A, res, spp, n)
    dev = device_outputs(device_render(scene, scene.full_tile(), 0, spp))
    p = ceiling_expectation(A)
    assert abs(float(dev["film"][..., 0].astype(np.float64).mean()) - p) < 5 * math.sqrt(p * (1 - p) / (res * res * spp * n))
    scene = ceiling_scene(1.0, 32, 1, 7)
    dev = device_outputs(device_render(scene, scene.full_tile(), 0, 1))
    allowed = {float(np.float32(1.0) - np.float32(k) / np.float32(7)) for k in range(8)}
    assert set(np.unique(dev["film"][..., 0]).tolist()) <= allowed


@pytest.mark.gpu
def test_gpu_ao_first_hit_aovs_equal_direct():
    """at 1 spp the camera draws of 'ao' and 'direct' are the same: first-hit AOVs and sample counts are bit-identical"""
    scene = prb.Scene.from_file(scene_path("c2_cornellbox.prc"))
    direct = device_render(scene, scene.full_tile(), 0, 1)
    ao = device_render(scene, scene.full_tile(), 0, 1, sample_count=10)
    a, b = direct.film_aov(), ao.film_aov()
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert np.array_equal(direct.film()[1], ao.film()[1])


@pytest.mark.gpu
def test_gpu_ao_no_state_leak_and_upload_resets():
    scene = prb.Scene.from_file(scene_path("c2_cornellbox.prc"))
    tiles = scene.tiles(8, 8)
    fresh = device_outputs(device_render(scene, tiles, 0, 4))
    ctx = device_render(scene, tiles, 0, 4)
    ctx.set_integrator("ao", 7)
    ctx.upload_rng(scene.rng_map())
    ctx.render_tiles(tiles, 0, 4)
    ctx.set_integrator("direct")
    ctx.upload_rng(scene.rng_map())
    ctx.reset_stats()
    ctx.render_tiles(tiles, 0, 4)
    again = device_outputs(ctx)
    for k in ("film", "count", "aov", "rng"):
        assert np.array_equal(fresh[k].view(np.uint8), again[k].view(np.uint8)), k
    ctx.set_integrator("ao", 7)
    ctx.upload_scene(scene)
    assert ctx.integrator == (prb.INTEGRATOR["direct"], 0)


@pytest.mark.gpu
def test_gpu_ao_set_integrator_errors():
    ctx = prb.Context(0)
    rec = prb.Integrator(prb.INTEGRATOR["ao"], 4)
    assert prb.device_lib().prb_set_integrator(ctx._h, C.byref(rec)) == -3  # PRB_ERR_NO_SCENE
    ctx.upload_scene(prb.Scene.from_file(scene_path("c2_cornellbox.prc")))
    for t, n, code in ((7, 1, -1), (prb.INTEGRATOR["ao"], 0, -1)):  # unknown type, 'ao' without rays: PRB_ERR_INVALID_ARG
        assert prb.device_lib().prb_set_integrator(ctx._h, C.byref(prb.Integrator(t, n))) == code
    from scene_strings import LPE_ZOO
    ctx.upload_scene(prb.Scene.from_string(LPE_ZOO))
    assert prb.device_lib().prb_set_integrator(ctx._h, C.byref(rec)) == -4  # PRB_ERR_UNSUPPORTED: LPE channels


@pytest.mark.gpu
def test_gpu_ao_through_render_and_render_context():
    scene = prb.Scene.from_string(LONE_FLOOR % dict(n=8))
    ctx, xyz, cnt = prb.render(scene)
    assert ctx.integrator == (prb.INTEGRATOR["ao"], 8)
    assert np.abs(xyz[..., 0] - cnt / np.float32(4)).max() <= 1e-6  # 4 spp of a floor no ray can miss from above
    host = prb.host_lib()
    rc = host.prh_render_context_create(scene._h, 0, 0, 1)
    assert rc
    dev = prb.Context.__new__(prb.Context)  # a view of the render context's device context, which the render context owns
    dev._h, dev._lib, dev.scene = C.c_void_p(host.prh_render_context_device(rc)), prb.device_lib(), scene
    try:
        assert host.prh_render_context_start(rc, 8, 8, 0) == 0
        assert dev.integrator == (prb.INTEGRATOR["ao"], 8)
        rxyz, rcnt = dev.film()
        assert np.array_equal(rxyz.view(np.uint32), xyz.view(np.uint32)) and np.array_equal(rcnt, cnt)
    finally:
        dev._h = None
        host.prh_render_context_destroy(rc)


@pytest.mark.gpu
def test_gpu_ao_tile_partition_on_two_gpus():
    if prb.device_lib().prb_device_count() < 2:
        pytest.skip("needs two GPUs")
    scene = scene_with_integrator(scene_path("c2_cornellbox.prc"), "(integrator :type 'ao' :sample_count 10)")
    tiles = scene.tiles(8, 8)
    single = device_outputs(device_render(scene, tiles, 0, 4))
    ctxs = []
    for r in range(2):
        c = prb.Context(r)
        c.upload_scene(scene)
        c.upload_rng(scene.rng_map())
        c.render_tiles([t for i, t in enumerate(tiles) if i % 2 == r], 0, 4)
        ctxs.append(c)
    prb.Context.film_reduce(ctxs, "tiles")
    xyz, cnt = ctxs[0].film()
    assert np.array_equal(xyz.view(np.uint32), single["film"].view(np.uint32)) and np.array_equal(cnt, single["count"])
