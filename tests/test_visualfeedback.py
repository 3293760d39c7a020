"""The visual-feedback integrator ('visualfeedback', 'vf'): loader and C ABI on the CPU, known answers on the oracle (oracle_ao/)
and on the device, and the device bit-exact against the oracle (`-m gpu`).

The known answers use an orthographic camera, the 'uniform' sampler (one fixed point per pixel) and a block filter of radius 0,
so each pixel's value is the colour of the one point its camera ray hits, folded as XYZ = M c."""
import ctypes as C
import math
import os

import numpy as np
import pytest

import pearray_b200 as prb
from conftest import scene_path
from oracle_binding import _p
from test_ao import ao_lib, assert_bit_exact, device_outputs, scene_with_integrator
from test_golden_oracle import STAT_NAMES
from test_image_output import read_exr

MODES = list(prb.VF_MODES)

# RGBConverter::fromXYZ (the film's sRGB tone mode) and M, its inverse rounded to fp32: the RGB -> XYZ fold of the integrator
FROM_XYZ = np.array([[3.240970e+00, -1.537383e+00, -4.986108e-01], [-9.692436e-01, 1.875968e+00, 4.155506e-02],
                     [5.563008e-02, -2.039770e-01, 1.056972e+00]], np.float32)
M = np.linalg.inv(FROM_XYZ.astype(np.float64)).astype(np.float32)


def palette(ids):
    """the integrator's palette(id) restated in float32 numpy: golden-ratio hue, S = 0.7, V = 0.9, textbook HSV -> RGB"""
    x = np.asarray(ids, np.uint32).astype(np.float32) * np.float32(0.618034)
    h6 = np.float32(6) * (x - np.floor(x))
    i = np.floor(h6)
    f = h6 - i
    one, S, V = np.float32(1), np.float32(0.7), np.float32(0.9)
    p, q, t = V * (one - S), V * (one - S * f), V * (one - S * (one - f))
    V = np.full_like(f, V)
    p = np.full_like(f, p)
    sector = i.astype(np.int64) % 6
    return np.stack([np.choose(sector, c) for c in ((V, q, p, p, t, V), (t, V, V, q, p, p), (p, p, t, V, V, q))], axis=-1)


def to_xyz(c):
    """XYZ = M c with the integrator's order of operations (fp32, no fused multiply-add)"""
    c = np.asarray(c, np.float32)
    return np.stack([(M[r, 0] * c[..., 0] + M[r, 1] * c[..., 1]) + M[r, 2] * c[..., 2] for r in range(3)], axis=-1)


def oracle_vf(scene, tiles, first, count, mode, rng=None, variance=False):
    """renders iterations [first, first + count) with the 'visualfeedback' oracle"""
    w, h = scene.width, scene.height
    rng = scene.rng_map() if rng is None else np.array(rng, dtype=np.uint64, copy=True)
    film, cnt = np.zeros((h, w, 3), np.float32), np.zeros((h, w), np.uint32)
    aov, aove, feedback = np.zeros((h, w, 10), np.float32), np.zeros((h, w, 11), np.float32), np.zeros((h, w), np.uint32)
    vm, vv = (np.zeros((h, w, 3), np.float32), np.zeros((h, w, 3), np.float32)) if variance else (None, None)
    stats = np.zeros(11, np.uint64)
    lib = ao_lib()
    if not hasattr(lib, "_vf_ready"):
        lib.orc_render_vf.argtypes = lib.orc_render_ao.argtypes
        lib._vf_ready = True
    hdl = lib.orc_scene_create(scene.desc)
    try:
        lib.orc_render_vf(hdl, _p(rng), prb.make_tiles(tiles), len(tiles), first, count, _p(film), _p(cnt), _p(aov), _p(stats), os.cpu_count() or 1,
                          _p(feedback), None if vm is None else _p(vm), None if vv is None else _p(vv), None, _p(aove),
                          mode if isinstance(mode, int) else prb.VF_MODES[mode])
    finally:
        lib.orc_scene_destroy(hdl)
    out = dict(film=film, count=cnt, aov=aov, aov_ext=aove, feedback=feedback, rng=rng, stats=dict(zip(STAT_NAMES, (int(x) for x in stats))))
    if variance:
        out["online_mean"], out["online_variance"] = vm, vv
    return out


# scenes of the known answers: entities %(entities)s under an orthographic camera at %(cam)s looking along %(dir)s
KNOWN = """
(scene :name 'vf_known' :render_width %(res)d :render_height %(res)d :camera 'Camera'
 (integrator :type 'visualfeedback' :mode '%(mode)s')
 (sampler :slot 'aa' :type 'uniform' :sample_count 4)
 (filter :slot 'pixel' :type 'block' :radius 0)
 (camera :name 'Camera' :type 'orthographic' :width %(extent)g :height %(extent)g :local_direction %(dir)s :local_up [0,1,0]
   :local_right [1,0,0] :position %(cam)s)
 (material :name 'm' :type 'diffuse' :albedo 0.8)
 %(entities)s
)
"""
FLOOR = "(entity :name 'floor' :type 'plane' :centering true :width 2 :height 2 :material 'm' :position [0,0,0])"


def known_scene(mode, entities=FLOOR, extent=4.0, res=32, below=False):
    return prb.Scene.from_string(KNOWN % dict(res=res, mode=mode, extent=extent, entities=entities,
                                              cam="[0,0,-2]" if below else "[0,0,2]", dir="[0,0,1]" if below else "[0,0,-1]"))


def tilted_plane(theta):
    c, s = math.cos(theta), math.sin(theta)
    return ("(entity :name 'tilted' :type 'plane' :centering true :width 8 :height 8 :material 'm' :transform [1,0,0,0, 0,%r,%r,0, 0,%r,%r,0, 0,0,0,1])"
            % (c, -s, s, c))


THREE = " ".join("(entity :name 'e%d' :type 'plane' :centering true :width 1 :height 3 :material 'm' :position [%g,0,0])" % (k, x)
                 for k, x in enumerate((-1.0, 0.0, 1.0)))


# ----------------------------------------------------------------------------- known answers (oracle and device)
def check_ndotv(render):
    for theta in (0.0, 0.3, 1.0):
        r = render(known_scene("ndotv", tilted_plane(theta), extent=2), 1)
        assert np.all(r["count"] == 1)
        c = np.float32(math.cos(theta))
        assert np.abs(r["film"] - to_xyz([c, c, c])).max() <= 2e-6
        assert np.abs(r["film"][..., 1] - c).max() <= 2e-6  # Y = cos(theta)


def check_inside(render):
    above = render(known_scene("inside"), 1)
    below = render(known_scene("inside", below=True), 1)
    for r, colour in ((above, [0, 1, 0]), (below, [1, 0, 0])):  # front face green, back face red
        hit = r["count"] > 0
        assert hit.any() and (~hit).any()
        assert np.array_equal(r["film"][hit], np.broadcast_to(to_xyz(colour), (int(hit.sum()), 3)))


def check_parameter(render):
    r = render(known_scene("parameter", extent=2), 1)  # the 2 x 2 floor fills the image
    assert np.all(r["count"] == 1)
    uv = r["film"].astype(np.float64) @ np.linalg.inv(M.astype(np.float64)).T
    assert np.abs(uv[..., 2]).max() <= 1e-6
    assert np.array_equal(r["film"], to_xyz(np.concatenate([r["aov"][..., 6:8], np.zeros_like(r["aov"][..., :1])], axis=-1)))
    n = uv.shape[0]
    # the plane's uv runs from 0 to 1 across its width and height: each of u and v steps by 1/n along one image axis and is
    # constant along the other, and the two run along different axes
    axes = []
    for a in (uv[..., 0], uv[..., 1]):
        assert a.min() >= -1e-6 and a.max() <= 1 + 1e-6
        steps = [np.abs(np.diff(a, axis=k)) for k in (0, 1)]
        moving = [k for k in (0, 1) if np.abs(steps[k] - 1 / n).max() <= 1e-5]
        assert len(moving) == 1 and steps[1 - moving[0]].max() <= 1e-5
        axes.append(moving[0])
    assert axes[0] != axes[1]


def check_entity_ids(render):
    r = render(known_scene("colored_entity_id", THREE, extent=4), 1)
    hit = r["count"] > 0
    ids = r["aov"][..., 9][hit].astype(np.uint32)
    assert set(ids.tolist()) == {0, 1, 2}
    assert np.array_equal(r["film"][hit], to_xyz(palette(ids)))
    assert len({tuple(c) for c in palette([0, 1, 2]).tolist()}) == 3


def check_misses(render):
    r = render(known_scene("colored_entity_id"), 3)
    miss = r["count"] == 0
    assert miss.any() and (~miss).any() and np.all(r["count"][~miss] == 3)
    assert not r["film"][miss].any()
    assert r["stats"]["background_hit_count"] == 3 * int(miss.sum())
    assert r["stats"]["entity_hit_count"] == 3 * int((~miss).sum())


CHECKS = [check_ndotv, check_inside, check_parameter, check_entity_ids, check_misses]


def oracle_render(scene, iters):
    return oracle_vf(scene, scene.full_tile(), 0, iters, scene.integrator.mode)


def device_render(scene, iters):
    ctx = prb.Context(0)
    ctx.upload_scene(scene)
    ctx.upload_rng(scene.rng_map())
    ctx.render_tiles(scene.full_tile(), 0, iters)
    return device_outputs(ctx)


# ----------------------------------------------------------------------------- CPU: loader and ABI
@pytest.mark.parametrize("name", ["visualfeedback", "vf"])
def test_loader_yields_the_integrator_record(name):
    for mode, value in prb.VF_MODES.items():
        scene = prb.Scene.from_string(KNOWN.replace("'visualfeedback'", "'%s'" % name) % dict(res=8, mode=mode, extent=4, entities=FLOOR, cam="[0,0,2]", dir="[0,0,-1]"))
        rec = scene.integrator
        assert (rec.type, rec.mode) == (prb.INTEGRATOR["visualfeedback"], value)
        assert scene.settings.max_ray_depth == 1
    default = prb.Scene.from_string((KNOWN % dict(res=8, mode="x", extent=4, entities=FLOOR, cam="[0,0,2]", dir="[0,0,-1]")).replace(" :mode 'x'", ""))
    assert (default.integrator.type, default.integrator.mode) == (prb.INTEGRATOR["visualfeedback"], prb.VF_MODES["colored_entity_id"])
    names = {l.split(":")[0]: l.split(":")[1].split() for l in default.plugins().strip().splitlines()}["integrator"]
    assert "visualfeedback" in names and "vf" in names


def test_unknown_mode_logs_an_error_and_falls_back_to_direct(capfd):
    scene = known_scene("colored_ray_id")
    assert "Unknown mode colored_ray_id" in "".join(capfd.readouterr())
    assert scene.integrator.type == prb.INTEGRATOR["direct"]
    assert scene.settings.max_ray_depth > 1 and scene.settings.do_nee


def test_mode_shares_the_record_word_with_sample_count():
    assert C.sizeof(prb.Integrator) == prb.host_lib().prh_abi_sizeof(b"prb_integrator") == 8
    rec = prb.Integrator(prb.INTEGRATOR["visualfeedback"])
    rec.mode = prb.VF_MODES["ndotv"]
    assert rec.sample_count == rec.mode == 6


def test_palette_restatement():
    """hues of consecutive ids are far apart and every colour keeps S = 0.7, V = 0.9"""
    c = palette(np.arange(64)).astype(np.float64)
    assert np.allclose(c.max(-1), 0.9, atol=1e-6) and np.allclose(c.min(-1), 0.9 * 0.3, atol=1e-6)
    assert np.all(np.abs(np.diff(c, axis=0)).max(-1) > 0.1)


# ----------------------------------------------------------------------------- CPU: known answers on the oracle
@pytest.mark.parametrize("check", CHECKS, ids=[c.__name__ for c in CHECKS])
def test_oracle_known_answers(check):
    check(oracle_render)


# ----------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("check", CHECKS, ids=[c.__name__ for c in CHECKS])
def test_gpu_known_answers(check):
    check(device_render)


# scene, tiles (crops: the oracle walks them on the CPU), iterations
GPU_CASES = {
    "c0": ("c0_evaluation.prc", [(64, 64, 128, 128), (150, 100, 214, 164)], 3),
    "c1": ("c1_sphere.prc", [(468, 400, 532, 464), (200, 700, 264, 764)], 3),
    "c2": ("c2_cornellbox.prc", [(100, 100, 164, 164), (300, 250, 364, 314)], 3),
    "c3": ("c3_cornellbox_glassy.prc", [(64, 64, 128, 128), (100, 150, 164, 214)], 3),
    "c4": ("c4_boltsandgears.prc", [(400, 400, 464, 464), (600, 500, 664, 564)], 2),
    "c4c": ("c4c_complex.prc", [(900, 500, 964, 548)], 2),
}
_scenes = {}


def vf_scene(name):
    """the case's scene with 'vf' in its default mode, the variance AOV and the extended AOVs (loaded once per module)"""
    if name not in _scenes:
        _scenes[name] = scene_with_integrator(scene_path(GPU_CASES[name][0]), "(integrator :type 'visualfeedback')",
                                              "(output :name 'vf' (channel :type 'variance') (channel :type 'tangent'))")
    return _scenes[name]


def gpu_vs_oracle(name, mode, tiles, iters):
    scene = vf_scene(name)
    assert scene.settings.want_variance and scene.settings.want_aov_ext
    ctx = prb.Context(0)
    ctx.upload_scene(scene)  # selects the scene's 'vf' record
    assert ctx.integrator == (prb.INTEGRATOR["visualfeedback"], prb.VF_MODES["colored_entity_id"])
    ctx.set_integrator("visualfeedback", mode=mode)
    ctx.upload_rng(scene.rng_map())
    ctx.render_tiles(tiles, 0, iters)
    dev = device_outputs(ctx, variance=True)
    assert_bit_exact(dev, oracle_vf(scene, tiles, 0, iters, mode, variance=True))
    return dev


@pytest.mark.gpu
@pytest.mark.parametrize("trace", [None, "bvh"])
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", list(GPU_CASES))
def test_gpu_vf_bit_exact_vs_oracle(name, mode, trace, monkeypatch):
    if trace is None:
        monkeypatch.delenv("PRB_TRACE_MODE", raising=False)
    else:
        monkeypatch.setenv("PRB_TRACE_MODE", trace)
    _, tiles, iters = GPU_CASES[name]
    dev = gpu_vs_oracle(name, mode, tiles, iters)
    assert dev["count"].sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("trace", ["static", "persistent"])
@pytest.mark.parametrize("mode", MODES)
def test_gpu_vf_trace_variants_on_a_bvh_scene(mode, trace, monkeypatch):
    monkeypatch.setenv("PRB_TRACE_MODE", trace)
    _, tiles, iters = GPU_CASES["c4"]
    gpu_vs_oracle("c4", mode, tiles, iters)


def fresh_context(scene, tiles, first, count, device=0):
    ctx = prb.Context(device)
    ctx.upload_scene(scene)
    ctx.upload_rng(scene.rng_map())
    ctx.render_tiles(tiles, first, count)
    return ctx


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["colored_entity_id", "ndotv"])
def test_gpu_vf_tiles_and_resume(mode):
    scene = scene_with_integrator(scene_path("c2_cornellbox.prc"), "(integrator :type 'visualfeedback' :mode '%s')" % mode)
    tiles = scene.tiles(8, 8)
    whole = device_outputs(fresh_context(scene, scene.full_tile(), 0, 8))
    # interleaved tile contexts, reduced into the first
    ctxs = []
    for r in range(2):
        c = prb.Context(0)
        c.upload_scene(scene)
        c.upload_rng(scene.rng_map())
        c.render_tiles([t for i, t in enumerate(tiles) if i % 2 == r], 0, 8)
        ctxs.append(c)
    prb.Context.film_reduce(ctxs, "tiles")
    xyz, cnt = ctxs[0].film()
    assert np.array_equal(xyz.view(np.uint32), whole["film"].view(np.uint32)) and np.array_equal(cnt, whole["count"])
    # iterations [0, 3) then [3, 8)
    ctx = fresh_context(scene, tiles, 0, 3)
    ctx.render_tiles(tiles, 3, 5)
    resumed = device_outputs(ctx)
    for k in ("film", "count", "aov", "rng"):
        assert np.array_equal(whole[k].view(np.uint8), resumed[k].view(np.uint8)), k


@pytest.mark.gpu
def test_gpu_no_state_leaks_between_integrators():
    scene = prb.Scene.from_file(scene_path("c2_cornellbox.prc"))
    tiles = scene.tiles(8, 8)
    fresh = device_outputs(fresh_context(scene, tiles, 0, 4))
    ctx = fresh_context(scene, tiles, 0, 4)
    ctx.set_integrator("visualfeedback", mode="inside")
    assert ctx.integrator == (prb.INTEGRATOR["visualfeedback"], prb.VF_MODES["inside"])
    ctx.upload_rng(scene.rng_map())
    ctx.render_tiles(tiles, 0, 4)
    ctx.set_integrator("direct")
    ctx.upload_rng(scene.rng_map())
    ctx.reset_stats()
    ctx.render_tiles(tiles, 0, 4)
    again = device_outputs(ctx)
    for k in ("film", "count", "aov", "rng"):
        assert np.array_equal(fresh[k].view(np.uint8), again[k].view(np.uint8)), k
    for n in STAT_NAMES:
        assert fresh["stats"][n] == again["stats"][n], n
    ctx.set_integrator("visualfeedback", mode="ndotv")
    ctx.upload_scene(scene)
    assert ctx.integrator == (prb.INTEGRATOR["direct"], 0)


@pytest.mark.gpu
def test_gpu_set_integrator_errors():
    vf = prb.INTEGRATOR["visualfeedback"]
    ctx = prb.Context(0)
    assert prb.device_lib().prb_set_integrator(ctx._h, C.byref(prb.Integrator(vf, 0))) == -3  # PRB_ERR_NO_SCENE
    ctx.upload_scene(prb.Scene.from_file(scene_path("c2_cornellbox.prc")))
    assert prb.device_lib().prb_set_integrator(ctx._h, C.byref(prb.Integrator(vf, len(MODES)))) == -1  # PRB_ERR_INVALID_ARG
    from scene_strings import LPE_ZOO
    ctx.upload_scene(prb.Scene.from_string(LPE_ZOO))
    assert prb.device_lib().prb_set_integrator(ctx._h, C.byref(prb.Integrator(vf, 0))) == -4  # PRB_ERR_UNSUPPORTED: LPE channels


@pytest.mark.gpu
def test_gpu_output_file_gives_back_the_palette(tmp_path):
    """through RenderContext: the sRGB image written for a 'colored_entity_id' render holds the palette colours"""
    scene = prb.Scene.from_string((KNOWN % dict(res=32, mode="colored_entity_id", extent=4, entities=THREE, cam="[0,0,2]", dir="[0,0,-1]"))
                                  .replace("(filter", "(output :name 'image' (channel :type 'color' :color 'srgb'))\n (filter"))
    host = prb.host_lib()
    rc = host.prh_render_context_create(scene._h, 0, 0, 1)
    assert rc
    dev = prb.Context.__new__(prb.Context)  # a view of the render context's device context, which the render context owns
    dev._h, dev._lib, dev.scene = C.c_void_p(host.prh_render_context_device(rc)), prb.device_lib(), scene
    try:
        assert host.prh_render_context_start(rc, 8, 8, 0) == 0
        assert dev.integrator == (prb.INTEGRATOR["visualfeedback"], prb.VF_MODES["colored_entity_id"])
        ids = dev.film_aov()[..., 9] / np.maximum(dev.film()[1], 1)
        hit = dev.film()[1] > 0
        assert host.prh_render_context_save_outputs(rc, str(tmp_path).encode()) >= 1
    finally:
        dev._h = None
        host.prh_render_context_destroy(rc)
    _, _, pl = read_exr(os.path.join(tmp_path, "results", "image.exr"))
    rgb = np.stack([pl[c] for c in "RGB"], axis=-1)
    assert np.abs(rgb[hit] - palette(ids[hit].astype(np.uint32))).max() <= 1e-5
    assert not rgb[~hit].any()


@pytest.mark.gpu
def test_gpu_ndotv_scene_file_renders_through_render_context(tmp_path):
    scene = scene_with_integrator(scene_path("c2_cornellbox.prc"), "(integrator :type 'visualfeedback' :mode 'ndotv')")
    scene.set_spp(2)
    host = prb.host_lib()
    rc = host.prh_render_context_create(scene._h, 0, 0, 1)
    assert rc
    try:
        assert host.prh_render_context_start(rc, 8, 8, 0) == 0
        assert host.prh_render_context_save_outputs(rc, str(tmp_path).encode()) >= 1
    finally:
        host.prh_render_context_destroy(rc)
    exrs = [f for f in os.listdir(os.path.join(tmp_path, "results")) if f.endswith(".exr")]
    assert exrs
    _, chans, pl = read_exr(os.path.join(tmp_path, "results", exrs[0]))
    y = pl["G"] if "G" in pl else next(iter(pl.values()))
    assert np.isfinite(y).all() and y.max() > 0.1
