"""Sky / sun host models (pearray_b200/host/skysun.cpp) against the reference: the vendored Hosek-Wilkie C sources
(golden vectors written by tools/make_golden_sky.py from the reference's own sources), the documented default sun
position (src/skysun/skysun/SunLocation.h:7-8) and structural properties of the tables handed to the device
(Distribution2D normalisation, sky.cpp:134-166)."""
import ctypes as C
import os

import numpy as np
import pytest

import pearray_b200 as prb
from conftest import ROOT, scene_path
from scene_strings import SKYSUN_ZOO


def _host():
    h = prb.host_lib()
    h.prh_hosek_sky_radiance.restype = C.c_double
    h.prh_hosek_sky_radiance.argtypes = [C.c_double] * 6
    h.prh_sun_position.restype = None
    h.prh_sun_position.argtypes = [C.c_int] * 5 + [C.c_float] * 4 + [C.POINTER(C.c_float)] * 2
    h.prh_sun_radiance.restype = C.c_float
    h.prh_sun_radiance.argtypes = [C.c_float] * 3
    return h


def test_hosek_model_matches_reference_golden_vectors():
    g = np.load(os.path.join(ROOT, "tests", "golden", "hosek_reference.npz"))
    h = _host()
    ours = np.array([h.prh_hosek_sky_radiance(*row) for row in g["inputs"]])
    # same formula, same double arithmetic: bit equality up to libm pow/exp/cos differences between boxes
    np.testing.assert_allclose(ours, g["radiance"], rtol=1e-12, atol=0)


def test_hosek_model_matches_reference_library_bit_for_bit():
    """the stored radiances are the reference library's own results (x86-64, glibc); with that C library the restatement
    reproduces every one of them exactly, not only within the rtol above"""
    g = np.load(os.path.join(ROOT, "tests", "golden", "hosek_reference.npz"))
    h = _host()
    ours = np.array([h.prh_hosek_sky_radiance(*row) for row in g["inputs"]])
    assert np.array_equal(ours.view(np.uint64), g["radiance"].view(np.uint64))


def test_default_sun_position_is_the_documented_one():
    """SunLocation.h: 'Default is Saarbruecken 2020.05.06 12:00:00 (midday) which results in Elevation: 52.87 Azimuth: 143.27'"""
    el, az = C.c_float(), C.c_float()
    _host().prh_sun_position(2020, 5, 6, 12, 0, 0.0, 49.235422, 6.9965744, 2.0, C.byref(el), C.byref(az))
    assert abs(np.degrees(el.value) - 52.87) < 0.05
    assert abs(np.degrees(az.value) - 143.27) < 0.05


def test_sun_radiance_is_attenuated_solar_spectrum():
    h = _host()
    # zenith sun, clear air: between 30 % and 100 % of the extraterrestrial table value (25060.2 at 560 nm), SunRadiance.cpp:64-75
    r = h.prh_sun_radiance(560.0, 0.0, 2.0)
    assert 0.3 * 25060.2 < r < 25060.2
    # more air mass / more turbidity attenuate; blue more than red
    assert h.prh_sun_radiance(560.0, 1.3, 2.0) < r
    assert h.prh_sun_radiance(560.0, 0.0, 8.0) < r
    assert h.prh_sun_radiance(450.0, 1.4, 3.0) / h.prh_sun_radiance(450.0, 0.0, 3.0) < h.prh_sun_radiance(650.0, 1.4, 3.0) / h.prh_sun_radiance(650.0, 0.0, 3.0)
    assert h.prh_sun_radiance(900.0, 0.2, 3.0) >= 0.0


@pytest.mark.parametrize("which", ["complex", "zoo"])
def test_sky_tables_in_the_scene_description(which):
    scene = prb.Scene.from_file(scene_path("c4c_complex.prc")) if which == "complex" else prb.Scene.from_string(SKYSUN_ZOO)
    d = scene.desc.contents
    pool = np.ctypeslib.as_array(d.pool, shape=(d.n_pool,))
    lights = [d.lights[i] for i in range(d.n_lights)]
    sky = [l for l in lights if l.type == 2]
    sun = [l for l in lights if l.type in (3, 4)]
    assert len(sky) == 1 and len(sun) >= 1
    l = sky[0]
    extend = which == "complex"
    assert l.sky_extend == (1 if extend else 0)
    assert (l.az_count, l.el_count) == ((512, 256) if extend else (64, 32))
    assert (l.dist_w, l.dist_h) == (l.az_count, l.el_count * (2 if extend else 1))
    table = pool[l.table_offset:l.table_offset + l.table_count].reshape(l.el_count, l.az_count, 11)
    assert np.all(np.isfinite(table)) and table.min() >= 0 and table.max() > 0
    marginal = pool[l.dist_offset:l.dist_offset + l.dist_h + 1]
    cond = pool[l.dist_offset + l.dist_h + 1:l.dist_offset + l.dist_h + 1 + l.dist_h * (l.dist_w + 1)].reshape(l.dist_h, l.dist_w + 1)
    for cdf in (marginal, cond[0], cond[-1], cond[l.dist_h // 2]):
        assert cdf[0] == 0 and cdf[-1] == 1 and np.all(np.diff(cdf) >= 0)
    if extend:  # GROUND_PENALTY: almost all of the marginal mass is above the horizon
        assert marginal[l.dist_h // 2] < 0.01
    # light selection: a valid CDF over all lights, the pdfs are its increments
    cdf = np.ctypeslib.as_array(d.light_cdf, shape=(d.n_lights + 1,))
    assert cdf[0] == 0 and cdf[-1] == 1
    np.testing.assert_allclose([x.select_pdf for x in lights], np.diff(cdf), rtol=1e-6)
    for s in sun:
        n = np.array(list(s.sun_dir))
        assert abs(np.linalg.norm(n) - 1) < 1e-5
        assert abs(np.dot(n, list(s.sun_dx))) < 1e-5 and abs(np.dot(n, list(s.sun_dy))) < 1e-5
        spec = pool[s.table_offset:s.table_offset + s.table_count]
        assert s.table_count == 64 and (s.table_start, s.table_end) == (360.0, 760.0) and spec.max() > 0
        if s.type == 4:
            assert s.sun_cos_theta == 1.0
        else:
            assert 0.99 < s.sun_cos_theta < 1.0 and abs(s.sun_pdf - 1 / (2 * np.pi * (1 - s.sun_cos_theta))) / s.sun_pdf < 1e-3


@pytest.mark.parametrize("which", ["complex", "zoo"])
def test_infinite_light_sampling_is_consistent_with_its_evaluation(which):
    """the analogue of src/tests/materials.cpp for lights: a direction drawn by SkyLight / SunLight::sampleDir evaluates (eval)
    to the same radiance and the same solid-angle pdf it was drawn with; the sky pdf integrates to one over the sphere and
    its samples stay above the horizon as far as the ground penalty allows; the delta sun returns its fixed direction"""
    from oracle_binding import OracleScene
    scene = prb.Scene.from_file(scene_path("c4c_complex.prc")) if which == "complex" else prb.Scene.from_string(SKYSUN_ZOO)
    d = scene.desc.contents
    ora = OracleScene(scene)
    wvl = [560.0, 540.0, 400.0, 600.0]
    for li in range(d.n_lights):
        l = d.lights[li]
        state, up, inv_pdf = 0x853C49E6748FEA9B | 3, 0, []
        for _ in range(3000):
            r, state = ora.light_sample_and_eval(li, (0.0, 0.0, 0.5), wvl, state)
            if l.type == 4:  # delta sun: its direction, pdf 1, never evaluated
                assert r["delta"] and r["pdf"] == 1.0 and np.allclose(r["outgoing"], list(l.sun_dir), atol=1e-6)
                continue
            assert not r["delta"] and abs(np.linalg.norm(r["outgoing"]) - 1) < 1e-5
            if r["pdf"] == 0:
                continue
            # cell-boundary samples may land in the neighbouring table cell when re-evaluated: compare with a tolerance and
            # allow a few such samples
            ok = abs(r["pdf"] - r["eval_pdf"]) <= 2e-3 * r["pdf"] and np.allclose(r["radiance"], r["eval_radiance"], rtol=2e-3, atol=1e-6)
            up += ok
            inv_pdf.append(1.0 / r["pdf"])
            if l.type == 3:  # cone sun: inside the cone, uniform pdf
                assert np.dot(r["outgoing"], list(l.sun_dir)) >= l.sun_cos_theta - 1e-6 and abs(r["pdf"] - l.sun_pdf) <= 1e-6 * l.sun_pdf
        if l.type == 4:
            continue
        assert up >= 0.97 * len(inv_pdf), (li, l.type, up, len(inv_pdf))
        if l.type == 2:
            # E[1 / pdf] = measure of the support = 4 pi for the extended sky.  The non-extended sky maps v to [0, pi/2] but keeps
            # the extended form's Jacobian 2 pi^2 cos(el) (sky.cpp:69-70,97-99), i.e. half the true density: 2 x 2 pi as well.
            want = 4 * np.pi
            assert abs(np.mean(inv_pdf) - want) < 0.35 * want
        if l.type == 3:
            assert abs(np.mean(inv_pdf) - 2 * np.pi * (1 - l.sun_cos_theta)) < 1e-3 * np.mean(inv_pdf)
