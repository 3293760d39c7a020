"""pearray_b200 -- B200-native spectral path-tracing hot path behind PearRay's plugin API.

Python is only a thin ctypes shim here (tests, bench, FFI illustration).  The product is
  libprb200.so       hand-written CUDA (sm_100a) + the C ABI of include/prb200_abi.h
  libprb200_host.so  C++17 host layer mirroring PearRay's loader / plugin factories / render driver
There is NO CPU fallback: every compute entry point raises when the CUDA library or a GPU is missing.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
INVALID_ID = 0xFFFFFFFF


class PrbError(RuntimeError):
    pass


# ----------------------------------------------------------------------------- ctypes mirrors of prb200_abi.h
class Tile(C.Structure):
    _fields_ = [("sx", C.c_uint32), ("sy", C.c_uint32), ("ex", C.c_uint32), ("ey", C.c_uint32)]


class RaySoA(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("org_x", "org_y", "org_z", "dir_x", "dir_y", "dir_z", "tmin", "tmax")]


class HitSoA(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("entity_id", "primitive_id", "u", "v", "t")]


class Settings(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("film_width", C.c_uint32), ("film_height", C.c_uint32),
                ("view_x", C.c_uint32), ("view_y", C.c_uint32), ("view_w", C.c_uint32), ("view_h", C.c_uint32),
                ("max_sample_count", C.c_uint32), ("max_ray_depth", C.c_uint32), ("soft_max_ray_depth", C.c_uint32),
                ("mis_power", C.c_uint32), ("do_nee", C.c_uint32), ("do_direct", C.c_uint32), ("emissive_scatter", C.c_uint32),
                ("spectral_mono", C.c_uint32), ("spectral_hero", C.c_uint32),
                ("spectral_start", C.c_float), ("spectral_end", C.c_float),
                ("light_range_start", C.c_float), ("light_range_end", C.c_float),
                ("time_alpha", C.c_float), ("time_beta", C.c_float),
                ("filter_radius", C.c_int32), ("filter_offset", C.c_uint32), ("film_monotonic", C.c_uint32), ("want_variance", C.c_uint32), ("want_aov_ext", C.c_uint32)]


class Camera(C.Structure):
    _fields_ = [("origin", C.c_float * 3), ("right", C.c_float * 3), ("up", C.c_float * 3), ("dir", C.c_float * 3),
                ("near_t", C.c_float), ("far_t", C.c_float), ("type", C.c_uint32), ("has_dof", C.c_uint32),
                ("aperture_x", C.c_float * 3), ("aperture_y", C.c_float * 3)]


class Sampler(C.Structure):
    _fields_ = [("type", C.c_uint32), ("max_samples", C.c_uint32), ("bins_1d", C.c_uint32), ("m2d_x", C.c_uint32),
                ("m2d_y", C.c_uint32), ("seed", C.c_uint32), ("table_offset", C.c_uint32), ("_pad", C.c_uint32)]


class SpectralMapper(C.Structure):
    _fields_ = [("type", C.c_uint32), ("cdf_offset", C.c_uint32), ("cdf_size", C.c_uint32), ("trunc_cdf_start", C.c_float),
                ("trunc_cdf_end", C.c_float)]


class Node(C.Structure):
    _fields_ = [("type", C.c_uint32), ("flags", C.c_uint32), ("a", C.c_uint32), ("b", C.c_uint32), ("p", C.c_float * 4)]


class Material(C.Structure):
    _fields_ = [("type", C.c_uint32), ("flags", C.c_uint32), ("node", C.c_uint32 * 4), ("f", C.c_float * 12)]


class Emission(C.Structure):
    _fields_ = [("radiance_node", C.c_uint32), ("_pad", C.c_uint32)]


class Mesh(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("vertex_offset", "vertex_count", "face_offset", "face_count", "features",
                                          "blas_root", "uv_offset", "normal_offset")]


class Entity(C.Structure):
    _fields_ = [("type", C.c_uint32), ("mesh_id", C.c_uint32), ("material_offset", C.c_uint32), ("material_count", C.c_uint32),
                ("emission_id", C.c_uint32), ("light_id", C.c_uint32), ("visibility", C.c_uint32), ("blas_root", C.c_uint32),
                ("local_to_world", C.c_float * 12), ("world_to_local", C.c_float * 12), ("normal_matrix", C.c_float * 9),
                ("jacobian_det", C.c_float), ("world_area", C.c_float), ("pdf_area", C.c_float), ("geo", C.c_float * 45)]


class Light(C.Structure):
    _fields_ = [("type", C.c_uint32), ("entity_id", C.c_uint32), ("emission_id", C.c_uint32), ("radiance_node", C.c_uint32),
                ("background_node", C.c_uint32), ("env_split", C.c_uint32), ("select_pdf", C.c_float), ("scene_radius", C.c_float),
                ("normal_matrix", C.c_float * 9), ("inv_normal_matrix", C.c_float * 9),
                ("table_offset", C.c_uint32), ("table_count", C.c_uint32), ("table_start", C.c_float), ("table_end", C.c_float),
                ("az_count", C.c_uint32), ("el_count", C.c_uint32), ("dist_offset", C.c_uint32), ("dist_w", C.c_uint32),
                ("dist_h", C.c_uint32), ("sky_extend", C.c_uint32), ("sun_dir", C.c_float * 3), ("sun_dx", C.c_float * 3),
                ("sun_dy", C.c_float * 3), ("sun_cos_theta", C.c_float), ("sun_pdf", C.c_float)]


MAX_LPE = 8


class LPE(C.Structure):
    _fields_ = [("next_offset", C.c_uint32), ("final_offset", C.c_uint32), ("n_states", C.c_uint32), ("start_state", C.c_uint32)]


class SceneDesc(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("settings", Settings), ("camera", Camera),
                ("aa_sampler", Sampler), ("lens_sampler", Sampler), ("time_sampler", Sampler), ("pixel_mapper", SpectralMapper),
                ("n_nodes", C.c_uint32), ("nodes", C.POINTER(Node)),
                ("n_materials", C.c_uint32), ("materials", C.POINTER(Material)),
                ("n_emissions", C.c_uint32), ("emissions", C.POINTER(Emission)),
                ("n_entities", C.c_uint32), ("entities", C.POINTER(Entity)),
                ("n_entity_materials", C.c_uint32), ("entity_materials", C.POINTER(C.c_uint32)),
                ("n_meshes", C.c_uint32), ("meshes", C.POINTER(Mesh)),
                ("n_vertices", C.c_uint32), ("vertices", C.POINTER(C.c_float)),
                ("normals", C.POINTER(C.c_float)), ("uvs", C.POINTER(C.c_float)),
                ("n_faces", C.c_uint32), ("face_indices", C.POINTER(C.c_uint32)), ("face_slots", C.POINTER(C.c_uint32)),
                ("n_lights", C.c_uint32), ("lights", C.POINTER(Light)), ("light_cdf", C.POINTER(C.c_float)),
                ("inf_light_selection_probability", C.c_float),
                ("tlas_root", C.c_uint32), ("n_bvh_nodes", C.c_uint32), ("bvh_nodes", C.c_void_p),
                ("n_bvh_tris", C.c_uint32), ("bvh_tris", C.c_void_p),
                ("n_tlas_refs", C.c_uint32), ("tlas_refs", C.POINTER(C.c_uint32)),
                ("n_pool", C.c_uint32), ("pool", C.POINTER(C.c_float)),
                ("cie_offset", C.c_uint32), ("_pad", C.c_uint32),
                ("upsampler_offset", C.c_uint32), ("upsampler_res", C.c_uint32),
                ("n_lpe", C.c_uint32), ("n_lpe_bytes", C.c_uint32), ("lpe_tables", C.POINTER(C.c_uint8)), ("lpe", LPE * MAX_LPE)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("camera_ray_count", "light_ray_count", "primary_ray_count", "bounce_ray_count",
                                          "shadow_ray_count", "monochrome_ray_count", "pixel_sample_count", "entity_hit_count",
                                          "background_hit_count", "camera_depth_count", "light_depth_count",
                                          "kernel_launches", "wavefront_iterations")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}

    @property
    def ray_count(self):  # RenderStatistics::rayCount, reference src/core/renderer/RenderStatistics.h:33-36
        return int(self.primary_ray_count + self.bounce_ray_count + self.shadow_ray_count)


INTEGRATOR = {"direct": 0, "ao": 1, "visualfeedback": 2}  # PRB_INTEGRATOR_*
# PRB_VF_*: what the colour of a 'visualfeedback' pixel shows
VF_MODES = {"colored_entity_id": 0, "colored_material_id": 1, "colored_emission_id": 2, "colored_primitive_id": 3, "parameter": 4,
            "inside": 5, "ndotv": 6}


class Integrator(C.Structure):
    """prb_integrator; its second word is a union: sample_count ('ao') or mode ('visualfeedback')"""
    _fields_ = [("type", C.c_uint32), ("sample_count", C.c_uint32)]
    mode = property(lambda self: self.sample_count, lambda self, v: setattr(self, "sample_count", v))


class MaterialQuery(C.Structure):
    _fields_ = [("V", C.c_float * 3), ("L", C.c_float * 3), ("wavelength_nm", C.c_float * 4), ("uv", C.c_float * 2),
                ("ray_flags", C.c_uint32), ("material_id", C.c_uint32), ("rng_state", C.c_uint64)]


class MaterialResult(C.Structure):
    _fields_ = [("weight", C.c_float * 4), ("pdf_s", C.c_float * 4), ("L", C.c_float * 3), ("flags", C.c_uint32),
                ("type", C.c_uint32), ("rng_state", C.c_uint64)]


# ----------------------------------------------------------------------------- library loading
_dev = None
_host = None

# every symbol include/prb200_abi.h declares
ABI_SYMBOLS = ["prb_create", "prb_destroy", "prb_last_error", "prb_device_count", "prb_upload_scene", "prb_upload_rng",
               "prb_download_rng", "prb_render_tiles", "prb_sync", "prb_film_clear", "prb_film_download",
               "prb_film_download_aov", "prb_film_download_feedback", "prb_film_download_variance", "prb_film_export_device", "prb_film_import_device", "prb_trace_closest",
               "prb_trace_any", "prb_trace_closest_device", "prb_trace_any_device", "prb_generate_camera_rays",
               "prb_material_eval", "prb_material_sample", "prb_get_stats", "prb_reset_stats", "prb_last_device_ms",
               "prb_set_profiling", "prb_get_stage_times", "prb_film_reduce", "prb_comm_unique_id", "prb_comm_init",
               "prb_comm_destroy", "prb_film_reduce_comm", "prb_last_reduce_ms", "prb_set_shading_mode", "prb_get_shading_mode", "prb_film_download_lpe", "prb_film_download_aov_ext",
               "prb_set_integrator", "prb_get_integrator"]


def device_lib():
    """libprb200.so (CUDA + C ABI).  Raises when the extension has not been built -- there is no fallback."""
    global _dev
    if _dev is None:
        path = os.path.join(_HERE, "libprb200.so")
        if not os.path.exists(path):
            raise PrbError("libprb200.so is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(the product has no CPU fallback)")
        lib = C.CDLL(path, mode=C.RTLD_GLOBAL)
        lib.prb_last_error.restype = C.c_char_p
        lib.prb_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        lib.prb_destroy.argtypes = [C.c_void_p]
        lib.prb_upload_scene.argtypes = [C.c_void_p, C.POINTER(SceneDesc)]
        lib.prb_upload_rng.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        lib.prb_download_rng.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        lib.prb_render_tiles.argtypes = [C.c_void_p, C.POINTER(Tile), C.c_size_t, C.c_uint32, C.c_uint32]
        lib.prb_sync.argtypes = [C.c_void_p]
        lib.prb_film_clear.argtypes = [C.c_void_p]
        lib.prb_film_download.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        lib.prb_film_download_aov.argtypes = [C.c_void_p, C.c_void_p]
        lib.prb_film_download_feedback.argtypes = [C.c_void_p, C.c_void_p]
        lib.prb_film_download_variance.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        lib.prb_film_export_device.argtypes = [C.c_void_p, C.c_void_p]
        lib.prb_film_import_device.argtypes = [C.c_void_p, C.c_void_p]
        for n in ("prb_trace_closest", "prb_trace_closest_device"):
            getattr(lib, n).argtypes = [C.c_void_p, C.POINTER(RaySoA), C.c_size_t, C.POINTER(HitSoA)]
        for n in ("prb_trace_any", "prb_trace_any_device"):
            getattr(lib, n).argtypes = [C.c_void_p, C.POINTER(RaySoA), C.c_size_t, C.c_void_p]
        lib.prb_generate_camera_rays.argtypes = [C.c_void_p, C.POINTER(Tile), C.c_size_t, C.c_uint32, C.c_void_p, C.c_void_p,
                                                 C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        for n in ("prb_material_eval", "prb_material_sample"):
            getattr(lib, n).argtypes = [C.c_void_p, C.POINTER(MaterialQuery), C.c_size_t, C.POINTER(MaterialResult)]
        lib.prb_film_reduce.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int]
        lib.prb_comm_unique_id.argtypes = [C.c_void_p]
        lib.prb_comm_init.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        lib.prb_comm_destroy.argtypes = [C.c_void_p]
        lib.prb_film_reduce_comm.argtypes = [C.c_void_p, C.c_int, C.c_uint32, C.c_int]
        lib.prb_last_reduce_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        lib.prb_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
        lib.prb_reset_stats.argtypes = [C.c_void_p]
        lib.prb_last_device_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        lib.prb_set_profiling.argtypes = [C.c_void_p, C.c_int]
        lib.prb_get_stage_times.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_uint64)]
        lib.prb_film_download_lpe.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
        lib.prb_film_download_aov_ext.argtypes = [C.c_void_p, C.c_void_p]
        lib.prb_set_shading_mode.argtypes = [C.c_void_p, C.c_int]
        lib.prb_get_shading_mode.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
        lib.prb_set_integrator.argtypes = [C.c_void_p, C.POINTER(Integrator)]
        lib.prb_get_integrator.argtypes = [C.c_void_p, C.POINTER(Integrator)]
        _dev = lib
    return _dev


def host_lib():
    """libprb200_host.so (C++17 loader / plugin factories / BVH builder / render driver)."""
    global _host
    if _host is None:
        device_lib()  # dependency, resolved through RTLD_GLOBAL / rpath
        path = os.path.join(_HERE, "libprb200_host.so")
        if not os.path.exists(path):
            raise PrbError("libprb200_host.so is missing: run __graft_entry__.build()")
        lib = C.CDLL(path, mode=C.RTLD_GLOBAL)
        lib.prh_last_error.restype = C.c_char_p
        lib.prh_load_scene_file.restype = C.c_void_p
        lib.prh_load_scene_file.argtypes = [C.c_char_p]
        lib.prh_load_scene_string.restype = C.c_void_p
        lib.prh_load_scene_string.argtypes = [C.c_char_p, C.c_char_p]
        lib.prh_make_soup.restype = C.c_void_p
        lib.prh_make_soup.argtypes = [C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32]
        lib.prh_free_scene.argtypes = [C.c_void_p]
        lib.prh_scene_desc.restype = C.POINTER(SceneDesc)
        lib.prh_scene_desc.argtypes = [C.c_void_p]
        lib.prh_scene_integrator.argtypes = [C.c_void_p, C.POINTER(Integrator)]
        lib.prh_scene_bvh_seconds.restype = C.c_double
        lib.prh_scene_bvh_seconds.argtypes = [C.c_void_p]
        lib.prh_scene_radius.restype = C.c_float
        lib.prh_scene_radius.argtypes = [C.c_void_p]
        lib.prh_scene_set_spp.argtypes = [C.c_void_p, C.c_uint32]
        lib.prh_build_rng_map.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]
        lib.prh_build_tile_map.restype = C.c_uint32
        lib.prh_build_tile_map.argtypes = [C.c_uint32] * 6 + [C.POINTER(Tile), C.c_uint32]
        lib.prh_upsample_rgb.argtypes = [C.c_void_p, C.c_void_p]
        lib.prh_upsample_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32]
        lib.prh_cie_eval.restype = C.c_float
        lib.prh_cie_eval.argtypes = [C.c_int, C.c_float]
        lib.prh_random_stream.argtypes = [C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p]
        lib.prh_random_advance.restype = C.c_uint64
        lib.prh_random_advance.argtypes = [C.c_uint64, C.c_uint64]
        lib.prh_list_plugins.argtypes = [C.c_void_p, C.c_char_p, C.c_uint32]
        lib.prh_set_verbosity.argtypes = [C.c_int]
        lib.prh_lpe_match.restype = C.c_int
        lib.prh_lpe_match.argtypes = [C.c_char_p, C.c_void_p, C.c_uint32]
        lib.prh_abi_sizeof.restype = C.c_uint32
        lib.prh_abi_sizeof.argtypes = [C.c_char_p]
        lib.prh_render_context_create.restype = C.c_void_p
        lib.prh_render_context_create.argtypes = [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32]
        lib.prh_render_context_start.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]
        lib.prh_render_context_wait.argtypes = [C.c_void_p]
        lib.prh_render_context_device.restype = C.c_void_p
        lib.prh_render_context_device.argtypes = [C.c_void_p]
        lib.prh_render_context_destroy.argtypes = [C.c_void_p]
        lib.prh_render_context_join_communicator.argtypes = [C.c_void_p, C.c_void_p]
        lib.prh_render_contexts_combine.argtypes = [C.POINTER(C.c_void_p), C.c_int]
        lib.prh_render_context_save_outputs.restype = C.c_int
        lib.prh_render_context_save_outputs.argtypes = [C.c_void_p, C.c_char_p]
        _host = lib
    return _host


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


# ----------------------------------------------------------------------------- host objects
class Scene:
    """A loaded + compiled scene (SceneLoader::loadFromFile + Environment::createRenderFactory set-up)."""

    def __init__(self, handle):
        if not handle:
            raise PrbError("scene load failed: " + host_lib().prh_last_error().decode())
        self._h = handle
        self.desc = host_lib().prh_scene_desc(handle)

    @classmethod
    def from_file(cls, path):
        return cls(host_lib().prh_load_scene_file(os.fspath(path).encode()))

    @classmethod
    def from_string(cls, source, virtual_path=""):
        return cls(host_lib().prh_load_scene_string(source.encode(), virtual_path.encode()))

    @classmethod
    def soup(cls, triangles, seed=1234, film=(2048, 2048)):
        """SURVEY 8(d) C5 synthetic triangle soup."""
        return cls(host_lib().prh_make_soup(triangles, seed, film[0], film[1]))

    @property
    def settings(self):
        return self.desc.contents.settings

    @property
    def width(self):
        return int(self.settings.film_width)

    @property
    def height(self):
        return int(self.settings.film_height)

    @property
    def bvh_build_seconds(self):
        return float(host_lib().prh_scene_bvh_seconds(self._h))

    @property
    def integrator(self):
        """the Integrator record of the scene's (integrator ...) block"""
        rec = Integrator()
        if host_lib().prh_scene_integrator(self._h, C.byref(rec)) != 0:
            raise PrbError("prh_scene_integrator: " + host_lib().prh_last_error().decode())
        return rec

    def set_spp(self, spp):
        host_lib().prh_scene_set_spp(self._h, spp)

    def rng_map(self, rng_delta=None):
        """RenderRandomMap states (reference src/core/renderer/RenderRandomMap.cpp:11-28)."""
        s = self.settings
        out = np.empty(self.width * self.height, dtype=np.uint64)
        host_lib().prh_build_rng_map(s.seed, s.film_width, s.film_height, s.max_sample_count if rng_delta is None else rng_delta, _ptr(out))
        return out

    def tiles(self, rtx=8, rty=8):
        s = self.settings
        buf = (Tile * (rtx * rty))()
        n = host_lib().prh_build_tile_map(s.view_x, s.view_y, s.view_w, s.view_h, rtx, rty, buf, rtx * rty)
        return [(buf[i].sx, buf[i].sy, buf[i].ex, buf[i].ey) for i in range(n)]

    def full_tile(self):
        return [(0, 0, self.width, self.height)]

    def plugins(self):
        buf = C.create_string_buffer(8192)
        host_lib().prh_list_plugins(self._h, buf, 8192)
        return buf.value.decode()

    def close(self):
        if self._h:
            host_lib().prh_free_scene(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


PARTITION = {"tiles": 0, "samples": 1}  # PRB_PARTITION_*


def make_tiles(tiles):
    arr = (Tile * len(tiles))()
    for i, t in enumerate(tiles):
        arr[i] = Tile(*t)
    return arr


class Context:
    """One GPU context (prb_ctx).  All methods go through the C ABI."""

    def __init__(self, device=0):
        lib = device_lib()
        h = C.c_void_p()
        st = lib.prb_create(device, C.byref(h))
        if st != 0:
            raise PrbError("prb_create: " + lib.prb_last_error().decode())
        self._h = h
        self._lib = lib
        self.scene = None

    def _chk(self, st, what):
        if st != 0:
            raise PrbError(what + ": " + self._lib.prb_last_error().decode())

    def upload_scene(self, scene):
        """uploads the scene and selects the integrator of its (integrator ...) block"""
        self._chk(self._lib.prb_upload_scene(self._h, scene.desc), "prb_upload_scene")
        self.scene = scene
        rec = scene.integrator
        if rec.type != INTEGRATOR["direct"]:  # 'direct' is what prb_upload_scene leaves selected
            self._chk(self._lib.prb_set_integrator(self._h, C.byref(rec)), "prb_set_integrator")

    def set_integrator(self, integrator, sample_count=0, mode="colored_entity_id"):
        """integrator: "direct" / "ao" / "visualfeedback" or a PRB_INTEGRATOR_* value; sample_count: occlusion rays per sample
        ('ao'); mode: a VF_MODES name or PRB_VF_* value ('visualfeedback')"""
        t = INTEGRATOR[integrator] if isinstance(integrator, str) else int(integrator)
        rec = Integrator(t, int(sample_count))
        if t == INTEGRATOR["visualfeedback"]:
            rec.mode = VF_MODES[mode] if isinstance(mode, str) else int(mode)
        self._chk(self._lib.prb_set_integrator(self._h, C.byref(rec)), "prb_set_integrator")

    @property
    def integrator(self):
        """(type, sample_count or mode) of the integrator prb_render_tiles runs"""
        rec = Integrator()
        self._chk(self._lib.prb_get_integrator(self._h, C.byref(rec)), "prb_get_integrator")
        return int(rec.type), int(rec.sample_count)

    def upload_rng(self, states):
        states = np.ascontiguousarray(states, dtype=np.uint64)
        self._chk(self._lib.prb_upload_rng(self._h, _ptr(states), states.size), "prb_upload_rng")

    def download_rng(self):
        out = np.empty(self.scene.width * self.scene.height, dtype=np.uint64)
        self._chk(self._lib.prb_download_rng(self._h, _ptr(out), out.size), "prb_download_rng")
        return out

    def film_clear(self):
        self._chk(self._lib.prb_film_clear(self._h), "prb_film_clear")

    def render_tiles(self, tiles, first_iteration, iteration_count):
        arr = make_tiles(tiles)
        self._chk(self._lib.prb_render_tiles(self._h, arr, len(tiles), first_iteration, iteration_count), "prb_render_tiles")

    def sync(self):
        self._chk(self._lib.prb_sync(self._h), "prb_sync")

    def film(self, out=None, count_out=None):
        w, h = self.scene.width, self.scene.height
        xyz = out if out is not None else np.empty((h, w, 3), dtype=np.float32)
        cnt = count_out if count_out is not None else np.empty((h, w), dtype=np.uint32)
        self._chk(self._lib.prb_film_download(self._h, _ptr(xyz), _ptr(cnt)), "prb_film_download")
        return xyz, cnt

    def film_aov(self):
        w, h = self.scene.width, self.scene.height
        aov = np.empty((h, w, 10), dtype=np.float32)
        self._chk(self._lib.prb_film_download_aov(self._h, _ptr(aov)), "prb_film_download_aov")
        return aov

    def film_aov_ext(self):
        """(H, W, 11) sums over the samples: tangent (3), bitangent (3), view direction (3), material id, emission id"""
        aov = np.empty((self.scene.height, self.scene.width, 11), dtype=np.float32)
        self._chk(self._lib.prb_film_download_aov_ext(self._h, _ptr(aov)), "prb_film_download_aov_ext")
        return aov

    def film_feedback(self):
        """AOV_Feedback: per pixel the OR of the PRB_FEEDBACK_* bits of rejected fragments"""
        fb = np.empty((self.scene.height, self.scene.width), dtype=np.uint32)
        self._chk(self._lib.prb_film_download_feedback(self._h, _ptr(fb)), "prb_film_download_feedback")
        return fb

    def film_variance(self):
        """(online_mean, online_variance), each (H, W, 3): AOV_OnlineMean / AOV_OnlineVariance"""
        shape = (self.scene.height, self.scene.width, 3)
        mean, var = np.empty(shape, np.float32), np.empty(shape, np.float32)
        self._chk(self._lib.prb_film_download_variance(self._h, _ptr(mean), _ptr(var)), "prb_film_download_variance")
        return mean, var

    def film_lpe(self, index):
        """(H, W, 3) XYZ film of the fragments accepted by light path expression `index` of the scene's output channels"""
        xyz = np.empty((self.scene.height, self.scene.width, 3), dtype=np.float32)
        self._chk(self._lib.prb_film_download_lpe(self._h, int(index), _ptr(xyz)), "prb_film_download_lpe")
        return xyz

    def film_export_device(self, device_ptr):
        self._chk(self._lib.prb_film_export_device(self._h, C.c_void_p(device_ptr)), "prb_film_export_device")

    def film_import_device(self, device_ptr):
        self._chk(self._lib.prb_film_import_device(self._h, C.c_void_p(device_ptr)), "prb_film_import_device")

    # ---- multi-GPU film combine (include/prb200_abi.h: prb_comm_*, prb_film_reduce*)
    @staticmethod
    def comm_unique_id():
        """128 bytes created by rank 0 (ncclGetUniqueId); ship them to the other ranks out of band"""
        lib = device_lib()
        buf = np.zeros(128, np.uint8)
        if lib.prb_comm_unique_id(_ptr(buf)) != 0:
            raise PrbError("prb_comm_unique_id: " + lib.prb_last_error().decode())
        return buf

    def comm_init(self, unique_id, rank, world):
        uid = np.ascontiguousarray(unique_id, dtype=np.uint8)
        assert uid.size == 128
        self._chk(self._lib.prb_comm_init(self._h, _ptr(uid), rank, world), "prb_comm_init")

    def comm_destroy(self):
        self._chk(self._lib.prb_comm_destroy(self._h), "prb_comm_destroy")

    def film_reduce_comm(self, partition, total_iterations, root=0):
        """collective over the communicator: the root context ends up with the combined film"""
        self._chk(self._lib.prb_film_reduce_comm(self._h, PARTITION[partition], total_iterations, root), "prb_film_reduce_comm")

    @staticmethod
    def film_reduce(contexts, partition):
        """single process, several contexts: contexts[0] ends up with the combined film (prb_film_reduce)"""
        arr = (C.c_void_p * len(contexts))(*[c._h for c in contexts])
        lib = device_lib()
        if lib.prb_film_reduce(arr, len(contexts), PARTITION[partition]) != 0:
            raise PrbError("prb_film_reduce: " + lib.prb_last_error().decode())

    def last_reduce_ms(self):
        ms = C.c_float()
        self._chk(self._lib.prb_last_reduce_ms(self._h, C.byref(ms)), "prb_last_reduce_ms")
        return float(ms.value)

    @staticmethod
    def _ray_soa(o, d, tmin, tmax, keep):
        cols = [np.ascontiguousarray(o[:, i], dtype=np.float32) for i in range(3)] + \
               [np.ascontiguousarray(d[:, i], dtype=np.float32) for i in range(3)]
        cols.append(None if tmin is None else np.ascontiguousarray(tmin, dtype=np.float32))
        cols.append(None if tmax is None else np.ascontiguousarray(tmax, dtype=np.float32))
        keep.extend(cols)
        return RaySoA(*[None if c is None else c.ctypes.data for c in cols])

    def trace_closest(self, origins, dirs, tmin=None, tmax=None):
        """Scene::traceRays over host arrays -> (entity, prim, u, v, t)."""
        n = len(origins)
        keep = []
        rays = self._ray_soa(np.asarray(origins), np.asarray(dirs), tmin, tmax, keep)
        ent = np.empty(n, np.uint32); prim = np.empty(n, np.uint32)
        u = np.empty(n, np.float32); v = np.empty(n, np.float32); t = np.empty(n, np.float32)
        hits = HitSoA(ent.ctypes.data, prim.ctypes.data, u.ctypes.data, v.ctypes.data, t.ctypes.data)
        self._chk(self._lib.prb_trace_closest(self._h, C.byref(rays), n, C.byref(hits)), "prb_trace_closest")
        return ent, prim, u, v, t

    def trace_any(self, origins, dirs, tmin=None, tmax=None):
        n = len(origins)
        keep = []
        rays = self._ray_soa(np.asarray(origins), np.asarray(dirs), tmin, tmax, keep)
        occ = np.empty(n, np.uint8)
        self._chk(self._lib.prb_trace_any(self._h, C.byref(rays), n, _ptr(occ)), "prb_trace_any")
        return occ

    def trace_closest_soa(self, cols, n, out):
        """prb_trace_closest over caller-owned host COLUMNS (8 float32 arrays: origin xyz, direction xyz, tmin, tmax -- the
        last two may be None) into caller-owned result columns (entity, prim: uint32; u, v, t: float32).  No conversion and no
        allocation on the way: with page-locked arrays the copies run at PCIe speed (the way bench.py's e2e leg calls it)."""
        rays = RaySoA(*[None if c is None else c.ctypes.data for c in cols])
        hits = HitSoA(*[a.ctypes.data for a in out])
        self._chk(self._lib.prb_trace_closest(self._h, C.byref(rays), n, C.byref(hits)), "prb_trace_closest")

    def trace_any_soa(self, cols, n, occluded):
        rays = RaySoA(*[None if c is None else c.ctypes.data for c in cols])
        self._chk(self._lib.prb_trace_any(self._h, C.byref(rays), n, _ptr(occluded)), "prb_trace_any")

    def trace_closest_device(self, ray_ptrs, n, hit_ptrs):
        rays = RaySoA(*ray_ptrs)
        hits = HitSoA(*hit_ptrs)
        self._chk(self._lib.prb_trace_closest_device(self._h, C.byref(rays), n, C.byref(hits)), "prb_trace_closest_device")

    def trace_any_device(self, ray_ptrs, n, occ_ptr):
        rays = RaySoA(*ray_ptrs)
        self._chk(self._lib.prb_trace_any_device(self._h, C.byref(rays), n, C.c_void_p(occ_ptr)), "prb_trace_any_device")

    def generate_camera_rays(self, tiles, iteration):
        arr = make_tiles(tiles)
        cap = sum((t[2] - t[0]) * (t[3] - t[1]) for t in tiles)
        org = np.empty((cap, 3), np.float32); dr = np.empty((cap, 3), np.float32)
        wvl = np.empty((cap, 4), np.float32); pix = np.empty(cap, np.uint32)
        n = C.c_size_t()
        self._chk(self._lib.prb_generate_camera_rays(self._h, arr, len(tiles), iteration, _ptr(org), _ptr(dr), _ptr(wvl), _ptr(pix), cap,
                                                     C.byref(n)), "prb_generate_camera_rays")
        return org[:n.value], dr[:n.value], wvl[:n.value], pix[:n.value]

    def material_eval(self, queries):
        out = (MaterialResult * len(queries))()
        self._chk(self._lib.prb_material_eval(self._h, queries, len(queries), out), "prb_material_eval")
        return out

    def material_sample(self, queries):
        out = (MaterialResult * len(queries))()
        self._chk(self._lib.prb_material_sample(self._h, queries, len(queries), out), "prb_material_sample")
        return out

    def stats(self):
        s = Stats()
        self._chk(self._lib.prb_get_stats(self._h, C.byref(s)), "prb_get_stats")
        return s

    def reset_stats(self):
        self._chk(self._lib.prb_reset_stats(self._h), "prb_reset_stats")

    def last_device_ms(self):
        ms = C.c_float()
        self._chk(self._lib.prb_last_device_ms(self._h, C.byref(ms)), "prb_last_device_ms")
        return float(ms.value)

    def set_shading_mode(self, mode):
        """-1 measure and pick (default), 0 single k_shade, 1 staged per-material-type kernels (bit-identical films)"""
        self._chk(self._lib.prb_set_shading_mode(self._h, int(mode)), "prb_set_shading_mode")

    def shading_mode(self):
        m = C.c_int()
        self._chk(self._lib.prb_get_shading_mode(self._h, C.byref(m)), "prb_get_shading_mode")
        return int(m.value)

    def set_profiling(self, enabled):
        self._chk(self._lib.prb_set_profiling(self._h, 1 if enabled else 0), "prb_set_profiling")

    def stage_times(self):
        """{stage: (ms, launches)} accumulated since set_profiling(True)"""
        ms = (C.c_float * 2)()
        ln = (C.c_uint64 * 2)()
        self._chk(self._lib.prb_get_stage_times(self._h, ms, ln), "prb_get_stage_times")
        return {n: (float(ms[i]), int(ln[i])) for i, n in enumerate(("trace", "shade"))}

    def close(self):
        if self._h:
            self._lib.prb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def render(scene, device=0, spp=None, tiles=None, rank=0, world=1, rtx=8, rty=8):
    """Convenience: what `pearray -i scene.prc` does for the hot path on one GPU (or one rank of a multi-GPU job).

    Returns (ctx, xyz, sample_count).  Tiles are interleaved over ranks (tile_id % world == rank)."""
    ctx = Context(device)
    ctx.upload_scene(scene)
    ctx.upload_rng(scene.rng_map())
    if tiles is None:
        all_tiles = scene.tiles(rtx, rty)
        tiles = [t for i, t in enumerate(all_tiles) if i % world == rank]
    n = scene.settings.max_sample_count if spp is None else spp
    ctx.render_tiles(tiles, 0, n)
    xyz, cnt = ctx.film()
    return ctx, xyz, cnt
