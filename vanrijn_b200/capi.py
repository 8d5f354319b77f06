"""ctypes view of the two in-tree libraries.

  libvanrijn_cuda.so  -- the C ABI of include/vanrijn_cuda.h (CUDA kernels; the product)
  libvanrijn_host.so  -- the C++ host mirror of the reference API (include/vanrijn.hpp) + C shim

There is no Python or CPU implementation of the render loop behind these calls: if the
libraries are missing, or there is no CUDA device, the calls raise.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIBDIR = os.environ.get("VRJ_LIBDIR") or os.path.join(HERE, "lib")  # VRJ_LIBDIR: kernel-variant experiments only

dp = C.POINTER(C.c_double)
u64p = C.POINTER(C.c_uint64)

MAT_LAMBERTIAN, MAT_PHONG, MAT_REFLECTIVE, MAT_DIELECTRIC = 0, 1, 2, 3
INTEGRATOR_SIMPLE_RANDOM, INTEGRATOR_WHITTED = 0, 1
FILTER_F32, FILTER_F64, FILTER_F32X4, FILTER_Q16 = 0, 1, 2, 3
MEM_HOST, MEM_DEVICE = 0, 1
PRECISION_F64, PRECISION_F32_FAST = 0, 1
TONEMAP_XYZ, TONEMAP_LINEAR_RGB = 0, 1
OK = 0

# every symbol include/vanrijn_cuda.h declares
CUDA_SYMBOLS = ["vrj_last_error", "vrj_abi_version", "vrj_device_count", "vrj_scene_create", "vrj_scene_destroy",
                "vrj_scene_device_bytes", "vrj_scene_upload_bytes", "vrj_render_tile", "vrj_trace_rays", "vrj_release_scratch", "vrj_alloc_host",
                "vrj_free_host", "vrj_alloc_device", "vrj_free_device", "vrj_copy_to_host", "vrj_comm_create", "vrj_comm_destroy", "vrj_comm_scene_create", "vrj_comm_scene_destroy",
                "vrj_render_sharded", "vrj_tone_map", "vrj_bvh_build", "vrj_render_adaptive"]


class VrjError(RuntimeError):
    pass


class Spectrum(C.Structure):
    _fields_ = [("shortest_wavelength", C.c_double), ("longest_wavelength", C.c_double),
                ("first_sample", C.c_uint32), ("n_samples", C.c_uint32)]


class Material(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("spectrum", C.c_uint32), ("p0", C.c_double), ("p1", C.c_double), ("p2", C.c_double)]


class Sphere(C.Structure):
    _fields_ = [("centre", C.c_double * 3), ("radius", C.c_double), ("material", C.c_uint32), ("pad", C.c_uint32)]


class Plane(C.Structure):
    _fields_ = [("normal", C.c_double * 3), ("tangent", C.c_double * 3), ("cotangent", C.c_double * 3),
                ("distance_from_origin", C.c_double), ("material", C.c_uint32), ("pad", C.c_uint32)]


class Bvh(C.Structure):
    _fields_ = [("first_node", C.c_uint64), ("n_nodes", C.c_uint64), ("first_triangle", C.c_uint64),
                ("n_triangles", C.c_uint64), ("depth", C.c_uint32), ("pad", C.c_uint32)]


class Item(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("index", C.c_uint32), ("object_id", C.c_uint32), ("prim_id", C.c_uint32)]


class SceneDesc(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("pad0", C.c_uint32), ("camera_location", C.c_double * 3), ("pad1", C.c_double),
                ("n_spectra", C.c_uint32), ("n_spectrum_samples", C.c_uint32),
                ("spectra", C.POINTER(Spectrum)), ("spectrum_samples", dp),
                ("n_materials", C.c_uint32), ("n_spheres", C.c_uint32),
                ("materials", C.POINTER(Material)), ("spheres", C.POINTER(Sphere)),
                ("n_planes", C.c_uint32), ("n_bvhs", C.c_uint32),
                ("planes", C.POINTER(Plane)), ("bvhs", C.POINTER(Bvh)),
                ("n_triangles", C.c_uint64),
                ("tri_v0", dp), ("tri_v1", dp), ("tri_v2", dp), ("tri_n0", dp), ("tri_n1", dp), ("tri_n2", dp),
                ("tri_material", C.POINTER(C.c_uint32)), ("tri_prim_id", C.POINTER(C.c_uint32)),
                ("n_nodes", C.c_uint64), ("node_min", dp), ("node_max", dp), ("node_child", C.POINTER(C.c_int32)),
                ("n_items", C.c_uint32), ("pad2", C.c_uint32), ("items", C.POINTER(Item))]


class Tile(C.Structure):
    _fields_ = [("start_column", C.c_uint64), ("end_column", C.c_uint64), ("start_row", C.c_uint64), ("end_row", C.c_uint64)]


class SpectrumData(C.Structure):
    _fields_ = [("shortest_wavelength", C.c_double), ("longest_wavelength", C.c_double),
                ("n_samples", C.c_uint32), ("pad", C.c_uint32), ("samples", dp)]


class Light(C.Structure):
    _fields_ = [("direction", C.c_double * 3), ("spectrum", SpectrumData)]


class RenderParams(C.Structure):
    _fields_ = [("spp", C.c_uint32), ("max_depth", C.c_uint32), ("sample_offset", C.c_uint64), ("seed", C.c_uint64),
                ("integrator", C.c_uint32), ("bvh_filter", C.c_uint32), ("bias", C.c_double),
                ("lights", C.POINTER(Light)), ("ambient_light", C.POINTER(SpectrumData)), ("n_lights", C.c_uint32),
                ("sample_stride", C.c_uint32), ("count_traversal", C.c_uint32), ("precision", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("primary_rays", "bounce_rays", "shadow_rays", "paths_missed", "paths_escaped",
                                          "paths_depth_limited", "node_visits", "triangle_tests", "kernel_launches")] + \
               [("device_ms", C.c_double), ("primary_ms", C.c_double), ("bounce_ms", C.c_double), ("resolve_ms", C.c_double),
                ("primary_launches", C.c_uint64), ("bounce_launches", C.c_uint64), ("resolve_launches", C.c_uint64),
                ("shade_ms", C.c_double), ("shade_launches", C.c_uint64), ("staged_rays", C.c_uint64),
                ("tail_ms", C.c_double), ("tail_launches", C.c_uint64), ("coalesced_calls", C.c_uint64)]

    @property
    def rays(self):
        return int(self.primary_rays + self.bounce_rays + self.shadow_rays)

    def as_dict(self):
        return {n: (float(getattr(self, n)) if t is C.c_double else int(getattr(self, n))) for n, t in self._fields_}


class BvhBuildStats(C.Structure):
    _fields_ = [("device_ms", C.c_double), ("global_levels", C.c_uint32), ("radix_passes", C.c_uint32),
                ("small_subtrees", C.c_uint32), ("pad", C.c_uint32)]


class AccumOut(C.Structure):
    _fields_ = [("memory", C.c_uint32), ("accumulate", C.c_uint32), ("colour", C.c_void_p), ("colour_sum", C.c_void_p),
                ("colour_bias", C.c_void_p), ("weight", C.c_void_p), ("weight_bias", C.c_void_p), ("photons", C.c_void_p),
                ("stats", C.POINTER(Stats)), ("srgb8", C.c_void_p)]


class AdaptiveParams(C.Structure):
    _fields_ = [("min_samples", C.c_uint32), ("max_samples", C.c_uint32), ("pass_samples", C.c_uint32), ("pad", C.c_uint32),
                ("rel_error", C.c_double), ("abs_floor", C.c_double)]


class AdaptiveStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("passes", "samples", "pixels_converged", "pixels_unconverged")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


_cuda = None
_host = None


def _load(name):
    path = os.path.join(LIBDIR, name)
    if not os.path.exists(path):
        raise VrjError("%s is not built: run `python -c 'import __graft_entry__ as g; g.build()'` or `make` "
                       "(the render loop has no Python/CPU fallback)" % path)
    return C.CDLL(path, mode=C.RTLD_GLOBAL)


def cuda():
    """libvanrijn_cuda.so with argument types declared."""
    global _cuda
    if _cuda is None:
        L = _load("libvanrijn_cuda.so")
        L.vrj_last_error.restype = C.c_char_p
        L.vrj_abi_version.restype = C.c_int32
        L.vrj_device_count.restype = C.c_int32
        L.vrj_scene_create.restype = C.c_int32
        L.vrj_scene_create.argtypes = [C.POINTER(SceneDesc), C.c_int32, C.POINTER(C.c_void_p)]
        L.vrj_scene_destroy.argtypes = [C.c_void_p]
        L.vrj_scene_device_bytes.restype = C.c_uint64
        L.vrj_scene_device_bytes.argtypes = [C.c_void_p]
        L.vrj_scene_upload_bytes.restype = C.c_uint64
        L.vrj_scene_upload_bytes.argtypes = [C.c_void_p]
        L.vrj_alloc_host.restype = C.c_void_p
        L.vrj_alloc_host.argtypes = [C.c_uint64]
        L.vrj_free_host.argtypes = [C.c_void_p]
        L.vrj_alloc_device.restype = C.c_void_p
        L.vrj_alloc_device.argtypes = [C.c_int32, C.c_uint64]
        L.vrj_free_device.argtypes = [C.c_void_p]
        L.vrj_copy_to_host.restype = C.c_int32
        L.vrj_copy_to_host.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_uint64]
        L.vrj_render_tile.restype = C.c_int32
        L.vrj_render_tile.argtypes = [C.c_void_p, C.POINTER(Tile), C.c_uint64, C.c_uint64, C.POINTER(RenderParams),
                                      C.POINTER(AccumOut)]
        L.vrj_render_adaptive.restype = C.c_int32
        L.vrj_render_adaptive.argtypes = [C.c_void_p, C.POINTER(Tile), C.c_uint64, C.c_uint64, C.POINTER(RenderParams),
                                          C.POINTER(AdaptiveParams), C.POINTER(AccumOut), C.c_void_p, C.POINTER(AdaptiveStats)]
        L.vrj_comm_create.restype = C.c_int32
        L.vrj_comm_create.argtypes = [C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_void_p)]
        L.vrj_comm_destroy.argtypes = [C.c_void_p]
        L.vrj_comm_scene_create.restype = C.c_int32
        L.vrj_comm_scene_create.argtypes = [C.c_void_p, C.POINTER(SceneDesc), C.POINTER(C.c_void_p)]
        L.vrj_comm_scene_destroy.argtypes = [C.c_void_p]
        L.vrj_render_sharded.restype = C.c_int32
        L.vrj_render_sharded.argtypes = [C.c_void_p, C.POINTER(Tile), C.c_uint64, C.c_uint64, C.POINTER(RenderParams),
                                         C.POINTER(AccumOut)]
        L.vrj_tone_map.restype = C.c_int32
        L.vrj_tone_map.argtypes = [C.c_int32, C.c_uint32, C.c_uint32, dp, C.c_uint64, C.c_void_p]
        L.vrj_bvh_build.restype = C.c_int32
        L.vrj_bvh_build.argtypes = [C.c_int32, C.c_uint64, dp, C.POINTER(C.c_uint32), dp, dp, C.POINTER(C.c_int32),
                                    C.POINTER(C.c_uint32), C.POINTER(BvhBuildStats)]
        L.vrj_trace_rays.restype = C.c_int32
        L.vrj_trace_rays.argtypes = [C.c_void_p, C.c_uint64, dp, dp, C.c_uint32, C.POINTER(C.c_int32),
                                     C.POINTER(C.c_int32), dp, C.POINTER(Stats)]
        _cuda = L
    return _cuda


def host():
    """libvanrijn_host.so (C shim over include/vanrijn.hpp) with argument types declared."""
    global _host
    if _host is None:
        cuda()  # dependency, loaded RTLD_GLOBAL first
        L = _load("libvanrijn_host.so")
        L.vrjh_last_error.restype = C.c_char_p
        L.vrjh_scene_new.restype = C.c_void_p
        L.vrjh_scene_new.argtypes = [C.c_double] * 3
        L.vrjh_scene_free.argtypes = [C.c_void_p]
        L.vrjh_add_spectrum.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_int, dp]
        L.vrjh_add_spectrum_rgb.argtypes = [C.c_void_p] + [C.c_double] * 3
        L.vrjh_add_spectrum_grey.argtypes = [C.c_void_p, C.c_double]
        L.vrjh_add_spectrum_diamond.argtypes = [C.c_void_p]
        L.vrjh_get_spectrum.argtypes = [C.c_void_p, C.c_int, dp, dp, dp, C.c_int]
        L.vrjh_add_material.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_double] * 3
        L.vrjh_begin_list.argtypes = [C.c_void_p]
        L.vrjh_list_add_sphere.argtypes = [C.c_void_p] + [C.c_double] * 4 + [C.c_int]
        L.vrjh_list_add_plane.argtypes = [C.c_void_p] + [C.c_double] * 4 + [C.c_int]
        L.vrjh_list_add_triangle.argtypes = [C.c_void_p, dp, dp, C.c_int]
        L.vrjh_add_bvh.argtypes = [C.c_void_p, C.c_int64, dp, dp, C.c_int, C.c_int]
        L.vrjh_add_bvh_obj.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int]
        L.vrjh_load_obj.restype = C.c_int64
        L.vrjh_load_obj.argtypes = [C.c_char_p, dp, dp, C.c_int64]
        L.vrjh_flatten.restype = C.POINTER(SceneDesc)
        L.vrjh_flatten.argtypes = [C.c_void_p]
        L.vrjh_device_scene.restype = C.c_void_p
        L.vrjh_device_scene.argtypes = [C.c_void_p, C.c_int]
        L.vrjh_partial_render_scene.argtypes = [C.c_void_p, u64p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64,
                                                dp, dp, dp, dp, dp]
        if hasattr(L, "vrjh_next_sample_index"):  # absent only from older kernel-variant builds (VRJ_LIBDIR experiments)
            L.vrjh_next_sample_index.restype = C.c_uint64
            L.vrjh_next_sample_index.argtypes = [C.c_uint64]
        if hasattr(L, "vrjh_render_like_main"):
            L.vrjh_render_like_main.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32,
                                                C.c_uint32, C.c_uint64, C.c_uint64, C.c_int, C.c_int, dp, dp, dp]
        L.vrjh_merge_tile.argtypes = [dp, dp, C.c_uint64, C.c_uint64, u64p, dp, dp]
        if hasattr(L, "vrjh_merge_tiles"):
            L.vrjh_merge_tiles.argtypes = [dp, dp, C.c_uint64, C.c_uint64, u64p, C.c_uint32, dp, dp, C.c_double]
        L.vrjh_scene_save_cache.argtypes = [C.c_void_p, C.c_char_p]
        L.vrjh_scene_load_cache.restype = C.c_void_p
        L.vrjh_scene_load_cache.argtypes = [C.c_char_p]
        L.vrjh_write_png.argtypes = [C.c_char_p, C.c_uint64, C.c_uint64, C.c_void_p]
        L.vrjh_tile_iterator.restype = C.c_int64
        L.vrjh_tile_iterator.argtypes = [C.c_uint64] * 3 + [u64p, C.c_int64]
        _host = L
    return _host


def check(status):
    if status != OK:
        raise VrjError("vanrijn_cuda status %d: %s" % (status, cuda().vrj_last_error().decode()))
