"""ctypes binding of include/b200rt.h (the C-ABI shared library libb200rt.so).

This is the Python-side "reference-facing plugin": it only marshals numpy arrays into the C ABI. There is no CPU
fallback — if the library is missing, or no CUDA device is present, the compute entry points raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200RT_LIB") or os.path.join(HERE, "libb200rt.so")     # B200RT_LIB: another build of the library (A/B comparisons)

INTEGRATOR_MEGAKERNEL = 0
INTEGRATOR_WAVEFRONT = 1
INTEGRATOR_PERSISTENT = 2
FLAG_FB_IS_ZERO = 1
FLAG_SKIP_DEAD_RAYS = 2
FLAG_DIAG_SLABS = 4
FLAG_SIMPLE_TRACE = 8
FLAG_BVH2 = 16
FLAG_ENV_ALIAS = 32
FLAG_BVH8 = 64
FLAG_TIME_KERNELS = 128
FLAG_LINEAR_TILES = 256
FLAG_TIME_INLINE = 512
FLAG_WF_PASSES_ONLY = 1024
TILE_DIM = 16
TILE_PIXELS = 256


class B200RTError(RuntimeError):
    pass


class BvhOptions(C.Structure):
    _fields_ = [("max_leaf_size", C.c_int), ("sah_bins", C.c_int), ("use_diag_slabs", C.c_int), ("num_threads", C.c_int)]


class BvhInfo(C.Structure):
    _fields_ = [("n_triangles", C.c_int), ("n_inner_nodes", C.c_int), ("n_leaves", C.c_int), ("max_leaf_size", C.c_int),
                ("max_depth", C.c_int), ("has_diag_slabs", C.c_int), ("build_seconds", C.c_double), ("sah_cost", C.c_double),
                ("n_wide_nodes", C.c_int), ("wide_max_depth", C.c_int)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class RenderOptions(C.Structure):
    _fields_ = [("integrator", C.c_int), ("flags", C.c_int), ("rank", C.c_int), ("world", C.c_int)]


class Stats(C.Structure):
    _fields_ = [("rays", C.c_ulonglong), ("samples", C.c_ulonglong), ("kernel_ms", C.c_double), ("total_ms", C.c_double),
                ("gpu_launches", C.c_int), ("h2d_bytes", C.c_ulonglong), ("d2h_bytes", C.c_ulonglong),
                ("trace_ms", C.c_double), ("shade_ms", C.c_double), ("trace_launches", C.c_int), ("shade_launches", C.c_int),
                ("trace_union_ms", C.c_double), ("tail_ms", C.c_double), ("tail_launches", C.c_int)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# every symbol include/b200rt.h declares (tests check the library exports each of them)
EXPORTS = [
    "b200rt_bvh_default_options", "b200rt_bvh_build", "b200rt_bvh_build_device", "b200rt_bvh_get_info", "b200rt_bvh_get_arrays", "b200rt_bvh_get_wide_nodes", "b200rt_bvh_check",
    "b200rt_bvh_destroy", "b200rt_scene_create", "b200rt_scene_destroy", "b200rt_scene_set_materials", "b200rt_scene_build_env_alias", "b200rt_env_alias_table",
    "b200rt_scene_get_bvh_info", "b200rt_scene_device_bytes", "b200rt_default_render_options", "b200rt_render",
    "b200rt_trace_primary", "b200rt_trace_rays", "b200rt_tiles_for_rank", "b200rt_render_tiles_device",
    "b200rt_scene_create_multi", "b200rt_scene_device_count", "b200rt_scene_get_env_alias", "b200rt_scene_get_env_cdf",
    "b200rt_accum_create", "b200rt_accum_add", "b200rt_accum_samples", "b200rt_accum_resolve", "b200rt_accum_resolve_rgba8", "b200rt_accum_destroy",
    "b200rt_denoise", "b200rt_obj_load", "b200rt_obj_get", "b200rt_obj_destroy", "b200rt_hdr_load", "b200rt_hdr_get", "b200rt_hdr_destroy", "b200rt_env_cdf_search", "b200rt_render_rgba8", "b200rt_render_region", "b200rt_rng_stream", "b200rt_host_alloc", "b200rt_host_free", "b200rt_untile_accumulate_device",
    "b200rt_untile_device", "b200rt_trace_primary_device", "b200rt_trace_rays_device", "b200rt_quantise_rgba8", "b200rt_quantise_rgba8_device", "b200rt_last_error", "b200rt_version",
    "b200rt_render_aovs", "b200rt_render_aovs_device", "b200rt_denoise_guided",
    "b200rt_scene_update_triangles", "b200rt_scene_update_triangles_device", "b200rt_scene_get_bvh_arrays",
    "b200rt_scene_rebuild_bvh", "b200rt_scene_rebuild_bvh_device",
]

_lib = None


def load_library(path: str = LIB_PATH) -> C.CDLL:
    """Loads libb200rt.so. Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(path):
        raise B200RTError(f"{path} not found: build it with `python sycl-ray-tracing_b200/build.py` "
                          "(b200rt has no CPU fallback)")
    L = C.CDLL(path)
    VP, FP, IP, I = C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int), C.c_int
    L.b200rt_last_error.restype = C.c_char_p
    L.b200rt_version.restype = C.c_char_p
    L.b200rt_bvh_default_options.argtypes = [C.POINTER(BvhOptions)]
    L.b200rt_bvh_build.argtypes = [FP, I, C.POINTER(BvhOptions), C.POINTER(VP)]
    L.b200rt_bvh_build_device.argtypes = [FP, I, I, C.POINTER(VP)]
    L.b200rt_bvh_get_info.argtypes = [VP, C.POINTER(BvhInfo)]
    L.b200rt_bvh_get_arrays.argtypes = [VP, C.POINTER(FP), C.POINTER(FP), C.POINTER(FP)]
    L.b200rt_bvh_get_wide_nodes.argtypes = [VP, C.POINTER(VP), C.POINTER(I)]
    L.b200rt_bvh_check.argtypes = [VP, FP, I]
    L.b200rt_bvh_destroy.argtypes = [VP]
    L.b200rt_bvh_destroy.restype = None
    L.b200rt_scene_create.argtypes = [FP, I, IP, I, FP, I, IP, I, VP, I, FP, I, I, FP, VP, I, C.POINTER(VP)]
    L.b200rt_scene_create_multi.argtypes = [FP, I, IP, I, FP, I, IP, I, VP, I, FP, I, I, I, FP, VP, IP, I, C.POINTER(VP)]
    L.b200rt_scene_device_count.argtypes = [VP]
    L.b200rt_scene_get_env_alias.argtypes = [VP, FP, IP, C.POINTER(C.c_double)]
    L.b200rt_scene_get_env_cdf.argtypes = [VP, FP]
    L.b200rt_render_rgba8.argtypes = [VP, FP, I, I, I, I, FP, I, C.POINTER(C.c_ubyte), C.POINTER(RenderOptions), C.POINTER(Stats)]
    L.b200rt_render_region.argtypes = [VP, FP, I, I, I, I, I, I, I, I, FP, C.POINTER(RenderOptions), C.POINTER(Stats)]
    L.b200rt_accum_create.argtypes = [VP, FP, I, I, I, I, C.POINTER(VP)]
    L.b200rt_accum_add.argtypes = [VP, I, C.POINTER(RenderOptions), C.POINTER(Stats)]
    L.b200rt_accum_samples.argtypes = [VP]
    L.b200rt_accum_resolve.argtypes = [VP, FP, FP]
    L.b200rt_accum_resolve_rgba8.argtypes = [VP, FP, I, C.POINTER(C.c_ubyte)]
    L.b200rt_accum_destroy.argtypes = [VP]
    L.b200rt_accum_destroy.restype = None
    L.b200rt_denoise.argtypes = [FP, I, I, I, C.c_float, I, C.c_float, FP]
    L.b200rt_denoise_guided.argtypes = [FP, I, FP, FP, I, I, C.c_float, I, C.c_float, FP]
    L.b200rt_obj_load.argtypes = [C.c_char_p, C.POINTER(VP)]
    L.b200rt_obj_get.argtypes = [VP, C.POINTER(FP), IP, C.POINTER(IP), C.POINTER(FP), IP, C.POINTER(IP), IP]
    L.b200rt_obj_destroy.argtypes = [VP]
    L.b200rt_obj_destroy.restype = None
    L.b200rt_hdr_load.argtypes = [C.c_char_p, I, C.POINTER(VP)]
    L.b200rt_hdr_get.argtypes = [VP, C.POINTER(FP), IP, IP]
    L.b200rt_hdr_destroy.argtypes = [VP]
    L.b200rt_hdr_destroy.restype = None
    L.b200rt_env_cdf_search.argtypes = [VP, FP, I, I, IP]
    L.b200rt_rng_stream.argtypes = [I, I, I, I, C.POINTER(C.c_uint32), FP]
    L.b200rt_host_alloc.argtypes = [C.c_size_t, C.POINTER(VP)]
    L.b200rt_host_free.argtypes = [VP]
    L.b200rt_host_free.restype = None
    L.b200rt_untile_accumulate_device.argtypes = [VP, VP, I, I, I, I, VP, VP]
    L.b200rt_scene_destroy.argtypes = [VP]
    L.b200rt_scene_destroy.restype = None
    L.b200rt_scene_set_materials.argtypes = [VP, FP, I]
    L.b200rt_scene_update_triangles.argtypes = [VP, FP, I, C.POINTER(Stats)]
    L.b200rt_scene_update_triangles_device.argtypes = [VP, VP, I, VP, C.POINTER(Stats)]
    L.b200rt_scene_rebuild_bvh.argtypes = [VP, FP, I, C.POINTER(Stats)]
    L.b200rt_scene_rebuild_bvh_device.argtypes = [VP, VP, I, VP, C.POINTER(Stats)]
    L.b200rt_scene_get_bvh_arrays.argtypes = [VP, I, VP, FP, FP, FP]
    L.b200rt_scene_build_env_alias.argtypes = [VP]
    L.b200rt_env_alias_table.argtypes = [FP, I, I, FP, C.POINTER(C.c_int), C.POINTER(C.c_double)]
    L.b200rt_quantise_rgba8.argtypes = [FP, I, I, I, C.POINTER(C.c_ubyte)]
    L.b200rt_quantise_rgba8_device.argtypes = [VP, I, I, I, VP, VP]
    L.b200rt_scene_get_bvh_info.argtypes = [VP, C.POINTER(BvhInfo)]
    L.b200rt_scene_device_bytes.argtypes = [VP]
    L.b200rt_scene_device_bytes.restype = C.c_size_t
    L.b200rt_default_render_options.argtypes = [C.POINTER(RenderOptions)]
    L.b200rt_render.argtypes = [VP, FP, I, I, I, I, FP, C.POINTER(RenderOptions), C.POINTER(Stats)]
    L.b200rt_trace_primary.argtypes = [VP, FP, I, I, I, I, IP, FP, C.POINTER(RenderOptions), C.POINTER(Stats)]
    L.b200rt_trace_rays.argtypes = [VP, FP, I, I, IP, FP, FP, C.POINTER(RenderOptions)]
    L.b200rt_tiles_for_rank.argtypes = [I, I, I, I]
    L.b200rt_render_tiles_device.argtypes = [VP, FP, I, I, I, I, VP, C.POINTER(RenderOptions), VP, C.POINTER(Stats)]
    L.b200rt_untile_device.argtypes = [VP, VP, I, I, I, I, VP, VP]
    L.b200rt_trace_primary_device.argtypes = [VP, FP, I, I, I, I, VP, VP, C.POINTER(RenderOptions), VP, C.POINTER(Stats)]
    L.b200rt_render_aovs.argtypes = [VP, FP, I, I, I, FP, FP, C.POINTER(RenderOptions), C.POINTER(Stats)]
    L.b200rt_render_aovs_device.argtypes = [VP, FP, I, I, I, VP, VP, C.POINTER(RenderOptions), VP, C.POINTER(Stats)]
    L.b200rt_trace_rays_device.argtypes = [VP, VP, I, I, VP, VP, VP, C.POINTER(RenderOptions), VP, C.POINTER(Stats)]
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != 0:
        raise B200RTError(f"b200rt error {rc}: {load_library().b200rt_last_error().decode()}")


def fptr(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_float))


def iptr(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_int))


def tiles_for_rank(w: int, h: int, rank: int, world: int) -> int:
    return int(load_library().b200rt_tiles_for_rank(w, h, rank, world))
