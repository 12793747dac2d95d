"""sycl-ray-tracing_b200 — B200-native (sm_100a CUDA) implementation of the per-pixel path-tracing hot path of
TomClabault/SYCL-ray-tracing behind the reference's RenderKernel / Camera / Image / SimpleMaterial / FlattenedBVH API.

Import as `sycl_ray_tracing_b200` (see sycl_ray_tracing_b200.py at the repo root: the directory name carries a hyphen).
"""
from . import binding
from .api import (Accumulator, BVH, OIDN_denoise, Camera, FlattenedBVH, Identity, Image, RenderKernel, RotationX, RotationY, Scene, SimpleMaterial,
                  Translation, compute_env_map_cdf, constant_env, materials_to_array, quantise_rgba8, env_alias_table,
                  pinned_array, rng_stream, parse_obj, read_image_float)
from .binding import (B200RTError, FLAG_SIMPLE_TRACE, FLAG_BVH2, FLAG_ENV_ALIAS, FLAG_BVH8, FLAG_TIME_KERNELS, FLAG_LINEAR_TILES, FLAG_TIME_INLINE, FLAG_WF_PASSES_ONLY, FLAG_DIAG_SLABS, FLAG_FB_IS_ZERO, FLAG_SKIP_DEAD_RAYS, INTEGRATOR_MEGAKERNEL, INTEGRATOR_PERSISTENT,
                      INTEGRATOR_WAVEFRONT, load_library, tiles_for_rank)

__all__ = ["Accumulator", "BVH", "OIDN_denoise", "Camera", "FlattenedBVH", "Identity", "Image", "RenderKernel", "RotationX", "RotationY", "Scene",
           "SimpleMaterial", "Translation", "compute_env_map_cdf", "constant_env", "materials_to_array", "quantise_rgba8", "env_alias_table", "pinned_array", "rng_stream", "parse_obj", "read_image_float", "B200RTError",
           "load_library", "tiles_for_rank", "binding"]
