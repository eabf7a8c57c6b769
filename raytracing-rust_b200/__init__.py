"""ptb200 — B200-native path-tracing backend for nonl4331/raytracing-rust (`--backend cuda`).

The directory name carries a hyphen (the repository contract), so import it through the root-level shim:
    import ptb200
"""
from . import _lib
from ._lib import (METHOD_MIS, METHOD_NAIVE, MAT_EMIT, MAT_LAMBERTIAN, MAT_REFLECT, MAT_REFRACT, MAT_TROWBRIDGE_REITZ,
                   PTB_AOV_ALBEDO, PTB_AOV_COVERAGE, PTB_AOV_DEPTH, PTB_AOV_NORMAL, PTB_MISS, TEX_CHECKERED, TEX_IMAGE, TEX_LERP, TEX_PERLIN, TEX_SOLID, PtbError, Stats, hit_dtype,
                   instance_xform_dtype, mesh_instance_dtype, mesh_triangle_dtype, occlusion_ray_dtype, ray_dtype)
from .backend import (Bvh, Context, RandomSampler, RenderOptions, Scene, denoise_opts, make_occlusion_rays, make_rays,
                      render_multi, temporal_opts)
from .multi import accumulator_tensor, reduce_accumulators, shard_samples
from .scene import HostScene, IndexedMesh, index_triangles, instance_xform, load_file, load_image, load_str, save_image
from . import meshgen

__all__ = [
    "Bvh", "Context", "RandomSampler", "RenderOptions", "Scene", "make_rays", "make_occlusion_rays", "render_multi", "HostScene",
    "IndexedMesh", "index_triangles", "instance_xform", "load_file", "load_str",
    "save_image", "load_image", "meshgen", "shard_samples", "accumulator_tensor", "reduce_accumulators", "PtbError", "Stats",
    "METHOD_MIS", "METHOD_NAIVE", "PTB_MISS", "hit_dtype", "ray_dtype", "occlusion_ray_dtype", "mesh_triangle_dtype",
    "mesh_instance_dtype", "instance_xform_dtype", "PTB_AOV_ALBEDO", "PTB_AOV_NORMAL", "PTB_AOV_DEPTH", "PTB_AOV_COVERAGE",
    "denoise_opts", "temporal_opts",
]
