"""ctypes binding of include/ptb200.h (libptb200.so).

The library is the product: there is no Python or CPU fallback. The shared object is mapped on the FIRST use of any
entry point (`lib.<symbol>`), not at import: `bench.py --impl reference` imports this package only for the numpy scene
generators and must provably not map the CUDA library. If the shared object is missing that first use fails loudly
with the build command; if no CUDA device is present `ptb_create` fails with PTB_ERR_CUDA and `Context()` raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PTB200_LIB") or os.path.join(_HERE, "libptb200.so")  # PTB200_LIB: tuning builds only

PTB_OK = 0
ERR_NAMES = {
    1: "PTB_ERR_INVALID", 2: "PTB_ERR_CUDA", 3: "PTB_ERR_OOM", 4: "PTB_ERR_PARSE", 5: "PTB_ERR_IO",
    6: "PTB_ERR_MISSING", 7: "PTB_ERR_ABORTED", 8: "PTB_ERR_UNSUPPORTED",
}
PTB_MISS = 0xFFFFFFFF
PTB_LEAF_BIT = 0x80000000
PTB_RR_DEFAULT = 0xFFFFFFFF
MAT_EMIT, MAT_LAMBERTIAN, MAT_TROWBRIDGE_REITZ, MAT_REFLECT, MAT_REFRACT = range(5)
TEX_CHECKERED, TEX_SOLID, TEX_IMAGE, TEX_LERP, TEX_PERLIN = range(5)
METHOD_NAIVE, METHOD_MIS = 0, 1
PERLIN_TABLE_WORDS = 1024
OPT_TIME_KERNELS, OPT_COUNT_TRAVERSAL = 1, 2
BUILD_DEFAULT, BUILD_BINARY, BUILD_WIDE, BUILD_SAH, BUILD_REFIT = 0, 1, 2, 4, 8
PTB_AOV_ALBEDO, PTB_AOV_NORMAL, PTB_AOV_DEPTH, PTB_AOV_COVERAGE = range(4)

# numpy mirrors of the POD structs (sizes asserted against the header's layout in tests/test_abi.py)
sphere_dtype = np.dtype([("center", "<f4", 3), ("radius", "<f4"), ("material", "<u4")])
triangle_dtype = np.dtype([("p", "<f4", (3, 3)), ("n", "<f4", (3, 3)), ("material", "<u4")])
mesh_triangle_dtype = np.dtype([("p", "<u4", 3), ("n", "<u4", 3), ("material", "<u4")])  # indices into vertices / normals
mesh_instance_dtype = np.dtype([("first_triangle", "<u4"), ("n_triangles", "<u4"), ("material", "<u4")])
instance_xform_dtype = np.dtype([("m", "<f4", (3, 4)), ("n", "<f4", (3, 3))])  # row-major object-to-world, normal matrix
material_dtype = np.dtype([("kind", "<u4"), ("texture", "<u4"), ("param", "<f4"), ("ior", "<f4", 3), ("metallic", "<f4")])
texture_dtype = np.dtype([("kind", "<u4"), ("a", "<f4", 3), ("b", "<f4", 3)])
camera_dtype = np.dtype([("origin", "<f4", 3), ("lower_left", "<f4", 3), ("horizontal", "<f4", 3), ("vertical", "<f4", 3)])
sky_dtype = np.dtype([("texture", "<u4"), ("sampler_res_x", "<u4"), ("sampler_res_y", "<u4")])
ray_dtype = np.dtype([("o", "<f4", 3), ("_pad0", "<f4"), ("d", "<f4", 3), ("_pad1", "<f4")])
hit_dtype = np.dtype([("t", "<f4"), ("prim", "<u4"), ("u", "<f4"), ("v", "<f4")])
occlusion_ray_dtype = np.dtype([("o", "<f4", 3), ("tmax", "<f4"), ("d", "<f4", 3), ("exclude", "<u4")])
bvh_node_dtype = np.dtype([("lmin", "<f4", 3), ("lmax", "<f4", 3), ("rmin", "<f4", 3), ("rmax", "<f4", 3),
                           ("left", "<u4"), ("right", "<u4"), ("parent", "<u4"), ("_pad", "<u4")])


class RenderOpts(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("samples_per_pixel", C.c_uint32),
                ("sample_offset", C.c_uint32), ("method", C.c_uint32), ("max_depth", C.c_uint32),
                ("rr_threshold", C.c_uint32), ("flags", C.c_uint32), ("seed", C.c_uint64),
                ("row_begin", C.c_uint32), ("row_count", C.c_uint32)]


class DenoiseOpts(C.Structure):
    _fields_ = [("iterations", C.c_uint32), ("sigma_luminance", C.c_float), ("sigma_normal", C.c_float),
                ("sigma_depth", C.c_float), ("flags", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [("rays_camera", C.c_uint64), ("rays_bounce", C.c_uint64), ("rays_shadow_light", C.c_uint64),
                ("rays_shadow_sky", C.c_uint64), ("rays_reference", C.c_uint64), ("paths", C.c_uint64),
                ("wavefront_iterations", C.c_uint64), ("kernel_launches", C.c_uint64), ("nodes_fetched", C.c_uint64),
                ("prims_tested", C.c_uint64), ("rays_counted", C.c_uint64), ("trace_launches", C.c_uint64),
                ("build_ms", C.c_double), ("render_ms", C.c_double), ("ms_generate", C.c_double),
                ("ms_trace", C.c_double), ("ms_shade", C.c_double), ("ms_shadow", C.c_double), ("ms_tail", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}

    @property
    def rays_total(self):
        """Rays as this repo defines them: every BVH traversal launched (SURVEY.md §8d)."""
        return self.rays_camera + self.rays_bounce + self.rays_shadow_light + self.rays_shadow_sky


class Vec3(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float)]


SAMPLER_LAMBERTIAN, SAMPLER_TR_VNDF, SAMPLER_SKY, SAMPLER_LIGHT, SAMPLER_UNIFORM_SPHERE = range(5)


class SamplerQuery(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("alpha", C.c_float), ("normal", Vec3), ("aux", Vec3), ("light_index", C.c_uint32),
                ("seed", C.c_uint64)]


PROGRESS_FN = C.CFUNCTYPE(C.c_int32, C.c_void_p, C.c_uint64, C.c_uint64)
PASS_FN = C.CFUNCTYPE(C.c_int32, C.c_void_p, C.POINTER(C.c_float), C.c_size_t, C.c_uint64, C.c_uint64)

# every symbol include/ptb200.h declares: (name, restype, argtypes)
_P = C.c_void_p
SYMBOLS = [
    ("ptb_abi_version", C.c_uint32, []),
    ("ptb_device_count", C.c_int32, [C.POINTER(C.c_int32)]),
    ("ptb_create", C.c_int32, [C.c_int32, C.POINTER(_P)]),
    ("ptb_destroy", C.c_int32, [_P]),
    ("ptb_last_error", C.c_char_p, [_P]),
    ("ptb_set_stream", C.c_int32, [_P, _P]),
    ("ptb_synchronize", C.c_int32, [_P]),
    ("ptb_set_option", C.c_int32, [_P, C.c_uint32, C.c_uint32]),
    ("ptb_scene_set_spheres", C.c_int32, [_P, _P, C.c_size_t]),
    ("ptb_scene_set_triangles", C.c_int32, [_P, _P, C.c_size_t]),
    ("ptb_scene_set_materials", C.c_int32, [_P, _P, C.c_size_t]),
    ("ptb_scene_set_textures", C.c_int32, [_P, _P, C.c_size_t]),
    ("ptb_scene_set_texture_data", C.c_int32, [_P, C.c_uint32, C.c_uint32, C.c_uint32, _P, C.c_size_t]),
    ("ptb_scene_set_camera", C.c_int32, [_P, _P]),
    ("ptb_scene_set_sky", C.c_int32, [_P, _P]),
    ("ptb_scene_update_spheres", C.c_int32, [_P, C.c_size_t, _P, C.c_size_t]),
    ("ptb_scene_update_triangles", C.c_int32, [_P, C.c_size_t, _P, C.c_size_t]),
    ("ptb_scene_update_spheres_device", C.c_int32, [_P, C.c_size_t, _P, C.c_size_t]),
    ("ptb_scene_update_triangles_device", C.c_int32, [_P, C.c_size_t, _P, C.c_size_t]),
    ("ptb_scene_set_mesh", C.c_int32, [_P, _P, C.c_size_t, _P, C.c_size_t, _P, C.c_size_t]),
    ("ptb_scene_update_mesh_vertices", C.c_int32, [_P, C.c_size_t, _P, C.c_size_t]),
    ("ptb_scene_update_mesh_normals", C.c_int32, [_P, C.c_size_t, _P, C.c_size_t]),
    ("ptb_scene_update_mesh_triangles", C.c_int32, [_P, C.c_size_t, _P, C.c_size_t]),
    ("ptb_scene_update_mesh_vertices_device", C.c_int32, [_P, C.c_size_t, _P, C.c_size_t]),
    ("ptb_scene_update_mesh_normals_device", C.c_int32, [_P, C.c_size_t, _P, C.c_size_t]),
    ("ptb_scene_update_mesh_triangles_device", C.c_int32, [_P, C.c_size_t, _P, C.c_size_t]),
    ("ptb_scene_set_mesh_instances", C.c_int32, [_P, _P, _P, C.c_size_t]),
    ("ptb_scene_update_instance_xforms", C.c_int32, [_P, C.c_size_t, _P, C.c_size_t]),
    ("ptb_scene_update_instance_xforms_device", C.c_int32, [_P, C.c_size_t, _P, C.c_size_t]),
    ("ptb_scene_commit", C.c_int32, [_P, C.c_uint32]),
    ("ptb_bvh_sah_cost", C.c_int32, [_P, C.POINTER(C.c_double)]),
    ("ptb_bvh_info", C.c_int32, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    ("ptb_bvh_export", C.c_int32, [_P, _P, _P, _P]),
    ("ptb_bvh_export_quantised", C.c_int32, [_P, _P, _P]),
    ("ptb_bvh_wide_info", C.c_int32, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]),
    ("ptb_bvh_builder", C.c_int32, [_P, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    ("ptb_bvh_wide_export", C.c_int32, [_P, _P, _P]),
    ("ptb_closest_hit", C.c_int32, [_P, _P, C.c_size_t, _P]),
    ("ptb_closest_hit_device", C.c_int32, [_P, _P, C.c_size_t, _P]),
    ("ptb_check_hit_index", C.c_int32, [_P, _P, _P, C.c_size_t, _P]),
    ("ptb_check_hit_index_device", C.c_int32, [_P, _P, _P, C.c_size_t, _P]),
    ("ptb_occluded", C.c_int32, [_P, _P, C.c_size_t, _P]),
    ("ptb_occluded_device", C.c_int32, [_P, _P, C.c_size_t, _P]),
    ("ptb_render", C.c_int32, [_P, C.POINTER(RenderOpts), _P, _P]),
    ("ptb_render_passes", C.c_int32, [_P, C.POINTER(RenderOpts), _P, _P]),
    ("ptb_accum_clear", C.c_int32, [_P]),
    ("ptb_accum_read", C.c_int32, [_P, _P, C.c_size_t, C.c_int32]),
    ("ptb_accum_device_ptr", C.c_int32, [_P, C.POINTER(_P), C.POINTER(C.c_size_t)]),
    ("ptb_accum_set_samples", C.c_int32, [_P, C.c_uint64]),
    ("ptb_render_aov", C.c_int32, [_P, C.POINTER(RenderOpts)]),
    ("ptb_aov_clear", C.c_int32, [_P]),
    ("ptb_aov_read", C.c_int32, [_P, C.c_uint32, _P, C.c_size_t, C.c_int32]),
    ("ptb_denoise", C.c_int32, [_P, C.POINTER(DenoiseOpts), _P, C.c_size_t]),
    ("ptb_denoise_device", C.c_int32, [_P, C.POINTER(DenoiseOpts), _P]),
    ("ptb_shard_samples", None, [C.c_uint32, C.c_uint32, C.c_int32, C.c_int32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    ("ptb_shard_rows", None, [C.c_uint32, C.c_uint32, C.c_int32, C.c_int32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    ("ptb_render_multi", C.c_int32, [_P, C.c_int32, C.POINTER(RenderOpts)]),
    ("ptb_sample_only", C.c_int32, [_P, C.POINTER(SamplerQuery), C.c_size_t, _P, _P]),
    ("ptb_sampler_pdf", C.c_int32, [_P, C.POINTER(SamplerQuery), _P, C.c_size_t, _P]),
    ("ptb_stats_get", C.c_int32, [_P, C.POINTER(Stats)]),
    ("ptb_stats_reset", C.c_int32, [_P]),
    ("ptb_ssml_load_file", C.c_int32, [C.c_char_p, C.POINTER(_P)]),
    ("ptb_ssml_load_str", C.c_int32, [C.c_char_p, C.c_char_p, C.POINTER(_P)]),
    ("ptb_host_scene_free", None, [_P]),
    ("ptb_host_last_error", C.c_char_p, []),
    ("ptb_host_scene_spheres", C.c_size_t, [_P, C.POINTER(_P)]),
    ("ptb_host_scene_triangles", C.c_size_t, [_P, C.POINTER(_P)]),
    ("ptb_host_scene_materials", C.c_size_t, [_P, C.POINTER(_P)]),
    ("ptb_host_scene_textures", C.c_size_t, [_P, C.POINTER(_P)]),
    ("ptb_host_scene_texture_data", C.c_size_t, [_P, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(_P)]),
    ("ptb_host_scene_camera", C.c_int32, [_P, _P]),
    ("ptb_host_scene_sky", C.c_int32, [_P, _P]),
    ("ptb_camera_make", C.c_int32, [Vec3, Vec3, Vec3, C.c_float, C.c_float, C.c_float, C.c_float, _P]),
    ("ptb_perlin_tables", C.c_int32, [C.c_uint64, _P]),
    ("ptb_image_load", C.c_int32, [C.c_char_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(_P)]),
    ("ptb_image_free", None, [_P]),
    ("ptb_image_last_error", C.c_char_p, []),
    ("ptb_scene_upload", C.c_int32, [_P, _P]),
    ("ptb_image_save", C.c_int32, [C.c_char_p, C.c_uint32, C.c_uint32, _P, C.c_float]),
]


class PtbError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"{ERR_NAMES.get(code, code)}: {message}")
        self.code = code


def load_library(path: str = LIB_PATH) -> C.CDLL:
    if not os.path.exists(path):
        raise ImportError(
            f"{path} is missing: the CUDA extension is the product and there is no fallback. "
            "Build it with `make` at the repo root (or `python -c 'import __graft_entry__ as g; g.build()'`).")
    lib = C.CDLL(path)
    for name, restype, argtypes in SYMBOLS:
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = restype
        fn.argtypes = argtypes
    return lib


class _LazyLib:
    """`lib.ptb_xxx` maps libptb200.so on first use and checks every symbol the header declares."""

    _cdll = None

    def _load(self) -> C.CDLL:
        if _LazyLib._cdll is None:
            _LazyLib._cdll = load_library()
        return _LazyLib._cdll

    def __getattr__(self, name):
        return getattr(self._load(), name)


lib = _LazyLib()


def is_loaded() -> bool:
    return _LazyLib._cdll is not None


def ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)
