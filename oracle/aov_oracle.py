"""ORACLE — TEST INFRASTRUCTURE ONLY.

ctypes binding of oracle/libaov_oracle.so (oracle/aov_api.cpp): the denoiser feature buffers of ptb_render_aov (first-hit
albedo, normal, depth and coverage of the render's camera rays) restated over the reference's own camera, SAH tree,
materials and textures, summed in f32 in sample order. Only tests/ import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from oracle import RenderOpts, _p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libaov_oracle.so")
MISS = 0xFFFFFFFF


def _load():
    if not os.path.exists(LIB_PATH):
        subprocess.check_call(["make", "-C", os.path.dirname(_HERE), "-s", "oracle/libaov_oracle.so"])
    lib = C.CDLL(LIB_PATH)
    P = C.c_void_p
    lib.ora_scene_create.restype = P
    lib.ora_scene_create.argtypes = [P, C.c_size_t, P, C.c_size_t, P, C.c_size_t, P, C.c_size_t, P, P, P, P]
    lib.ora_scene_destroy.argtypes = [P]
    lib.ora_render_aov.argtypes = [P, C.POINTER(RenderOpts), P, P, C.c_int]
    return lib


lib = _load()


class AovOracle:
    """A host scene (primitives, materials, textures, camera, sky) in the reference's SAH tree."""

    def __init__(self, host_scene):
        s = host_scene
        self._keep = [np.ascontiguousarray(a) for a in (s.spheres, s.triangles, s.materials, s.textures, s.camera, s.sky)]
        sp, tr, ma, te, cam, sky = self._keep
        tex_ptrs = (C.c_void_p * max(len(te), 1))()
        tex_dims = np.zeros(3 * max(len(te), 1), np.uint32)
        for i, (w, h, words) in getattr(s, "texture_data", {}).items():
            words = np.ascontiguousarray(words, dtype=np.float32)
            self._keep.append(words)
            tex_ptrs[i] = words.ctypes.data
            tex_dims[3 * i:3 * i + 3] = (w, h, words.size)
        self._keep.append(tex_dims)
        self._h = lib.ora_scene_create(_p(sp), len(sp), _p(tr), len(tr), _p(ma), len(ma), _p(te), len(te), _p(cam), _p(sky),
                                       C.cast(tex_ptrs, C.c_void_p), _p(tex_dims))

    def __del__(self):
        if getattr(self, "_h", None):
            lib.ora_scene_destroy(self._h)
            self._h = None

    def render_aov(self, width, height, spp, seed=0, sample_offset=0, row_begin=0, row_count=0, sums=None, threads=0):
        """Adds the samples into `sums` ((H, W, 8) float32: albedo.rgb, coverage, normal.xyz, depth; zeros when None) and
        returns (sums, prims): prims ((rows * W, spp) uint32) is the original id of each sample's hit, MISS on a miss."""
        o = RenderOpts(width, height, spp, sample_offset, 0, 0, 0, 0, seed, row_begin, row_count)
        if sums is None:
            sums = np.zeros((height, width, 8), np.float32)
        assert sums.dtype == np.float32 and sums.shape == (height, width, 8) and sums.flags.c_contiguous
        rows = row_count or height - row_begin
        prims = np.zeros((rows * width, spp), np.uint32)
        lib.ora_render_aov(self._h, C.byref(o), _p(sums), _p(prims), threads)
        return sums, prims


def split(sums, samples):
    """The four buffers of `sums` as ptb_aov_read(normalise=1) returns them: albedo, normal and coverage over `samples`,
    depth over the coverage sum (0 where nothing was hit)."""
    cov = sums[..., 3]
    with np.errstate(divide="ignore", invalid="ignore"):
        depth = np.where(cov > 0, sums[..., 7] / np.where(cov > 0, cov, np.float32(1)), np.float32(0)).astype(np.float32)
    n = np.float32(samples)
    return dict(albedo=sums[..., 0:3] / n, normal=sums[..., 4:7] / n, depth=depth, coverage=cov / n)
