"""ORACLE — TEST INFRASTRUCTURE ONLY.

ctypes binding of oracle/libmotion_oracle.so (oracle/motion_api.cpp): the motion vectors ptb_render_aov adds after
ptb_motion_mark, restated over the AOV oracle's scene (the reference's camera and SAH tree) with the marked primitives and
camera as extra inputs, summed in f32 in sample order. Only tests/ import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from oracle import RenderOpts, _p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmotion_oracle.so")


def _load():
    if not os.path.exists(LIB_PATH):
        subprocess.check_call(["make", "-C", os.path.dirname(_HERE), "-s", "oracle/libmotion_oracle.so"])
    lib = C.CDLL(LIB_PATH)
    P = C.c_void_p
    lib.ora_scene_create.restype = P
    lib.ora_scene_create.argtypes = [P, C.c_size_t, P, C.c_size_t, P, C.c_size_t, P, C.c_size_t, P, P, P, P]
    lib.ora_scene_destroy.argtypes = [P]
    lib.ora_render_motion.argtypes = [P, C.POINTER(RenderOpts), P, P, P, P, C.c_int]
    return lib


lib = _load()


class MotionOracle:
    """The committed frame: a host scene (primitives, materials, textures, camera, sky) in the reference's SAH tree."""

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
        self.n_spheres, self.n_tris = len(sp), len(tr)
        self._h = lib.ora_scene_create(_p(sp), len(sp), _p(tr), len(tr), _p(ma), len(ma), _p(te), len(te), _p(cam), _p(sky),
                                       C.cast(tex_ptrs, C.c_void_p), _p(tex_dims))

    def __del__(self):
        if getattr(self, "_h", None):
            lib.ora_scene_destroy(self._h)
            self._h = None

    def render_motion(self, prev_scene, width, height, spp, seed=0, sample_offset=0, row_begin=0, row_count=0, sums=None,
                      threads=0):
        """Adds the motion of the samples into `sums` ((H, W, 4) float32: Σ Δx, Σ Δy, Σ t', valid count; zeros when None)
        against the marked frame `prev_scene` (its spheres, triangles and camera; the counts must equal this scene's)."""
        ps = np.ascontiguousarray(prev_scene.spheres)
        pt = np.ascontiguousarray(prev_scene.triangles)
        pc = np.ascontiguousarray(prev_scene.camera)
        assert len(ps) == self.n_spheres and len(pt) == self.n_tris
        o = RenderOpts(width, height, spp, sample_offset, 0, 0, 0, 0, seed, row_begin, row_count)
        if sums is None:
            sums = np.zeros((height, width, 4), np.float32)
        assert sums.dtype == np.float32 and sums.shape == (height, width, 4) and sums.flags.c_contiguous
        lib.ora_render_motion(self._h, C.byref(o), _p(sums), _p(ps), _p(pt), _p(pc), threads)
        return sums


def mean(sums):
    """The (H, W, 3) image ptb_motion_read returns: the sums over the valid count, 0 where there is none."""
    cnt = sums[..., 3:4]
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(cnt > 0, sums[..., 0:3] / np.where(cnt > 0, cnt, np.float32(1)), np.float32(0)).astype(np.float32)
