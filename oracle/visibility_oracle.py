"""ORACLE — TEST INFRASTRUCTURE ONLY.

ctypes binding of oracle/libvisibility_oracle.so (oracle/visibility_api.cpp): the reference's check_hit_index
(acceleration/mod.rs:226-263) and its blocker scan as an occlusion query, for a batch of rays, over the reference's own
SAH tree with BFS candidates — and the occlusion query by brute force over every primitive. Only tests/ import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from oracle import SPLIT_SAH, _p, hit_dtype, ray_dtype

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvisibility_oracle.so")
MISS = 0xFFFFFFFF

occlusion_ray_dtype = np.dtype([("o", "<f4", 3), ("tmax", "<f4"), ("d", "<f4", 3), ("exclude", "<u4")])


def _load():
    if not os.path.exists(LIB_PATH):
        subprocess.check_call(["make", "-C", os.path.dirname(_HERE), "-s", "oracle/libvisibility_oracle.so"])
    lib = C.CDLL(LIB_PATH)
    P = C.c_void_p
    lib.orv_scene_create.restype = P
    lib.orv_scene_create.argtypes = [P, C.c_size_t, P, C.c_size_t, C.c_int]
    lib.orv_scene_destroy.argtypes = [P]
    lib.orv_check_hit_index.argtypes = [P, P, P, C.c_size_t, P, C.c_int]
    lib.orv_occluded.argtypes = [P, P, C.c_size_t, P, C.c_int, C.c_int]
    return lib


lib = _load()


class VisibilityOracle:
    """The primitives of a host scene in the reference's SAH tree; ids are original (loader-order) primitive ids."""

    def __init__(self, host_scene, split_type: int = SPLIT_SAH):
        self._keep = [np.ascontiguousarray(host_scene.spheres), np.ascontiguousarray(host_scene.triangles)]
        sp, tr = self._keep
        self.n_prims = len(sp) + len(tr)
        self._h = lib.orv_scene_create(_p(sp), len(sp), _p(tr), len(tr), split_type)

    def __del__(self):
        if getattr(self, "_h", None):
            lib.orv_scene_destroy(self._h)
            self._h = None

    def check_hit_index(self, rays, index, threads=0):
        """Per ray towards original primitive id index[i]: its hit record when it is the first thing the ray hits,
        {0, PTB_MISS, 0, 0} when it is blocked, missed or out of range."""
        rays = np.ascontiguousarray(rays, dtype=ray_dtype)
        index = np.ascontiguousarray(index, dtype=np.uint32)
        assert index.shape == (len(rays),)
        out = np.zeros(len(rays), hit_dtype)
        lib.orv_check_hit_index(self._h, _p(rays), _p(index), len(rays), _p(out), threads)
        return out

    def occluded(self, rays, brute=False, threads=0):
        """bool per occlusion ray: a primitive other than `exclude` at 0 < t < tmax (BFS candidates, or every primitive)."""
        rays = np.ascontiguousarray(rays, dtype=occlusion_ray_dtype)
        out = np.zeros(len(rays), np.uint8)
        lib.orv_occluded(self._h, _p(rays), len(rays), _p(out), 1 if brute else 0, threads)
        return out.view(bool)
