"""ORACLE — TEST INFRASTRUCTURE ONLY.

ctypes binding of oracle/librefit_oracle.so (oracle/refit_api.cpp): the CPU statement of PTB_BUILD_REFIT. A binary tree is
built once over a host scene's primitives (the Karras LBVH of lbvh_ref.hpp, or the SAH tree of sah_ref.hpp), then
`refit(new_scene)` swaps in primitives of the same counts and recomputes every box bottom-up, topology and primitive order
kept. `export()` and `closest_hit()` describe the tree as it stands, like OracleScene.lbvh_export / lbvh_closest_hit.
Only tests/ and scripts/ import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from oracle import _p, bvh_node_dtype, hit_dtype, ray_dtype

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librefit_oracle.so")
BUILDERS = {"lbvh": 0, "sah": 1}


def _load():
    if not os.path.exists(LIB_PATH):
        subprocess.check_call(["make", "-C", os.path.dirname(_HERE), "-s", "oracle/librefit_oracle.so"])
    lib = C.CDLL(LIB_PATH)
    P = C.c_void_p
    lib.orr_create.restype = P
    lib.orr_create.argtypes = [P, C.c_size_t, P, C.c_size_t, C.c_int, C.c_int, C.c_uint32]
    lib.orr_destroy.argtypes = [P]
    lib.orr_num_nodes.restype = C.c_size_t
    lib.orr_num_nodes.argtypes = [P]
    lib.orr_refit.restype = C.c_int
    lib.orr_refit.argtypes = [P, P, C.c_size_t, P, C.c_size_t]
    lib.orr_export.argtypes = [P, P, P, P]
    lib.orr_closest_hit.argtypes = [P, P, C.c_size_t, P, C.c_int, P]
    return lib


lib = _load()


class RefitOracle:
    """A binary tree built over `host_scene` by `builder` ("lbvh" or "sah", as PTB_BUILD_BINARY / PTB_BUILD_SAH build it)."""

    def __init__(self, host_scene, builder: str = "lbvh", nbins: int = 8, max_depth: int = 60):
        sp = np.ascontiguousarray(host_scene.spheres)
        tr = np.ascontiguousarray(host_scene.triangles)
        self.n_prims = len(sp) + len(tr)
        self._h = lib.orr_create(_p(sp), len(sp), _p(tr), len(tr), BUILDERS[builder], nbins, max_depth)

    def __del__(self):
        if getattr(self, "_h", None):
            lib.orr_destroy(self._h)
            self._h = None

    def refit(self, new_scene):
        """Keep the tree, take the primitives of `new_scene` (same number in all) and refit every box."""
        sp = np.ascontiguousarray(new_scene.spheres)
        tr = np.ascontiguousarray(new_scene.triangles)
        if lib.orr_refit(self._h, _p(sp), len(sp), _p(tr), len(tr)) != 0:
            raise ValueError("a refit keeps the tree: the new scene must have as many primitives as the tree")

    def export(self):
        """(Morton codes of the build, primitive order, nodes) as ptb_bvh_export returns them."""
        m = lib.orr_num_nodes(self._h)
        morton = np.zeros(self.n_prims, np.uint32)
        prims = np.zeros(self.n_prims, np.uint32)
        nodes = np.zeros(m, bvh_node_dtype)
        lib.orr_export(self._h, _p(morton), _p(prims), _p(nodes))
        return morton, prims, nodes

    def closest_hit(self, rays, threads=0):
        """(hits, nodes_fetched, prims_tested) of the ordered, t-culled walk over the tree as it stands."""
        rays = np.ascontiguousarray(rays, dtype=ray_dtype)
        out = np.zeros(len(rays), hit_dtype)
        counts = np.zeros(2, np.uint64)
        lib.orr_closest_hit(self._h, _p(rays), len(rays), _p(out), threads, _p(counts))
        return out, int(counts[0]), int(counts[1])
