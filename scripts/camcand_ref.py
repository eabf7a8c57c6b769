"""ctypes binding of scripts/camcand_ref.cpp: the CPU statement of the per-pixel camera candidate lists on the device SAH
tree's CPU definition, and the bit-for-bit check of list-answered camera rays against the ordered walk. The library is
compiled on first use into a temporary directory (the tree may be read-only)."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "camcand_ref.cpp")
_lib = None


def _load():
    global _lib
    if _lib is not None:
        return _lib
    deps = [_SRC] + [os.path.join(_HERE, "..", "oracle", f) for f in sorted(os.listdir(os.path.join(_HERE, "..", "oracle")))
                     if f.endswith(".hpp")] + [os.path.join(_HERE, "..", "include", "ptb200.h")]
    h = hashlib.sha1()
    for f in deps:
        with open(f, "rb") as fh:
            h.update(fh.read())
    out_dir = os.path.join(tempfile.gettempdir(), f"ptb200_camcand_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"libcamcand_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fno-fast-math", "-ffp-contract=off", "-fPIC",
                               "-pthread", "-shared", "-o", tmp, _SRC])
        os.replace(tmp, so)
    lib = C.CDLL(so)
    P = C.c_void_p
    lib.ccr_create.restype = P
    lib.ccr_create.argtypes = [P, C.c_size_t, P, C.c_size_t, P]
    lib.ccr_destroy.argtypes = [P]
    u32 = C.c_uint32
    lib.ccr_lists.argtypes = [P, u32, u32, u32, u32, u32, P, P, P, P, P, C.c_int]
    lib.ccr_check.argtypes = [P, u32, u32, u32, u32, u32, P, P, P, P, u32, u32, C.c_uint64, C.c_int, P, P]
    _lib = lib
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class Lists:
    """Candidate lists of the pixels of rows [row_begin, row_begin + rows): count (full candidate count; > K: overflowed),
    keys / refs / nodes (K entries per pixel, nearest key first), visits (beam-walk node expansions per pixel)."""

    def __init__(self, W, H, row_begin, rows, K, count, keys, refs, nodes, visits):
        self.W, self.H, self.row_begin, self.rows, self.K = W, H, row_begin, rows, K
        self.count, self.keys, self.refs, self.nodes, self.visits = count, keys, refs, nodes, visits

    @property
    def overflowed(self):
        return self.count > self.K


class CamCandScene:
    def __init__(self, host_scene):
        lib = _load()
        self._keep = [np.ascontiguousarray(a) for a in (host_scene.spheres, host_scene.triangles, host_scene.camera)]
        sp, tr, cam = self._keep
        self._h = lib.ccr_create(_p(sp), len(sp), _p(tr), len(tr), _p(cam))

    def __del__(self):
        if getattr(self, "_h", None):
            _lib.ccr_destroy(self._h)
            self._h = None

    def lists(self, W, H, K, row_begin=0, rows=None, threads=0) -> Lists:
        rows = H - row_begin if rows is None else rows
        n = W * rows
        count = np.zeros(n, np.uint32)
        visits = np.zeros(n, np.uint32)
        keys = np.zeros(n * K, np.float32)
        refs = np.zeros(n * K, np.uint32)
        nodes = np.zeros(n * K, np.uint32)
        _lib.ccr_lists(self._h, W, H, row_begin, rows, K, _p(count), _p(keys), _p(refs), _p(nodes), _p(visits), threads)
        return Lists(W, H, row_begin, rows, K, count, keys, refs, nodes, visits)

    def check(self, L: Lists, spp, sample_offset=0, seed=0, threads=0) -> dict:
        """Sums over the rays (see ccr_check) and, under "hist", per-list-ray histograms of entries tested, primitive
        tests and ordered-walk nodes (256 bins each, the last one open)."""
        out = np.zeros(9, np.uint64)
        hist = np.zeros((3, 256), np.uint64)
        _lib.ccr_check(self._h, L.W, L.H, L.row_begin, L.rows, L.K, _p(L.count), _p(L.keys), _p(L.refs), _p(L.nodes), spp,
                       sample_offset, seed, threads, _p(out), _p(hist))
        names = ("rays", "list_rays", "mismatches", "list_entries", "list_prim_tests", "walk_nodes", "walk_prims",
                 "box_rejected_hits", "key_above_tkey")
        r = {k: int(v) for k, v in zip(names, out)}
        r["hist"] = dict(zip(("list_entries", "list_prim_tests", "walk_nodes"), hist))
        return r
