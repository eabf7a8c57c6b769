"""ORACLE — TEST INFRASTRUCTURE ONLY.

ctypes binding of oracle/libdenoise_oracle.so (oracle/denoise_api.cpp): ptb_denoise's spatial SVGF filter restated on the
CPU in f32, in the device's order of operations, over the raw sums. Only tests/ import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdenoise_oracle.so")


def _load():
    if not os.path.exists(LIB_PATH):
        subprocess.check_call(["make", "-C", os.path.dirname(_HERE), "-s", "oracle/libdenoise_oracle.so"])
    lib = C.CDLL(LIB_PATH)
    P = C.c_void_p
    lib.ora_denoise.restype = C.c_int
    lib.ora_denoise.argtypes = [P, P, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint32, C.c_float, C.c_float,
                                C.c_float, P, C.c_uint32]
    return lib


lib = _load()


def denoise(beauty_sums, aov_sums, beauty_samples, aov_samples, iterations=0, sigma_luminance=0.0, sigma_normal=0.0,
            sigma_depth=0.0, threads=0):
    """beauty_sums (H, W, 3) and aov_sums (H, W, 8: albedo.rgb, coverage, normal.xyz, depth) as float32 sums of
    `beauty_samples` / `aov_samples` samples; 0 selects an option's default. Returns the denoised image (H, W, 3), the
    same bits for any number of threads (0: one per core)."""
    b = np.ascontiguousarray(beauty_sums, np.float32)
    a = np.ascontiguousarray(aov_sums, np.float32)
    h, w = b.shape[:2]
    assert b.shape == (h, w, 3) and a.shape == (h, w, 8)
    out = np.zeros((h, w, 3), np.float32)
    rc = lib.ora_denoise(b.ctypes.data, a.ctypes.data, w, h, int(beauty_samples), int(aov_samples), int(iterations),
                         float(sigma_luminance), float(sigma_normal), float(sigma_depth), out.ctypes.data, int(threads))
    if rc != 0:
        raise ValueError("ora_denoise: invalid arguments")
    return out
