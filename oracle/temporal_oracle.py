"""ORACLE — TEST INFRASTRUCTURE ONLY.

ctypes binding of oracle/libtemporal_oracle.so (oracle/temporal_api.cpp): one step of ptb_denoise_temporal (SVGF's
temporal accumulation in front of the spatial filter) on the CPU in f32, in the device's order of operations. The step is
stateless: the caller carries the history from one frame to the next. Only tests/ import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtemporal_oracle.so")


def _load():
    if not os.path.exists(LIB_PATH):
        subprocess.check_call(["make", "-C", os.path.dirname(_HERE), "-s", "oracle/libtemporal_oracle.so"])
    lib = C.CDLL(LIB_PATH)
    P = C.c_void_p
    lib.ora_denoise_temporal.restype = C.c_int
    lib.ora_denoise_temporal.argtypes = [P, P, P, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint32, C.c_float,
                                         C.c_float, C.c_float, C.c_float, C.c_float, C.c_uint32, C.c_int, P, P, P, P, P, P,
                                         P, P, P, P, P, C.c_uint32]
    return lib


lib = _load()


def empty_history(h, w):
    return dict(e=np.zeros((h, w, 4), np.float32), m=np.zeros((h, w, 4), np.float32), nz=np.zeros((h, w, 4), np.float32),
                alpha=np.zeros((h, w), np.float32), grad=np.zeros((h, w, 2), np.float32))


def denoise_temporal(beauty_sums, aov_sums, motion_sums, beauty_samples, aov_samples, history=None, iterations=0,
                     sigma_luminance=0.0, sigma_normal=0.0, sigma_depth=0.0, alpha_color=0.0, alpha_moments=0.0,
                     max_history=0, threads=0):
    """beauty_sums (H, W, 3), aov_sums (H, W, 8), motion_sums (H, W, 4) as float32 sums; `history` is the dict a previous
    call returned (None: no history). Returns (image (H, W, 3), the next history)."""
    b = np.ascontiguousarray(beauty_sums, np.float32)
    a = np.ascontiguousarray(aov_sums, np.float32)
    m = np.ascontiguousarray(motion_sums, np.float32)
    h, w = b.shape[:2]
    assert b.shape == (h, w, 3) and a.shape == (h, w, 8) and m.shape == (h, w, 4)
    have = history is not None
    hin = history if have else empty_history(h, w)
    assert hin["e"].shape == (h, w, 4)
    hout = empty_history(h, w)
    out = np.zeros((h, w, 3), np.float32)
    P = lambda x: np.ascontiguousarray(x, np.float32).ctypes.data  # noqa: E731
    keep = {k: np.ascontiguousarray(v, np.float32) for k, v in hin.items()}
    rc = lib.ora_denoise_temporal(b.ctypes.data, a.ctypes.data, m.ctypes.data, w, h, int(beauty_samples), int(aov_samples),
                                  int(iterations), float(sigma_luminance), float(sigma_normal), float(sigma_depth),
                                  float(alpha_color), float(alpha_moments), int(max_history), 1 if have else 0,
                                  P(keep["e"]), P(keep["m"]), P(keep["nz"]), P(keep["alpha"]), P(keep["grad"]),
                                  out.ctypes.data, hout["e"].ctypes.data, hout["m"].ctypes.data, hout["nz"].ctypes.data,
                                  hout["alpha"].ctypes.data, hout["grad"].ctypes.data, int(threads))
    if rc != 0:
        raise ValueError("ora_denoise_temporal: invalid arguments")
    return out, hout
