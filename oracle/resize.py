"""Oracle for the bilinear resize of predicted depth (TEST INFRASTRUCTURE).

Restates ``cv2.resize(depth, (W, H), interpolation=cv2.INTER_LINEAR)`` of ``edge.py:76-78`` (the resize of a
prediction to the GT size in front of Canny) for float32 planes with at least two rows and two columns, in
oracle/csrc/resize.c.  PINNED against the opencv-python 4.13.0 wheel with its IPP HAL on (the default): bit-exact on
the shape and value matrix of tests/test_resize_cpu.py.  With ``cv2.ipp.setUseIPP(False)`` OpenCV computes different
values, so what "cv2.resize" means is a property of the OpenCV build (DESIGN.md section 2).

The C file is compiled by this module into ``oracle/_build/libresize_oracle.so`` (git-ignored) on first use, with
``-ffp-contract=off`` and libm's ``fmaf``, apart from the matcher's ``liboracle.so``.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "csrc", "resize.c")
_SO = os.path.join(_HERE, "_build", "libresize_oracle.so")
_LIB = None


def build():
    """Compile csrc/resize.c when the library is missing or older than the source."""
    if os.path.exists(_SO) and os.path.getmtime(_SO) >= os.path.getmtime(_SRC):
        return _SO
    os.makedirs(os.path.dirname(_SO), exist_ok=True)
    tmp = f"{_SO}.{os.getpid()}.tmp"
    subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-Wall", "-ffp-contract=off",
                           "-o", tmp, _SRC, "-lm"])
    os.replace(tmp, _SO)
    return _SO


def _lib():
    global _LIB
    if _LIB is None:
        lib = ctypes.CDLL(build())
        lib.oracle_resize_linear_f32.restype = ctypes.c_int
        lib.oracle_resize_linear_f32.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                 ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
        _LIB = lib
    return _LIB


def resize_linear(src, size):
    """src float32 [h,w] or [N,h,w] (h, w >= 2), size (H, W) -> float32 [H,W] or [N,H,W]."""
    s = np.ascontiguousarray(src, dtype=np.float32)
    squeeze = s.ndim == 2
    if squeeze:
        s = s[None]
    if s.ndim != 3:
        raise ValueError("src must be [h,w] or [N,h,w]")
    n, h, w = s.shape
    H, W = (int(v) for v in size)
    out = np.empty((n, H, W), np.float32)
    rc = _lib().oracle_resize_linear_f32(s.ctypes.data, n, h, w, out.ctypes.data, H, W)
    if rc != 0:
        raise ValueError(f"oracle resize does not take {n}x{h}x{w} -> {H}x{W} (code {rc})")
    return out[0] if squeeze else out
