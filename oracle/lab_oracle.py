"""TEST INFRASTRUCTURE ONLY -- ctypes binding of oracle/liblab_oracle.so (oracle/lab_oracle.c): the plain-C restatement
of OpenCV's 8-bit cvtColor(COLOR_BGR2Lab).

Used by tests/ and __graft_entry__.smoke() as the CPU checker.  Never imported by the product package.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "lab_oracle.c")
# the same flags as oracle/Makefile's C oracle: no FMA contraction, baseline x86-64 ISA
CFLAGS = ["-O2", "-std=c11", "-fPIC", "-ffp-contract=off", "-fvisibility=hidden", "-Wall", "-Wextra"]


def _so_path() -> str:
    # next to the source; in a read-only checkout, under the temporary directory instead
    d = _HERE if os.access(_HERE, os.W_OK) else os.path.join(tempfile.gettempdir(), f"dcmt_lab_oracle_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    return os.path.join(d, "liblab_oracle.so")


def build(force: bool = False) -> str:
    so = _so_path()
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(_SRC):
        cc = os.environ.get("CC", "gcc")
        subprocess.run([cc] + CFLAGS + ["-shared", "-o", so, _SRC, "-lm"], check=True, capture_output=True)
    return so


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.dcmt_oracle_bgr2lab.restype = None
        _lib.dcmt_oracle_bgr2lab.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    return _lib


def bgr2lab(bgr):
    """OpenCV's 8-bit cvtColor(COLOR_BGR2Lab) (main_lc.cpp:182-183): (rows, cols, 3) uint8 BGR -> uint8 Lab."""
    src = np.ascontiguousarray(bgr, np.uint8)
    if src.ndim != 3 or src.shape[2] != 3:
        raise ValueError("bgr must be (rows, cols, 3)")
    out = np.empty_like(src)
    lib().dcmt_oracle_bgr2lab(src.ctypes.data, out.ctypes.data, src.shape[0], src.shape[1])
    return out
