"""Per-sample colours from the CPU oracle (tests/native/oracle_samples.c, which compiles oracle/rt_oracle.c into
itself): rto_sample_colors.  Built on first use into a temporary directory, with the oracle's compiler flags."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import oracle_lib as O

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "native", "oracle_samples.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="rto_samples_"), "librto_samples.so")
        subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-std=c11", "-pthread",
                        "-shared", "-o", out, SRC, "-lm", "-pthread"], check=True, capture_output=True)
        _lib = C.CDLL(out)
        _lib.rto_sample_colors.restype = C.c_int
        _lib.rto_sample_colors.argtypes = [C.POINTER(O.Scene), C.POINTER(O.Camera), C.POINTER(O.Params), C.c_int,
                                           C.c_int, C.c_void_p]
    return _lib


def sample_colors(soa, cam, spp, max_depth, seed=1, flags=O.FLAGS_MAIN, rows=None) -> np.ndarray:
    """float64 [rows, W, spp, 3]: the colour of every sample of each pixel of `rows` (default: all)."""
    sc, cm = O.make_scene(soa), O.make_camera(cam)
    prm = O.Params(int(spp), int(max_depth), int(seed), int(flags) & 0xffff, 0)
    r0, r1 = (0, cm.height) if rows is None else rows
    out = np.zeros((r1 - r0, cm.width, int(spp), 3), dtype=np.float64)
    rc = lib().rto_sample_colors(C.byref(sc), C.byref(cm), C.byref(prm), int(r0), int(r1), out.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"rto_sample_colors failed: {rc}")
    return out
