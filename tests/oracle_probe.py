"""What the CPU oracle's scans see (tests/native/oracle_probe.c, which compiles oracle/rt_oracle.c into itself with a
probe on trace_sample's closest-hit scan): rto_probe_render.  Built on first use into a temporary directory, with
the oracle's compiler flags."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import oracle_lib as O

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "native", "oracle_probe.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="rto_probe_"), "librto_probe.so")
        subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-std=c11", "-pthread",
                        "-shared", "-o", out, SRC, "-lm", "-pthread"], check=True, capture_output=True)
        _lib = C.CDLL(out)
        _lib.rto_probe_render.restype = C.c_int
        _lib.rto_probe_render.argtypes = [C.POINTER(O.Scene), C.POINTER(O.Camera), C.POINTER(O.Params),
                                          C.POINTER(C.c_uint64)]
    return _lib


def scans(soa, cam, spp, max_depth, seed=1, flags=O.FLAGS_MAIN) -> dict:
    """{"scans", "degenerate", "nan_roots", "segments"} of the oracle's render: closest-hit scans, scans of a direction
    the kernels route to the exhaustive scan, and scans that accept a NaN root."""
    sc, cm = O.make_scene(soa), O.make_camera(cam)
    prm = O.Params(int(spp), int(max_depth), int(seed), int(flags) & 0xffff, 0)
    out = (C.c_uint64 * 4)()
    rc = lib().rto_probe_render(C.byref(sc), C.byref(cm), C.byref(prm), out)
    if rc != 0:
        raise RuntimeError(f"rto_probe_render failed: {rc}")
    return dict(zip(("scans", "degenerate", "nan_roots", "segments"), (int(x) for x in out)))
