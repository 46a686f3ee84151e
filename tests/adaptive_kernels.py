"""The adaptive-sampling kernels on their own (tests/native/adaptive_kernels.cu, which includes
raytracing-clj_b200/csrc/rtclj_adaptive.cuh unchanged): the compaction, unit_stderr and finalize_adaptive_kernel
launched on device pointers.  Built on first use into a temporary directory, with the library's nvcc flags."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "native", "adaptive_kernels.cu")
CSRC = os.path.join(os.path.dirname(HERE), "raytracing-clj_b200", "csrc")
_lib = None


def nvcc() -> str | None:
    found = shutil.which("nvcc")
    if found:
        return found
    cand = "/usr/local/cuda/bin/nvcc"
    return cand if os.path.exists(cand) else None


def build(out_dir: str) -> str:
    """Compiles the harness for sm_100a into out_dir; returns the shared library's path."""
    out = os.path.join(out_dir, "libadaptive_kernels.so")
    r = subprocess.run([nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "--fmad=false",
                        "-Xcompiler", "-ffp-contract=off", "-Xcompiler", "-fPIC", "-shared", "-I", CSRC,
                        "-o", out, SRC], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed on {SRC}:\n{r.stderr}")
    return out


class AParams(C.Structure):
    """rtclj::AParams, field for field (layout() checks the offsets against the compiler's)."""
    _fields_ = [("sample_buf", C.c_void_p), ("sample_stride", C.c_uint64), ("partial", C.c_void_p),
                ("out_linear", C.c_void_p), ("out_rgb8", C.c_void_p), ("W", C.c_int), ("spp", C.c_int),
                ("nchunks", C.c_int), ("shard_index", C.c_int), ("shard_count", C.c_int), ("shard_rows", C.c_int),
                ("flags", C.c_uint), ("local_pixels", C.c_uint64), ("acc", C.c_void_p), ("acc2", C.c_void_p),
                ("samples", C.c_void_p), ("live", C.c_void_p), ("seeded", C.c_int), ("strict", C.c_int),
                ("mean_n", C.c_int), ("decide", C.c_int), ("unit", C.c_int), ("target", C.c_int),
                ("min_samples", C.c_int), ("abs_tol", C.c_double), ("rel_tol", C.c_double)]


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build(tempfile.mkdtemp(prefix="rtclj_adaptive_kernels_")))
        _lib.ak_relist.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.ak_unit_stderr.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_void_p,
                                        C.c_void_p, C.c_void_p]
        _lib.ak_finalize.argtypes = [C.POINTER(AParams), C.c_void_p]
        _lib.ak_aparams_layout.argtypes = [C.POINTER(C.c_uint64), C.c_int]
        check_layout(_lib)
    return _lib


def check_layout(so) -> None:
    v = (C.c_uint64 * 64)()
    n = so.ak_aparams_layout(v, 64)
    want = [C.sizeof(AParams)] + [getattr(AParams, f).offset for f, _ in AParams._fields_]
    assert list(v[:n]) == want, ("AParams layout differs from rtclj_adaptive.cuh", list(v[:n]), want)


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _check(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what}: CUDA error {rc}")


def relist(live):
    """live: uint8 cuda tensor [n] -> (list as numpy uint32 [count], count)."""
    import torch
    n = live.numel()
    tiles = (n + list_tile() - 1) // list_tile()
    # poisoned, so that a count or entry the compaction does not write shows
    aux = torch.full((1 + max(tiles, 1),), -1, dtype=torch.int32, device=live.device)
    lst = torch.full((max(n, 1),), -1, dtype=torch.int32, device=live.device)
    _check(lib().ak_relist(live.data_ptr(), n, aux.data_ptr(), lst.data_ptr(), _stream()), "ak_relist")
    torch.cuda.synchronize()
    count = int(aux[0].item()) & 0xFFFFFFFF
    return lst[:count].cpu().numpy().view("uint32").copy(), count


def unit_stderr(s1, s2, n, u):
    """s1, s2 float64 and n int32 cuda tensors of one shape -> (stderr, moments_overflow) as numpy."""
    import torch
    out = torch.empty_like(s1)
    ovf = torch.empty(s1.shape, dtype=torch.uint8, device=s1.device)
    _check(lib().ak_unit_stderr(s1.data_ptr(), s2.data_ptr(), n.data_ptr(), int(u), s1.numel(), out.data_ptr(),
                                ovf.data_ptr(), _stream()), "ak_unit_stderr")
    torch.cuda.synchronize()
    return out.cpu().numpy(), ovf.cpu().numpy().astype(bool)


def finalize(A: AParams):
    import torch
    _check(lib().ak_finalize(C.byref(A), _stream()), "ak_finalize")
    torch.cuda.synchronize()


def list_tile() -> int:
    return lib().ak_list_tile()
