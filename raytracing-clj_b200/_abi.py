"""ctypes binding of librtclj_b200.so (include/rtclj_b200.h).  Loading fails LOUDLY:
there is no CPU fallback and no pure-Python path behind these calls."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RTCLJ_LIB") or os.path.join(HERE, "librtclj_b200.so")  # RTCLJ_LIB: tuning experiments only

LAMBERTIAN, METAL, DIELECTRIC = 0, 1, 2
F_NEAR_ZERO_GUARD, F_SCHLICK, F_REVERSE_PRODUCT, F_MEAN_DIVIDE = 1, 2, 4, 8
F_NORMAL_SHADING, F_QUANT_LINEAR, F_NO_CULL, F_SMEM_TABLE = 16, 32, 1 << 16, 1 << 17
F_LANE_KERNEL, F_WAVE_KERNEL, F_LANE2_KERNEL, F_SPLIT_KERNEL = 1 << 18, 1 << 19, 1 << 20, 1 << 21
FLAGS_MAIN = F_NEAR_ZERO_GUARD | F_SCHLICK | F_REVERSE_PRODUCT | F_MEAN_DIVIDE
FLAGS_REALM = 0
FLAGS_I = F_NORMAL_SHADING | F_QUANT_LINEAR
OK, E_INVALID, E_NO_DEVICE, E_CUDA, E_TOO_LARGE, E_BUFFER = range(6)


class Scene(C.Structure):
    _fields_ = [("n", C.c_int32), ("_pad", C.c_int32), ("center_xyz", C.c_void_p),
                ("radius", C.c_void_p), ("material", C.c_void_p), ("albedo_rgb", C.c_void_p),
                ("fuzz", C.c_void_p), ("ior", C.c_void_p)]


class Camera(C.Structure):
    _fields_ = [("pixel00", C.c_double * 3), ("pixel_du", C.c_double * 3),
                ("pixel_dv", C.c_double * 3), ("center", C.c_double * 3),
                ("defocus_u", C.c_double * 3), ("defocus_v", C.c_double * 3),
                ("defocus_angle", C.c_double), ("width", C.c_int32), ("height", C.c_int32)]


class Params(C.Structure):
    _fields_ = [("spp", C.c_int32), ("max_depth", C.c_int32), ("seed", C.c_uint64),
                ("flags", C.c_uint32), ("samples_per_unit", C.c_int32),
                ("shard_index", C.c_int32), ("shard_count", C.c_int32), ("shard_rows", C.c_int32),
                ("device", C.c_int32), ("_pad", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("samples", C.c_uint64), ("segments", C.c_uint64), ("exact_tests", C.c_uint64),
                ("list_overflows", C.c_uint64), ("prefilter_tests", C.c_uint64), ("device_ms", C.c_double), ("kernel_ms", C.c_double), ("total_ms", C.c_double),
                ("samples_per_unit", C.c_int32), ("n_devices", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


#: every symbol include/rtclj_b200.h declares (tests/test_abi.py checks the list against the header)
SYMBOLS = {
    "rtclj_abi_version": (C.c_int, []),
    "rtclj_last_error": (C.c_char_p, []),
    "rtclj_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "rtclj_render": (C.c_int, [C.POINTER(Scene), C.POINTER(Camera), C.POINTER(Params), C.c_void_p,
                               C.c_void_p, C.POINTER(Stats)]),
    "rtclj_render_multi": (C.c_int, [C.POINTER(Scene), C.POINTER(Camera), C.POINTER(Params),
                                     C.POINTER(C.c_int32), C.c_int32, C.c_void_p, C.c_void_p,
                                     C.POINTER(Stats)]),
    "rtclj_render_multi_ppm": (C.c_int, [C.POINTER(Scene), C.POINTER(Camera), C.POINTER(Params),
                                         C.POINTER(C.c_int32), C.c_int32, C.c_void_p, C.c_size_t,
                                         C.POINTER(C.c_size_t), C.POINTER(Stats)]),
    "rtclj_shard_plan": (C.c_int, [C.c_int32, C.c_size_t, C.c_int32, C.c_int32, C.c_int32, C.c_size_t,
                                   C.POINTER(C.c_uint64), C.c_size_t, C.POINTER(C.c_size_t)]),
    "rtclj_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "rtclj_host_free": (C.c_int, [C.c_void_p]),
    "rtclj_host_register": (C.c_int, [C.c_void_p, C.c_size_t]),
    "rtclj_host_unregister": (C.c_int, [C.c_void_p]),
    "rtclj_ctx_create": (C.c_int, [C.c_int32, C.POINTER(C.c_void_p)]),
    "rtclj_ctx_destroy": (None, [C.c_void_p]),
    "rtclj_ctx_set_scene": (C.c_int, [C.c_void_p, C.POINTER(Scene)]),
    "rtclj_ctx_render": (C.c_int, [C.c_void_p, C.POINTER(Camera), C.POINTER(Params), C.c_void_p,
                                   C.c_void_p, C.c_void_p]),
    "rtclj_ctx_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(Stats)]),
    "rtclj_ctx_render_frames": (C.c_int, [C.c_void_p, C.POINTER(Camera), C.c_int32, C.POINTER(Params), C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    "rtclj_render_frames": (C.c_int, [C.POINTER(Scene), C.POINTER(Camera), C.c_int32, C.POINTER(Params),
                                      C.POINTER(C.c_int32), C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(Stats)]),
    "rtclj_ctx_accum_begin": (C.c_int, [C.c_void_p, C.POINTER(Camera), C.POINTER(Params), C.POINTER(C.c_int32),
                                        C.c_void_p]),
    "rtclj_ctx_accum_step": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32),
                                       C.c_void_p]),
    "rtclj_progressive_create": (C.c_int, [C.POINTER(Scene), C.POINTER(Camera), C.POINTER(Params),
                                           C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int32),
                                           C.POINTER(C.c_void_p)]),
    "rtclj_progressive_step": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32),
                                         C.POINTER(Stats)]),
    "rtclj_progressive_destroy": (C.c_int, [C.c_void_p]),
    "rtclj_ctx_accum_begin_adaptive": (C.c_int, [C.c_void_p, C.POINTER(Camera), C.POINTER(Params), C.POINTER(C.c_double),
                                                 C.c_int32, C.POINTER(C.c_int32), C.c_void_p]),
    "rtclj_ctx_accum_noise": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p]),
    "rtclj_progressive_create_adaptive": (C.c_int, [C.POINTER(Scene), C.POINTER(Camera), C.POINTER(Params),
                                                    C.POINTER(C.c_double), C.c_int32, C.POINTER(C.c_int32), C.c_int32,
                                                    C.POINTER(C.c_int32), C.POINTER(C.c_void_p)]),
    "rtclj_progressive_noise": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]),
    "rtclj_calibrate_peaks": (C.c_int, [C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                        C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "rtclj_quantise_rgb8": (C.c_int, [C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p]),
    "rtclj_encode_ppm_p3": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t,
                                      C.POINTER(C.c_size_t)]),
    "rtclj_encode_ppm_p3_gpu": (C.c_int, [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t,
                                          C.POINTER(C.c_size_t)]),
    "rtclj_ctx_encode_ppm_p3": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t,
                                          C.POINTER(C.c_size_t), C.c_void_p]),
    "rtclj_ctx_encode_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "rtclj_decode_ppm_p3": (C.c_int, [C.c_char_p, C.c_size_t, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_void_p,
                                      C.c_size_t]),
    "rtclj_encode_png": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t,
                                   C.POINTER(C.c_size_t)]),
    "rtclj_ctx_encode_png": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t,
                                       C.POINTER(C.c_size_t), C.c_void_p]),
    "rtclj_encode_png_gpu": (C.c_int, [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t,
                                       C.POINTER(C.c_size_t)]),
    "rtclj_render_multi_png": (C.c_int, [C.POINTER(Scene), C.POINTER(Camera), C.POINTER(Params),
                                         C.POINTER(C.c_int32), C.c_int32, C.c_void_p, C.c_size_t,
                                         C.POINTER(C.c_size_t), C.POINTER(Stats)]),
    "rtclj_ratio_to_double": (C.c_double, [C.c_int64, C.c_int64]),
    "rtclj_camera_main": (C.c_int, [C.c_int32, C.c_int32, C.c_double, C.POINTER(C.c_double),
                                    C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_double,
                                    C.c_double, C.POINTER(Camera)]),
    "rtclj_camera_realm": (C.c_int, [C.c_int32, C.c_int32, C.c_double, C.POINTER(C.c_double),
                                     C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(Camera)]),
    "rtclj_camera_i": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(Camera)]),
    "rtclj_scene_random_field": (C.c_int, [C.c_uint64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.POINTER(C.c_int32)]),
}

_lib = None


class RtcljError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"rtclj error {code}: {message}")
        self.code = code


def lib():
    """The loaded library; raises if it has not been built (run __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RtcljError(-1, f"{LIB_PATH} is missing: build it with `make -C {HERE}/csrc` "
                                 "(there is no CPU fallback)")
        handle = C.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SYMBOLS.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = restype, argtypes
        if handle.rtclj_abi_version() != 1:
            raise RtcljError(-1, "ABI version mismatch")
        _lib = handle
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise RtcljError(rc, lib().rtclj_last_error().decode("utf-8", "replace"))
