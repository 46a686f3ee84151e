"""The C-ABI library loads and exports every symbol include/rtclj_b200.h declares; host-only
entry points work; compute entry points fail LOUDLY without a GPU (no CPU fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import raytracing_clj_b200 as R
from raytracing_clj_b200 import _abi, render

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    text = open(os.path.join(ROOT, "include", "rtclj_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rtclj_[a-z0-9_]+)\s*\(", text)))


def test_every_declared_symbol_is_exported_and_bound():
    names = header_functions()
    assert len(names) >= 18
    lib = _abi.lib()
    for n in names:
        assert hasattr(lib, n), f"{n} declared in the header but not exported"
        assert n in _abi.SYMBOLS, f"{n} has no ctypes prototype"
    assert sorted(_abi.SYMBOLS) == names
    assert lib.rtclj_abi_version() == 1


def test_struct_layouts_match_the_header_comment_in_integration_md():
    assert C.sizeof(_abi.Scene) == 56 and C.sizeof(_abi.Camera) == 160 and C.sizeof(_abi.Params) == 48
    assert _abi.Camera.defocus_angle.offset == 144 and _abi.Camera.width.offset == 152
    assert _abi.Params.seed.offset == 8 and _abi.Params.flags.offset == 16 and _abi.Params.device.offset == 36


def _has_gpu():
    n = C.c_int()
    return _abi.lib().rtclj_device_count(C.byref(n)) == 0 and n.value > 0


def check_no_cpu_fallback():
    assert not _has_gpu()
    with pytest.raises(_abi.RtcljError) as e:
        render.render(R.scenes.main_hittables(), R.camera.main_camera(16), 1, 5)
    assert e.value.code == _abi.E_NO_DEVICE
    with pytest.raises(_abi.RtcljError):
        render.Context(0)
    assert b"CUDA" in _abi.lib().rtclj_last_error() or b"device" in _abi.lib().rtclj_last_error()


def test_no_cpu_fallback():
    """In a child process that sees no CUDA device, so that it runs on machines with a GPU as well."""
    import subprocess
    import sys
    code = "import sys; sys.path[:0] = sys.argv[1:]; import test_abi; test_abi.check_no_cpu_fallback()"
    subprocess.run([sys.executable, "-c", code, ROOT, os.path.join(ROOT, "tests")], check=True,
                   env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))


def test_missing_library_is_an_error(monkeypatch):
    monkeypatch.setattr(_abi, "_lib", None)
    monkeypatch.setattr(_abi, "LIB_PATH", "/nonexistent/librtclj_b200.so")
    with pytest.raises(_abi.RtcljError):
        _abi.lib()


def test_argument_validation_without_compute():
    lib = _abi.lib()
    assert lib.rtclj_device_count(None) == _abi.E_INVALID
    assert lib.rtclj_quantise_rgb8(None, 3, 0, None) == _abi.E_INVALID
    n = C.c_size_t()
    assert lib.rtclj_encode_ppm_p3(None, 0, 4, None, 0, C.byref(n)) == _abi.E_INVALID
    cam = _abi.Camera()
    assert lib.rtclj_camera_i(0, 10, C.byref(cam)) == _abi.E_INVALID


def build_c_client(tmp_path):
    """gcc -std=c11 -pedantic on a plain-C user of the header, linked against the library."""
    import subprocess
    libdir = os.path.join(ROOT, "raytracing-clj_b200")
    exe = str(tmp_path / "abi_c_client")
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                    "-o", exe, os.path.join(ROOT, "tests", "native", "abi_c_client.c"),
                    "-L", libdir, "-lrtclj_b200", "-Wl,-rpath," + libdir], check=True)
    return exe


def test_header_is_valid_c11_and_host_entry_points_work_from_c(tmp_path):
    import subprocess
    out = subprocess.run([build_c_client(tmp_path)], check=True, capture_output=True, text=True).stdout
    assert out.strip() == "ok host"


def test_every_entry_point_describes_its_error():
    """rtclj_last_error() after a failing HOST-side call (ADVICE r1: those returned bare codes)."""
    from raytracing_clj_b200 import _abi
    lib = _abi.lib()
    n = C.c_size_t()
    for call in (lambda: lib.rtclj_encode_ppm_p3(None, 0, 0, None, 0, C.byref(n)),
                 lambda: lib.rtclj_decode_ppm_p3(b"P6\n1 1\n255\n", 11, C.byref(C.c_int32()), C.byref(C.c_int32()), None, 0),
                 lambda: lib.rtclj_camera_i(0, 0, None),
                 lambda: lib.rtclj_quantise_rgb8(None, 3, 0, None)):
        rc = call()
        assert rc != 0 and lib.rtclj_last_error().decode() != ""
