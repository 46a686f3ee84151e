"""Camera sequences without a GPU (rtclj_render_frames / rtclj_ctx_render_frames): every argument check runs before a
device is touched, the calls fail loudly without a device, the CLI's turntable cameras are the reference's camera
moved along a circle, and the frame twins keep the code properties of the kernels they copy."""
import ctypes as C
import math
import os
import re
import shutil
import subprocess
import sys

import pytest

import raytracing_clj_b200 as R
from raytracing_clj_b200 import _abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "raytracing-clj_b200", "librtclj_b200.so")
CAM = R.camera


def _call(cams, n=None, flags=_abi.FLAGS_MAIN, spp=4, devices=(0,), scene=True):
    """rtclj_render_frames with these cameras; returns (code, message)."""
    lib = _abi.lib()
    soa = R.scenes.to_soa(R.scenes.main_hittables())
    sc = R.render._scene_struct(soa)
    arr = (_abi.Camera * max(1, len(cams)))(*[R.render._camera_struct(c) for c in cams]) if cams is not None else None
    prm = _abi.Params(spp, 5, 1, flags, 0, 0, 0, 0, 0, 0)
    devs = (C.c_int32 * len(devices))(*devices)
    rc = lib.rtclj_render_frames(C.byref(sc) if scene else None, arr, len(cams or []) if n is None else n,
                                 C.byref(prm), devs, len(devices), None, None, None)
    return rc, lib.rtclj_last_error().decode()


def test_arguments_are_checked_before_any_device():
    cams = [CAM.main_camera(32, look_from=CAM.turntable_look_from(k, 5)) for k in range(5)]
    assert _call(cams, n=0)[0] == _abi.E_INVALID
    assert _call(cams, n=-3)[0] == _abi.E_INVALID
    rc, msg = _call(None, n=2)
    assert rc == _abi.E_INVALID and "camera" in msg
    assert _call(cams, scene=False)[0] == _abi.E_INVALID
    rc, msg = _call(cams[:2] + [CAM.main_camera(48)] + cams[3:])
    assert rc == _abi.E_INVALID and "frame 2" in msg and "48x27" in msg
    bad = _abi.Camera.from_buffer_copy(R.render._camera_struct(cams[3]))
    bad.pixel_du[1] = math.nan
    rc, msg = _call(cams[:3] + [bad] + cams[4:])
    assert rc == _abi.E_INVALID and "frame 3" in msg and "non-finite" in msg
    bad = _abi.Camera.from_buffer_copy(R.render._camera_struct(cams[1]))
    bad.width = 0
    rc, msg = _call(cams[:1] + [bad])
    assert rc == _abi.E_INVALID and "frame 1" in msg
    for f in (_abi.F_WAVE_KERNEL, _abi.F_SPLIT_KERNEL):
        rc, msg = _call(cams, flags=_abi.FLAGS_MAIN | f)
        assert rc == _abi.E_INVALID and "sequence" in msg
    assert _call(cams, spp=0)[0] == _abi.E_INVALID
    lib = _abi.lib()
    prm = _abi.Params(4, 5, 1, _abi.FLAGS_MAIN, 0, 0, 0, 0, 0, 0)
    arr = (_abi.Camera * 1)(R.render._camera_struct(cams[0]))
    assert lib.rtclj_ctx_render_frames(None, arr, 1, C.byref(prm), None, None, None) == _abi.E_INVALID


def check_no_device():
    cams = [CAM.main_camera(16, look_from=CAM.turntable_look_from(k, 3)) for k in range(3)]
    rc, msg = _call(cams)
    assert rc == _abi.E_NO_DEVICE, (rc, msg)
    with pytest.raises(_abi.RtcljError) as e:
        R.render.render_frames(R.scenes.main_hittables(), cams, 2, 5)
    assert e.value.code == _abi.E_NO_DEVICE


def test_no_device_is_an_error():
    """In a child process that sees no CUDA device, so that it runs on machines with a GPU as well."""
    code = "import sys; sys.path[:0] = sys.argv[1:]; import test_frames; test_frames.check_no_device()"
    subprocess.run([sys.executable, "-c", code, ROOT, os.path.join(ROOT, "tests")], check=True,
                   env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))


def test_turntable_cameras():
    """Frame 0 is the reference's camera; frame k is rtclj_camera_main at look_from turned by k * 360/n degrees about
    the vertical axis through look_at (same height, same distance)."""
    n = 12
    cams = CAM.turntable_cameras(n)
    ref = CAM.main_camera()
    for name in ("pixel00", "pixel_du", "pixel_dv", "center", "defocus_u", "defocus_v", "defocus_angle", "width", "height"):
        assert getattr(cams[0], name) == getattr(ref, name), name
    lib = _abi.lib()
    vec = lambda v: (C.c_double * 3)(*v)  # noqa: E731
    for k in range(n):
        lf = CAM.turntable_look_from(k, n)
        assert lf[1] == 2.0 and math.isclose(math.hypot(lf[0], lf[2] + 1.0), math.hypot(-2.0, 2.0))
        assert math.isclose(math.atan2(lf[2] + 1.0, lf[0]) % (2 * math.pi),
                            (math.atan2(2.0, -2.0) - 2 * math.pi * k / n) % (2 * math.pi), abs_tol=1e-12)
        c = _abi.Camera()
        assert lib.rtclj_camera_main(400, cams[k].height, 20.0, vec(lf), vec((0.0, 0.0, -1.0)), vec((0.0, 1.0, 0.0)),
                                     10.0, 3.4, C.byref(c)) == 0
        for name in ("pixel00", "pixel_du", "pixel_dv", "center", "defocus_u", "defocus_v"):
            assert tuple(getattr(c, name)) == tuple(getattr(cams[k], name)), (k, name)
    assert len({tuple(c.center) for c in cams}) == n


def test_cli_refuses_a_bad_frame_count():
    for bad in (["main", "--frames"], ["main", "--frames", "0"], ["main", "--frames", "x"]):
        with pytest.raises(SystemExit):
            R.main._cli(bad)


# ---------------------------------------------------------------- the frame twins' code (tests/test_build_artifacts.py)
needs_cuobjdump = pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not installed")


@pytest.fixture(scope="module")
def sass():
    out = subprocess.run(["cuobjdump", "-sass", LIB], check=True, capture_output=True, text=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            funcs[name] = []
        elif name and re.match(r"\s+/\*[0-9a-f]{4,}\*/\s", line):
            funcs[name].append(line)
    return funcs


def kernels(funcs, key):
    names = [n for n in funcs if key in n]
    assert names, key
    return [funcs[n] for n in names]


@needs_cuobjdump
@pytest.mark.parametrize("key", ["render_frames_kernelILb1", "render_lane2_frames_kernel"])
def test_frame_twins_cull_through_uniform_registers(sass, key):
    """The constant-table twins keep the cull table's uniform operands (LDCU.64 -> FFMA2 .. UR).  Their per-lane
    constant loads (LDC R, c[0x0][R+..]) read the unit's frame camera, outside the cull loop: none lies between the
    first and the last FFMA2 with a uniform operand."""
    for body in kernels(sass, key):
        uniform = [l for l in body if re.search(r"LDCU\.64 UR\d+, c\[0x0\]\[UR\d+", l)]
        cull = [i for i, l in enumerate(body) if "FFMA2" in l and ".F32x2" in l and " UR" in l]
        per_lane = [i for i, l in enumerate(body) if re.search(r"LDC(?:\.64)? R\d+, c\[0x0\]\[R\d+", l)]
        assert len(uniform) >= 32 and len(cull) >= 48, (len(uniform), len(cull))
        assert per_lane and not [i for i in per_lane if cull[0] <= i <= cull[-1]]


@needs_cuobjdump
def test_chunked_frame_twins_fit_the_instruction_cache(sass):
    for key in ("render_frames_kernelILb1ELb0ELb0", "render_frames_kernelILb1ELb0ELb1", "render_lane2_frames_kernelILb0"):
        body = kernels(sass, key)[0]
        assert len(body) * 16 <= 34 * 1024, (key, len(body) * 16)


@needs_cuobjdump
def test_primary_frames_twin_reads_no_memory(sass):
    """render_primary_frames_kernel: the cameras, like the spheres, are kernel parameters -- no global or shared
    loads, one unit sum stored.  The instantiation with the defocus disk has no local memory either; the one without
    keeps one word (the loop bound) in local memory at 80 registers, an L1 hit per sample (DESIGN.md section 4.12)."""
    for key, local in (("render_primary_frames_kernelILb1", 0), ("render_primary_frames_kernelILb0", 2)):
        text = "\n".join(kernels(sass, key)[0])
        assert not re.search(r"\b(LDG|LDS|STS)\b", text), key
        assert len(re.findall(r"\b(LDL|STL)\b", text)) <= 2 * local, key
        assert len(re.findall(r"\bSTG\b", text)) == 3, key
