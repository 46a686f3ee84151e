"""Accumulations over frames without a GPU (rtclj_ctx_accum_begin_frames / rtclj_progressive_create_frames): every
refusal comes before a device is touched and names the frame, the calls are exported and bound with the header's
arity (ctypes and Clojure), the CLI routes --frames with --tolerance to the adaptive sequence, and the listed and seeded
frame twins keep the code properties of the kernels they copy."""
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
CLJ = os.path.join(ROOT, "integration", "clojure", "src", "rtclj", "native.clj")
CAM = R.camera
NEW = ("rtclj_ctx_accum_begin_frames", "rtclj_progressive_create_frames")


def _cams(n=4, width=32):
    return [CAM.main_camera(width, look_from=CAM.turntable_look_from(k, n)) for k in range(n)]


def _create(cams, n=None, flags=_abi.FLAGS_MAIN, spp=40, spu=0, tol=(0.01, 0.1), least=None, devices=(0,),
            scene=True):
    """rtclj_progressive_create_frames with these arguments; returns (code, message, handle)."""
    lib = _abi.lib()
    soa = R.scenes.to_soa(R.scenes.main_hittables())
    sc = R.render._scene_struct(soa)
    arr = (_abi.Camera * max(1, len(cams)))(*[R.render._camera_struct(c) for c in cams]) if cams is not None else None
    prm = _abi.Params(spp, 5, 1, flags, spu, 0, 0, 0, 0, 0)
    t = (C.c_double * 2)(*tol) if tol is not None else None
    if least is None:
        least = 2 * R.render.pass_unit(32, 18, spp, 5, flags, spu)
    devs = (C.c_int32 * len(devices))(*devices)
    out, unit = C.c_void_p(), C.c_int32()
    rc = lib.rtclj_progressive_create_frames(C.byref(sc) if scene else None, arr, len(cams or []) if n is None else n,
                                             C.byref(prm), t, least, devs, len(devices), C.byref(unit), C.byref(out))
    return rc, lib.rtclj_last_error().decode(), out


@pytest.mark.parametrize("tol", [(0.01, 0.1), None], ids=["adaptive", "plain"])
def test_refusals_before_any_device(tol):
    """What rtclj_ctx_render_frames refuses (naming the frame), what an accumulation refuses and what an adaptive one
    refuses: RTCLJ_E_INVALID with no handle, on a machine without a GPU as well (no device is ever asked)."""
    cams = _cams()

    def refused(*args, **kw):
        kw.setdefault("tol", tol)
        rc, msg, out = _create(*args, **kw)
        assert rc == _abi.E_INVALID and not out.value, (rc, msg)
        return msg

    assert "n_frames" in refused(cams, n=0)
    assert "n_frames" in refused(cams, n=-2)
    assert "camera" in refused(None, n=2)
    assert "scene" in refused(cams, scene=False)
    msg = refused(cams[:2] + [CAM.main_camera(48)] + cams[3:])
    assert "frame 2" in msg and "48x27" in msg
    bad = _abi.Camera.from_buffer_copy(R.render._camera_struct(cams[3]))
    bad.center[0] = math.inf
    msg = refused(cams[:3] + [bad])
    assert "frame 3" in msg and "non-finite" in msg
    bad = _abi.Camera.from_buffer_copy(R.render._camera_struct(cams[1]))
    bad.height = 0
    assert "frame 1" in refused(cams[:1] + [bad] + cams[2:])
    for f in (_abi.F_WAVE_KERNEL, _abi.F_SPLIT_KERNEL):
        refused(cams, flags=_abi.FLAGS_MAIN | f)
    assert "spp" in refused(cams, spp=0)
    assert "2^30" in refused(cams, spp=(1 << 30) + 1)
    assert "frame 0" in refused(cams, spp=-1)
    assert "empty device list" in refused(cams, devices=())
    if tol is not None:
        for t in ((math.nan, 0.1), (0.01, -1.0), (math.inf, 0.0)):
            assert "tolerances" in refused(cams, tol=t)
        unit = R.render.pass_unit(32, 18, 40, 5)
        assert "min_samples" in refused(cams, least=2 * unit - 1)


def test_ctx_begin_refuses_a_null_context():
    lib = _abi.lib()
    cams = _cams(2)
    arr = (_abi.Camera * 2)(*[R.render._camera_struct(c) for c in cams])
    prm = _abi.Params(40, 5, 1, _abi.FLAGS_MAIN, 0, 0, 0, 0, 0, 0)
    unit = C.c_int32(-7)
    assert lib.rtclj_ctx_accum_begin_frames(None, arr, 2, C.byref(prm), None, 0, C.byref(unit), None) == _abi.E_INVALID
    assert "ctx" in lib.rtclj_last_error().decode() and unit.value == -7


def check_no_device():
    rc, msg, out = _create(_cams(3))
    assert rc == _abi.E_NO_DEVICE and not out.value, (rc, msg)
    with pytest.raises(_abi.RtcljError) as e:
        R.render.ProgressiveFrames(R.scenes.main_hittables(), _cams(3), 40, 5, tolerance=(0.01, 0.1))
    assert e.value.code == _abi.E_NO_DEVICE
    with pytest.raises(_abi.RtcljError) as e:
        R.render.Context(0)
    assert e.value.code == _abi.E_NO_DEVICE


def test_no_device_is_an_error():
    """In a child process that sees no CUDA device, so that it runs on machines with a GPU as well."""
    code = "import sys; sys.path[:0] = sys.argv[1:]; import test_adaptive_frames as t; t.check_no_device()"
    subprocess.run([sys.executable, "-c", code, ROOT, os.path.join(ROOT, "tests")], check=True,
                   env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))


def test_exports_and_signatures():
    """The library exports both calls, and _abi binds them with the header's argument count."""
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "rtclj_b200.h")).read(), flags=re.S)
    lib = _abi.lib()
    for sym in NEW:
        assert hasattr(lib, sym)
        decl = re.search(r"\b%s\s*\(([^)]*)\)\s*;" % sym, hdr)
        assert decl, sym
        assert len(decl.group(1).split(",")) == len(_abi.SYMBOLS[sym][1]), sym
    assert _abi.SYMBOLS["rtclj_ctx_accum_begin_frames"][1][4] is C.POINTER(C.c_double)
    assert _abi.SYMBOLS["rtclj_progressive_create_frames"][1][2] is C.c_int32
    assert hasattr(R.render.Context, "accum_begin_frames") and issubclass(R.render.ProgressiveFrames, R.render.Progressive)


def test_clojure_binds_the_sequence_calls():
    """tests/test_clojure_binding.py checks every bound call's arity against the header; here: the new ones are bound
    and the two entry points exist."""
    text = open(CLJ).read()
    assert '(downcall "rtclj_progressive_create_frames"' in text
    assert "(defn progressive-frames\n" in text and "(defn progressive-frames-adaptive\n" in text


# ---------------------------------------------------------------- CLI
@pytest.fixture
def calls(monkeypatch):
    seen = []
    monkeypatch.setattr(R.main, "frames_variant", lambda *a, **k: seen.append(("frames", a, k)))
    monkeypatch.setattr(R.main, "main_variant", lambda *a, **k: seen.append(("main", a, k)))
    return seen


def test_cli_frames_with_tolerance(calls):
    R.main._cli(["main", "500", "50", "--frames", "60", "--tolerance", "0.004,0.04"])
    R.main._cli(["main", "200", "--tolerance", "0.01,0.1", "--frames", "8", "--every", "25", "--apng"])
    R.main._cli(["main", "--frames", "3", "--gpu-png", "--tolerance", "0,0.5"])
    assert calls == [
        ("frames", (500, 50, 60), {"gpu_png": False, "apng": False, "tolerance": (0.004, 0.04), "every": 0}),
        ("frames", (200, 50, 8), {"gpu_png": False, "apng": True, "tolerance": (0.01, 0.1), "every": 25}),
        ("frames", (100, 50, 3), {"gpu_png": True, "apng": False, "tolerance": (0.0, 0.5), "every": 0})]


def test_cli_frames_without_tolerance_is_unchanged(calls):
    R.main._cli(["main", "500", "50", "--frames", "60"])
    R.main._cli(["main", "--frames", "4", "--apng"])
    R.main._cli(["main", "64", "8", "--tolerance", "0.01,0.1", "--every", "16"])
    assert calls == [("frames", (500, 50, 60), {"gpu_png": False, "apng": False}),
                     ("frames", (100, 50, 4), {"gpu_png": False, "apng": True}),
                     ("main", (64, 8), {"every": 16, "tolerance": (0.01, 0.1), "gpu_png": False, "denoise": False})]


def test_cli_refusals(calls):
    for bad in (["main", "--frames", "4", "--tolerance", "0.1"], ["main", "--frames", "4", "--tolerance", "-1,0"],
                ["main", "--frames", "4", "--tolerance", "0,0", "--every", "0"], ["main", "--frames", "0", "--tolerance", "0,0"]):
        with pytest.raises(SystemExit):
            R.main._cli(bad)
    assert calls == []


# ---------------------------------------------------------------- the twins' code
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


@pytest.fixture(scope="module")
def usage():
    out = subprocess.run(["cuobjdump", "-res-usage", LIB], check=True, capture_output=True, text=True).stdout
    res = {}
    for name, line in re.findall(r"Function (\S+):\n\s*(REG:.*)", out):
        res[name] = {k: int(v) for k, v in re.findall(r"(\w+):(\d+)", line)}
    return res


def kernels(funcs, key):
    names = [n for n in funcs if key in n]
    assert names, key
    return {n: funcs[n] for n in names}


@needs_cuobjdump
@pytest.mark.parametrize("key", ["render_listed_frames_kernelILb1", "render_lane2_listed_frames_kernel"])
def test_listed_twins_cull_through_uniform_registers(sass, key):
    """The constant-table listed twins keep the cull table's uniform operands (LDCU.64 -> FFMA2 .. UR).  Their per-lane
    constant loads (LDC R, c[0x0][R+..]) read the unit's frame camera, outside the cull loop: none lies between the
    first and the last FFMA2 with a uniform operand."""
    for name, body in kernels(sass, key).items():
        uniform = [l for l in body if re.search(r"LDCU\.64 UR\d+, c\[0x0\]\[UR\d+", l)]
        cull = [i for i, l in enumerate(body) if "FFMA2" in l and ".F32x2" in l and " UR" in l]
        per_lane = [i for i, l in enumerate(body) if re.search(r"LDC(?:\.64)? R\d+, c\[0x0\]\[R\d+", l)]
        assert len(uniform) >= 32 and len(cull) >= 48, (name, len(uniform), len(cull))
        assert per_lane and not [i for i in per_lane if cull[0] <= i <= cull[-1]], name


# Each twin, the camera-sequence kernel of the same instantiation and the single-camera kernel whose tickets it takes
# (listed, seeded), with that kernel's base.  Spills (LOCAL) stay at the copied kernels' 0; the save area around the
# out-of-line calls (STACK) may grow by what each of the two twins adds to the base kernel, no more.
TWINS = [("render_listed_frames_kernelI" + t, "render_frames_kernelI" + t, "render_listed_kernelI" + t,
          "render_kernelI" + t)
         for t in ("Lb1ELb0ELb0E", "Lb1ELb0ELb1E", "Lb1ELb1ELb0E", "Lb1ELb1ELb1E", "Lb0ELb0ELb0E", "Lb0ELb1ELb0E")]
TWINS += [("render_lane2_listed_frames_kernelI" + t, "render_lane2_frames_kernelI" + t,
           "render_lane2_listed_kernelI" + t, "render_lane2_kernelI" + t) for t in ("Lb0E", "Lb1E")]
TWINS += [("render_primary_%s_frames_kernelI%s" % (v, t), "render_primary_frames_kernelI" + t,
           "render_primary_%s_kernelI%s" % (v, t), "render_primary_kernelI" + t)
          for v in ("seeded", "listed", "seeded_listed") for t in ("Lb0E", "Lb1E")]


@needs_cuobjdump
@pytest.mark.parametrize("twin,frames,tickets,base", TWINS)
def test_twins_use_no_more_local_memory(usage, twin, frames, tickets, base):
    def of(key):  # the kernel whose demangled name starts with key (_ZN5rtclj<length><name>...)
        (v,) = [v for n, v in usage.items() if n.startswith("_ZN5rtclj") and n[9:].lstrip("0123456789").startswith(key)]
        return v
    t, f, k, b = of(twin), of(frames), of(tickets), of(base)
    assert t["LOCAL"] == 0 and f["LOCAL"] == 0 and k["LOCAL"] == 0, (t, f, k)
    assert t["STACK"] <= f["STACK"] + max(0, k["STACK"] - b["STACK"]), (t, f, k, b)


@needs_cuobjdump
def test_primary_twins_read_only_their_state(sass):
    """The primary-ray twins keep the cameras and spheres in the kernel parameters: no shared loads or stores, and
    global loads only for the list entries and the running sums (seeded: three sums; moments: three more)."""
    for key, loads in (("render_primary_seeded_frames_kernelILb1", 3), ("render_primary_listed_frames_kernelILb1", 2),
                       ("render_primary_seeded_listed_frames_kernelILb1", 8)):
        (text,) = ["\n".join(b) for b in kernels(sass, key).values()]
        assert not re.search(r"\b(LDS|STS)\b", text), key
        assert 1 <= len(re.findall(r"\bLDG\b", text)) <= loads + 2, (key, len(re.findall(r"\bLDG\b", text)))
