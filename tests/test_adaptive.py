"""Adaptive sampling without a GPU: the entry points refuse to run without a device (no CPU fallback), bad
arguments and null handles are refused, the Clojure shim binds them, and the listed kernels -- the render
kernels that trace only the pixels of a list -- keep the properties of their unlisted twins in the built code."""
import ctypes as C
import math
import os
import re
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "raytracing-clj_b200", "librtclj_b200.so")
CLJ = os.path.join(ROOT, "integration", "clojure", "src", "rtclj", "native.clj")


def _structs():
    import raytracing_clj_b200 as R
    from raytracing_clj_b200 import _abi, render
    world, cam = R.scenes.main_hittables(), R.camera.main_camera(16)
    sc, cm = render._scene_struct(R.scenes.to_soa(world)), render._camera_struct(cam)
    prm = _abi.Params(16, 5, 1, _abi.FLAGS_MAIN, 4, 0, 0, 0, 0, 0)  # pass unit 4
    return world, cam, sc, cm, prm


def check_adaptive_needs_a_device():
    from raytracing_clj_b200 import _abi, render
    lib = _abi.lib()
    world, cam, sc, cm, prm = _structs()
    tol = (C.c_double * 2)(0.01, 0.05)
    devices = (C.c_int32 * 1)(0)
    unit, handle = C.c_int32(), C.c_void_p()
    rc = lib.rtclj_progressive_create_adaptive(C.byref(sc), C.byref(cm), C.byref(prm), tol, 8, devices, 1,
                                               C.byref(unit), C.byref(handle))
    assert rc == _abi.E_NO_DEVICE and not handle.value, rc
    assert lib.rtclj_last_error() != b""
    with pytest.raises(_abi.RtcljError) as e:
        render.Progressive(world, cam, 16, 5, samples_per_unit=4, tolerance=(0.01, 0.05))
    assert e.value.code == _abi.E_NO_DEVICE
    with pytest.raises(_abi.RtcljError) as e:
        render.Context(0)
    assert e.value.code == _abi.E_NO_DEVICE


def test_adaptive_render_fails_without_a_device():
    """In a child process that sees no CUDA device, so that it runs on machines with a GPU as well."""
    code = "import sys; sys.path[:0] = sys.argv[1:]; import test_adaptive; test_adaptive.check_adaptive_needs_a_device()"
    subprocess.run([sys.executable, "-c", code, ROOT, os.path.join(ROOT, "tests")], check=True,
                   env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))


def test_null_handles_and_bad_arguments_are_refused():
    """Checked before any device is touched: the same answer with and without a GPU."""
    from raytracing_clj_b200 import _abi
    lib = _abi.lib()
    _, _, sc, cm, prm = _structs()
    devices = (C.c_int32 * 1)(0)
    unit, handle, active = C.c_int32(), C.c_void_p(), C.c_uint64()
    tol = (C.c_double * 2)(0.01, 0.05)
    assert lib.rtclj_ctx_accum_begin_adaptive(None, C.byref(cm), C.byref(prm), tol, 8, C.byref(unit), None) == _abi.E_INVALID
    assert lib.rtclj_ctx_accum_noise(None, None, None, C.byref(active), None) == _abi.E_INVALID
    assert lib.rtclj_progressive_noise(None, None, None, C.byref(active)) == _abi.E_INVALID

    def create(t, least):
        handle.value = None
        arg = None if t is None else (C.c_double * 2)(*t)
        rc = lib.rtclj_progressive_create_adaptive(C.byref(sc), C.byref(cm), C.byref(prm), arg, least, devices, 1,
                                                   C.byref(unit), C.byref(handle))
        assert not handle.value
        return rc

    for bad in (None, (-1e-3, 0.0), (0.0, -0.5), (math.nan, 0.0), (0.0, math.inf)):
        assert create(bad, 8) == _abi.E_INVALID, bad
        assert lib.rtclj_last_error() != b""
    assert create((0.01, 0.05), 7) == _abi.E_INVALID  # min_samples below two pass units (4)
    assert create((0.01, 0.05), 0) == _abi.E_INVALID
    assert b"min_samples" in lib.rtclj_last_error()


def test_python_pass_unit_follows_the_library_rule():
    from raytracing_clj_b200 import _abi, render
    assert render.pass_unit(64, 36, 40, 50, _abi.FLAGS_MAIN, 8) == 8
    assert render.pass_unit(64, 36, 40, 50, _abi.FLAGS_MAIN, 40) == 1          # strict order
    assert render.pass_unit(64, 36, 40, 1, _abi.FLAGS_MAIN, 0) == 1            # primary rays: strict by default
    assert render.pass_unit(64, 36, 40, 50, _abi.FLAGS_I, 0) == 1
    assert render.pass_unit(1920, 1080, 500, 50, _abi.FLAGS_MAIN, 0) == 27     # auto_samples_per_unit: 19 chunks


def test_clojure_shim_binds_the_adaptive_entry_points():
    text = open(CLJ).read()
    bound = set(re.findall(r'\(downcall "(\w+)"', text))
    assert {"rtclj_progressive_create_adaptive", "rtclj_progressive_noise"} <= bound
    for fn in ("progressive-adaptive", "progressive-noise"):
        assert re.search(r"\(defn %s\s" % re.escape(fn), text), fn


@pytest.fixture(scope="module")
def sass():
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not installed")
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


def one(funcs, key):
    names = [n for n in funcs if key in n]
    assert len(names) == 1, (key, names)
    return funcs[names[0]]


# every listed kernel: (key of its mangled name, key of its unlisted twin)
LISTED = [("render_listed_kernelILb1ELb0ELb0", "render_kernelILb1ELb0ELb0"),
          ("render_listed_kernelILb1ELb1ELb0", "render_kernelILb1ELb1ELb0"),
          ("render_listed_kernelILb1ELb0ELb1", "render_kernelILb1ELb0ELb1"),
          ("render_listed_kernelILb1ELb1ELb1", "render_kernelILb1ELb1ELb1"),
          ("render_listed_kernelILb0ELb0ELb0", "render_kernelILb0ELb0ELb0"),
          ("render_listed_kernelILb0ELb1ELb0", "render_kernelILb0ELb1ELb0"),
          ("render_lane2_listed_kernelILb0", "render_lane2_kernelILb0"),
          ("render_lane2_listed_kernelILb1", "render_lane2_kernelILb1"),
          ("render_primary_listed_kernelILb0", "render_primary_kernelILb0"),
          ("render_primary_listed_kernelILb1", "render_primary_kernelILb1"),
          ("render_primary_seeded_listed_kernelILb0", "render_primary_seeded_kernelILb0"),
          ("render_primary_seeded_listed_kernelILb1", "render_primary_seeded_kernelILb1")]


@pytest.mark.parametrize("key", [k for k, _ in LISTED if k.startswith(("render_listed_kernelILb1", "render_lane2_listed"))])
def test_small_scene_listed_kernels_cull_through_uniform_registers(sass, key):
    """As test_build_artifacts: the cull table reaches FFMA2 as uniform operands, never through per-lane LDC."""
    body = one(sass, key)
    uniform = [l for l in body if re.search(r"LDCU\.64 UR\d+, c\[0x0\]\[UR\d+", l)]
    per_lane = [l for l in body if re.search(r"LDC\.64 R\d+, c\[0x0\]\[R\d+", l)]
    assert len(uniform) >= 32 and not per_lane, (len(uniform), len(per_lane))
    assert sum("FFMA2" in l and ".F32x2" in l and " UR" in l for l in body) >= 48


@pytest.mark.parametrize("key", ["render_listed_kernelILb0ELb0ELb0", "render_listed_kernelILb0ELb1ELb0"])
def test_large_scene_listed_kernels_stage_the_table_by_tma(sass, key):
    body = one(sass, key)
    assert any("UBLKCP" in l for l in body) and any("SYNCS" in l for l in body)


@pytest.mark.parametrize("key,twin", LISTED, ids=[k for k, _ in LISTED])
def test_listed_kernels_fit_the_budget_of_their_twins(sass, key, twin):
    """The listed kernels add the list lookup (and the seeded ones the sums of squares): within 2 KB of their twin's
    code, and within the instruction
    cache budgets test_build_artifacts holds the twins to (34 KB for the chunked lane kernels, 40 / 44 KB for the
    primary-ray kernels)."""
    body, twin_body = one(sass, key), one(sass, twin)
    assert len(body) * 16 <= len(twin_body) * 16 + 2048, (key, len(body) * 16, len(twin_body) * 16)
    budget = {"render_listed_kernelILb1ELb0ELb0": 34, "render_listed_kernelILb1ELb0ELb1": 34,
              "render_lane2_listed_kernelILb0": 34, "render_primary_listed_kernelILb0": 40,
              "render_primary_listed_kernelILb1": 44, "render_primary_seeded_listed_kernelILb0": 40,
              "render_primary_seeded_listed_kernelILb1": 44}.get(key)
    if budget:
        assert len(body) * 16 <= budget * 1024, (key, len(body) * 16)


@pytest.mark.parametrize("key", [k for k, _ in LISTED if "primary" in k])
def test_primary_listed_kernels_keep_off_shared_and_local_memory(sass, key):
    """The list and its count are global loads (LDG); the sums stay in registers: no shared or local memory."""
    text = "\n".join(one(sass, key))
    assert not re.search(r"\b(LDS|LDL|STL|STS)\b", text), key
    assert re.search(r"\bLDG\b", text) and re.search(r"\bDFMA\b", text), key
    # one unit sum (three doubles); the seeded variant also stores the sums of squares
    assert len(re.findall(r"\bSTG\b", text)) == (6 if "seeded" in key else 3), key


def test_kernel_harness_compiles_against_the_header(tmp_path):
    """tests/native/adaptive_kernels.cu includes rtclj_adaptive.cuh as it is: a header change that breaks the
    kernel tests shows here, without a GPU.  Its mirror of AParams matches the compiler's layout."""
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import adaptive_kernels as K
    if K.nvcc() is None:
        pytest.skip("nvcc not installed")
    so = C.CDLL(K.build(str(tmp_path)))
    K.check_layout(so)
    assert so.ak_list_tile() == 2048
