"""Progressive rendering without a GPU: the entry points refuse to run without a device (no CPU fallback),
the Clojure shim binds them, and the seeded primary-ray kernel is built like its unseeded twin."""
import ctypes as C
import os
import re
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "raytracing-clj_b200", "librtclj_b200.so")
CLJ = os.path.join(ROOT, "integration", "clojure", "src", "rtclj", "native.clj")


def check_progressive_needs_a_device():
    import raytracing_clj_b200 as R
    from raytracing_clj_b200 import _abi, render
    lib = _abi.lib()
    world, cam = R.scenes.main_hittables(), R.camera.main_camera(16)
    sc, cm = render._scene_struct(R.scenes.to_soa(world)), render._camera_struct(cam)
    prm = _abi.Params(4, 5, 1, _abi.FLAGS_MAIN, 0, 0, 0, 0, 0, 0)
    devices = (C.c_int32 * 1)(0)
    unit, handle = C.c_int32(), C.c_void_p()
    rc = lib.rtclj_progressive_create(C.byref(sc), C.byref(cm), C.byref(prm), devices, 1, C.byref(unit), C.byref(handle))
    assert rc == _abi.E_NO_DEVICE and not handle.value, rc
    assert lib.rtclj_last_error() != b""
    with pytest.raises(_abi.RtcljError) as e:
        render.Progressive(world, cam, 4, 5)
    assert e.value.code == _abi.E_NO_DEVICE
    # a null handle is refused without touching a device; destroying NULL is a no-op
    assert lib.rtclj_progressive_step(None, 1, None, None, None, None) == _abi.E_INVALID
    assert lib.rtclj_progressive_destroy(None) == 0
    assert lib.rtclj_ctx_accum_step(None, 1, None, None, None, None) == _abi.E_INVALID


def test_progressive_render_fails_without_a_device():
    """In a child process that sees no CUDA device, so that it runs on machines with a GPU as well."""
    code = "import sys; sys.path[:0] = sys.argv[1:]; import test_progressive; test_progressive.check_progressive_needs_a_device()"
    subprocess.run([sys.executable, "-c", code, ROOT, os.path.join(ROOT, "tests")], check=True,
                   env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))


def test_clojure_shim_binds_the_progressive_entry_points():
    text = open(CLJ).read()
    bound = set(re.findall(r'\(downcall "(\w+)"', text))
    assert {"rtclj_progressive_create", "rtclj_progressive_step", "rtclj_progressive_destroy"} <= bound
    for fn in ("progressive", "progressive-step!", "progressive-close!"):
        assert re.search(r"\(defn %s\s" % re.escape(fn), text), fn


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not installed")
def test_seeded_primary_kernel_is_built_like_its_twin():
    """render_primary_seeded_kernel loads the running sums once per pixel (LDG) and otherwise keeps
    render_primary_kernel's properties: no shared / local memory, no spills, the same i-cache budget."""
    out = subprocess.run(["cuobjdump", "-sass", LIB], check=True, capture_output=True, text=True).stdout
    funcs, name = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            funcs[name] = []
        elif name and re.match(r"\s+/\*[0-9a-f]{4,}\*/\s", line):
            funcs[name].append(line)
    for key, budget in (("render_primary_seeded_kernelILb0", 40), ("render_primary_seeded_kernelILb1", 44)):
        names = [n for n in funcs if key in n]
        assert len(names) == 1, (key, names)
        body = funcs[names[0]]
        text = "\n".join(body)
        assert not re.search(r"\b(LDS|LDL|STL|STS)\b", text), key
        assert re.search(r"\bLDG\b", text), key          # the seed: the pixel's running sums
        assert len(re.findall(r"\bSTG\b", text)) == 3, key  # one unit sum: three doubles
        assert len(body) * 16 <= budget * 1024, (key, len(body) * 16)
