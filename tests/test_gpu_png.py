"""The compressed PNG writer on the device (rtclj_ctx_encode_png, rtclj_encode_png_gpu, rtclj_render_multi_png):
byte for byte the numpy model of its definition (tests/png_model.py), decodable to the input, the same through
every entry point and on every device."""
import ctypes as C
import io
import os
import subprocess
import sys

import numpy as np
import pytest
from PIL import Image

import png_model as M
import raytracing_clj_b200 as R
from raytracing_clj_b200 import _abi, render

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = M.cpu_cases()


def n_devices():
    n = C.c_int()
    _abi.check(_abi.lib().rtclj_device_count(C.byref(n)))
    return n.value


def decoded(png: bytes) -> np.ndarray:
    return np.array(Image.open(io.BytesIO(png)).convert("RGB"))


def check(img, dev=0):
    got = render.encode_png(img, device=dev)
    want = M.encode(img)
    assert len(got) == len(want) and got == want
    assert np.array_equal(decoded(got), img)
    return got


@pytest.mark.parametrize("name", sorted(CASES))
def test_device_bytes_equal_the_model(name):
    check(CASES[name])


def main_render():
    return render.render(R.scenes.main_hittables(), R.camera.main_camera(), 100, 50, seed=1, want_linear=False)[1]


def test_main_scene_render():
    check(main_render())


def test_cover_render_1080p():
    cam = R.camera.main_camera(1920, 1080, **R.scenes.COVER_CAMERA)
    img = render.render(R.scenes.cover_hittables(7), cam, 2, 8, seed=1, want_linear=False)[1]
    check(img)


def test_config4_render_4k():
    img = render.render(R.scenes.i_hittables(), R.camera.i_camera(3840), 4, 50, seed=1, flags=_abi.FLAGS_I,
                        want_linear=False)[1]
    assert img.shape == (2160, 3840, 3)
    check(img)


@pytest.mark.parametrize("kind", ["noise", "constant"])
def test_8k_images_larger_than_l2(kind):
    if kind == "noise":
        img = np.random.default_rng(3).integers(0, 256, (4320, 7680, 3), dtype=np.uint8)
    else:
        img = np.full((4320, 7680, 3), 200, dtype=np.uint8)
    got = check(img)
    if kind == "noise":
        assert len(got) > img.size
    else:
        assert len(got) < img.size // 100


def test_entry_points_and_devices_agree():
    import torch
    img = CASES["scene_main"]
    H, W, _ = img.shape
    want = render.encode_png(img, device=0)
    assert render.encode_png(img, device=0) == want  # a second call on the cached context
    ctx = render.Context(0)
    stream = torch.cuda.current_stream().cuda_stream
    d_img = torch.from_numpy(img).cuda()
    cap = ctx.encode_png(d_img.data_ptr(), W, H)
    assert cap == M.stored_bound(W, H)
    d_out = torch.zeros(cap, dtype=torch.uint8, device="cuda:0")
    n = ctx.encode_png(d_img.data_ptr(), W, H, d_out.data_ptr(), cap, stream)
    assert bytes(d_out[:n].cpu().numpy()) == want
    # a tight buffer: the exact length first, then the bytes
    d_tight = torch.zeros(n, dtype=torch.uint8, device="cuda:0")
    assert ctx.encode_png(d_img.data_ptr(), W, H, d_tight.data_ptr(), n, stream) == n
    assert bytes(d_tight.cpu().numpy()) == want
    ctx.close()
    if n_devices() >= 2:
        assert render.encode_png(img, device=1) == want


def test_capacity_and_sizing():
    lib = _abi.lib()
    for name in ("scene_main", "noise", "constant", "1x1"):
        img = np.ascontiguousarray(CASES[name])
        H, W, _ = img.shape
        exact = len(M.encode(img))
        n = C.c_size_t()
        _abi.check(lib.rtclj_encode_png_gpu(0, img.ctypes.data, W, H, None, 0, C.byref(n)))
        assert n.value >= exact and n.value == M.stored_bound(W, H)
        buf = (C.c_char * exact)()
        n = C.c_size_t(0)
        assert lib.rtclj_encode_png_gpu(0, img.ctypes.data, W, H, buf, exact - 1, C.byref(n)) == _abi.E_BUFFER
        assert n.value == exact
    import torch
    img = CASES["scene_realm"]
    H, W, _ = img.shape
    exact = len(M.encode(img))
    ctx = render.Context(0)
    d_img = torch.from_numpy(img).cuda()
    d_out = torch.zeros(exact, dtype=torch.uint8, device="cuda:0")
    with pytest.raises(_abi.RtcljError) as e:
        ctx.encode_png(d_img.data_ptr(), W, H, d_out.data_ptr(), exact - 1)
    assert e.value.code == _abi.E_BUFFER
    n = C.c_size_t(0)
    assert lib.rtclj_ctx_encode_png(ctx._h, C.c_void_p(d_img.data_ptr()), W, H, C.c_void_p(d_out.data_ptr()),
                                    exact - 1, C.byref(n), None) == _abi.E_BUFFER
    assert n.value == exact
    for w, h in ((0, 5), (5, 0), (-1, 5)):
        assert lib.rtclj_ctx_encode_png(ctx._h, C.c_void_p(d_img.data_ptr()), w, h, C.c_void_p(d_out.data_ptr()),
                                        exact, C.byref(n), None) == _abi.E_INVALID
    assert lib.rtclj_ctx_encode_png(ctx._h, None, W, H, C.c_void_p(d_out.data_ptr()), exact, C.byref(n),
                                    None) == _abi.E_INVALID
    ctx.close()


@pytest.mark.parametrize("ndev", [1, 2])
def test_render_multi_png(ndev):
    if n_devices() < ndev:
        pytest.skip("needs two GPUs")
    world, cam = R.scenes.main_hittables(), R.camera.main_camera()
    _, rgb, _ = render.render(world, cam, 16, 50, seed=4, want_linear=False)
    png, st = render.render_png(world, cam, 16, 50, seed=4, devices=list(range(ndev)))
    assert st["n_devices"] == ndev
    assert png == render.encode_png(rgb, device=0)
    assert np.array_equal(decoded(png), rgb)
    n = C.c_size_t()
    sc, cm = render._scene_struct(render._as_soa(world)), render._camera_struct(cam)
    prm = _abi.Params(16, 50, 4, _abi.FLAGS_MAIN, 0, 0, 0, 0, 0, 0)
    arr = (C.c_int32 * 1)(0)
    _abi.check(_abi.lib().rtclj_render_multi_png(C.byref(sc), C.byref(cm), C.byref(prm), arr, 1, None, 0, C.byref(n),
                                                 None))
    assert n.value == M.stored_bound(cam.width, cam.height) >= len(png)
    buf = (C.c_char * len(png))()
    assert _abi.lib().rtclj_render_multi_png(C.byref(sc), C.byref(cm), C.byref(prm), arr, 1, buf, len(png) - 1,
                                             C.byref(n), None) == _abi.E_BUFFER
    assert n.value == len(png)


def test_encoding_mid_accumulation_leaves_the_next_pass_unchanged():
    import torch
    world, cam = R.scenes.main_hittables(), R.camera.main_camera()
    H, W = cam.height, cam.width
    outs = []
    for encode in (False, True):
        ctx = render.Context(0)
        ctx.set_scene(world)
        stream = torch.cuda.current_stream().cuda_stream
        lin = torch.zeros((H, W, 3), dtype=torch.float64, device="cuda:0")
        rgb = torch.zeros((H, W, 3), dtype=torch.uint8, device="cuda:0")
        ctx.accum_begin(cam, 24, 50, seed=2, samples_per_unit=4, stream=stream)
        ctx.accum_step(8, lin.data_ptr(), rgb.data_ptr(), stream)
        if encode:
            cap = ctx.encode_png(rgb.data_ptr(), W, H)
            d_out = torch.zeros(cap, dtype=torch.uint8, device="cuda:0")
            n = ctx.encode_png(rgb.data_ptr(), W, H, d_out.data_ptr(), cap, stream)
            assert bytes(d_out[:n].cpu().numpy()) == M.encode(rgb.cpu().numpy())
        ctx.accum_step(8, lin.data_ptr(), rgb.data_ptr(), stream)
        torch.cuda.synchronize()
        outs.append((lin.cpu().numpy().copy(), rgb.cpu().numpy().copy()))
        ctx.close()
    assert np.array_equal(outs[0][0].view(np.uint64), outs[1][0].view(np.uint64))
    assert np.array_equal(outs[0][1], outs[1][1])


def test_cli_gpu_png(tmp_path):
    env = dict(os.environ, PYTHONPATH=ROOT)
    for sub, extra in (("once", []), ("every", ["--every", "4", "--tolerance", "0.01,0.05"])):
        d = tmp_path / sub
        d.mkdir()
        subprocess.run([sys.executable, "-m", "raytracing_clj_b200.main", "main", "12", "10", "--gpu-png", *extra],
                       cwd=d, env=env, check=True, capture_output=True)
        ppm = render.decode_ppm((d / "scene.ppm").read_bytes())
        png = (d / "scene.png").read_bytes()
        assert np.array_equal(decoded(png), ppm)
        assert png == M.encode(ppm)
        if extra:
            samples = (d / "scene-samples.png").read_bytes()
            assert samples == M.encode(decoded(samples))
