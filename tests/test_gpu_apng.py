"""The animated PNG writer on the device (rtclj_ctx_encode_apng, rtclj_encode_apng_gpu, rtclj_render_frames_apng): byte
for byte the numpy model of its definition (tests/apng_model.py) on the model's cases, renders and a sequence encoded in
several groups; the same bytes through every entry point, device list and shard_rows; the capacity rules; the CLI."""
import ctypes as C
import io
import os
import subprocess
import sys

import numpy as np
import pytest
from PIL import Image

import apng_model as A
import raytracing_clj_b200 as R
from raytracing_clj_b200 import _abi, render

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = A.cpu_cases()


def n_devices():
    n = C.c_int()
    _abi.check(_abi.lib().rtclj_device_count(C.byref(n)))
    return n.value


def decoded_frames(data: bytes) -> np.ndarray:
    im = Image.open(io.BytesIO(data))
    out = []
    for k in range(im.n_frames):
        im.seek(k)
        out.append(np.array(im.convert("RGB")))
    return np.stack(out)


def check(frames, delay=(1, 30), plays=0):
    got = render.encode_apng(frames, device=0, delay=delay, plays=plays)
    want = A.encode(frames, delay, plays)
    assert len(got) == len(want) and got == want
    return got


@pytest.mark.parametrize("name", sorted(CASES))
def test_device_bytes_equal_the_model(name):
    frames, delay, plays = CASES[name]
    check(frames, delay, plays)


def turntable(n=60, spp=16, depth=50, width=400):
    return R.camera.turntable_cameras(n, width), spp, depth


def test_main_turntable_60_frames():
    cams, spp, depth = turntable()
    _, rgb, _ = render.render_frames(R.scenes.main_hittables(), cams, spp, depth, seed=1, want_linear=False)
    data = check(rgb)
    assert np.array_equal(decoded_frames(data), rgb)
    assert render.render_frames_apng(R.scenes.main_hittables(), cams, spp, depth, seed=1) == data


def test_cover_scene_8_frames_1080p():
    S, CAM = R.scenes, R.camera
    look = S.COVER_CAMERA["look_from"]
    args = {k: v for k, v in S.COVER_CAMERA.items() if k != "look_from"}
    cams = [CAM.main_camera(1920, 1080, look_from=CAM.turntable_look_from(k, 8, look, args["look_at"]), **args)
            for k in range(8)]
    _, rgb, _ = render.render_frames(S.cover_hittables(7), cams, 2, 8, seed=1, want_linear=False)
    check(rgb)


def test_8k_sequence_in_several_groups():
    """12 frames of 7680 x 4320: 199 MB of scratch per frame, so the 2 GiB cap makes groups of 10 and 2."""
    H, W = 4320, 7680
    y, x = np.mgrid[0:H, 0:W]
    grad = np.stack([(x // 30) % 256, (y // 17) % 256, ((x + y) // 64) % 256], axis=2).astype(np.uint8)
    const = np.full((H, W, 3), 200, np.uint8)
    distinct = [grad, const, np.ascontiguousarray(grad[::-1])]
    order = [k % 3 for k in range(12)]
    nseg = A.nseg(W, H)
    assert 12 * nseg * (65536 + 65552 + 16) > 2 << 30 > 10 * nseg * (65536 + 65552 + 16)
    frames = np.stack([distinct[k] for k in order])
    got = render.encode_apng(frames, device=0)
    per = [A.frame_chunks(d) for d in distinct]
    assert got == A.assemble([per[k] for k in order], W, H)


def test_entry_points_agree_and_capacity_rules():
    import torch
    frames, delay, plays = CASES["K3_main_shifted"]
    K, H, W, _ = frames.shape
    want = A.encode(frames, delay, plays)
    lib = _abi.lib()
    # host buffers: sizing, exact, one byte short
    img = np.ascontiguousarray(frames)
    n = C.c_size_t()
    _abi.check(lib.rtclj_encode_apng_gpu(0, img.ctypes.data, W, H, K, 1, 30, 0, None, 0, C.byref(n)))
    assert n.value == A.stored_bound(W, H, K) >= len(want)
    buf = (C.c_char * len(want))()
    _abi.check(lib.rtclj_encode_apng_gpu(0, img.ctypes.data, W, H, K, 1, 30, 0, buf, len(want), C.byref(n)))
    assert n.value == len(want) and bytes(buf) == want
    n = C.c_size_t(0)
    assert lib.rtclj_encode_apng_gpu(0, img.ctypes.data, W, H, K, 1, 30, 0, buf, len(want) - 1, C.byref(n)) == _abi.E_BUFFER
    assert n.value == len(want)
    # device buffers: sizing, the bound, exact, one byte short
    ctx = render.Context(0)
    stream = torch.cuda.current_stream().cuda_stream
    d_in = torch.from_numpy(img).cuda()
    cap = ctx.encode_apng(d_in.data_ptr(), W, H, K)
    assert cap == A.stored_bound(W, H, K)
    d_out = torch.zeros(cap, dtype=torch.uint8, device="cuda:0")
    got = ctx.encode_apng(d_in.data_ptr(), W, H, K, d_out.data_ptr(), cap, stream=stream)
    assert bytes(d_out[:got].cpu().numpy()) == want
    d_tight = torch.zeros(len(want), dtype=torch.uint8, device="cuda:0")
    assert ctx.encode_apng(d_in.data_ptr(), W, H, K, d_tight.data_ptr(), len(want), stream=stream) == len(want)
    assert bytes(d_tight.cpu().numpy()) == want
    n = C.c_size_t(0)
    assert lib.rtclj_ctx_encode_apng(ctx._h, C.c_void_p(d_in.data_ptr()), W, H, K, 1, 30, 0,
                                     C.c_void_p(d_tight.data_ptr()), len(want) - 1, C.byref(n), None) == _abi.E_BUFFER
    assert n.value == len(want)
    ctx.close()
    # render + encode: sizing, exact, one byte short
    world = R.scenes.main_hittables()
    cams = R.camera.turntable_cameras(3, 64)
    _, rgb, _ = render.render_frames(world, cams, 4, 8, seed=2, want_linear=False)
    data = render.render_frames_apng(world, cams, 4, 8, seed=2)
    assert data == render.encode_apng(rgb) == A.encode(rgb)
    sc = render._scene_struct(render._as_soa(world))
    arr, k = render._camera_array(cams)
    prm = _abi.Params(4, 8, 2, _abi.FLAGS_MAIN, 0, 0, 0, 0, 0, 0)
    devs = (C.c_int32 * 1)(0)
    n = C.c_size_t()
    _abi.check(lib.rtclj_render_frames_apng(C.byref(sc), arr, k, C.byref(prm), 1, 30, 0, devs, 1, None, 0, C.byref(n),
                                            None))
    assert n.value == A.stored_bound(64, 36, 3)
    buf = (C.c_char * len(data))()
    _abi.check(lib.rtclj_render_frames_apng(C.byref(sc), arr, k, C.byref(prm), 1, 30, 0, devs, 1, buf, len(data),
                                            C.byref(n), None))
    assert bytes(buf) == data
    assert lib.rtclj_render_frames_apng(C.byref(sc), arr, k, C.byref(prm), 1, 30, 0, devs, 1, buf, len(data) - 1,
                                        C.byref(n), None) == _abi.E_BUFFER
    assert n.value == len(data)


@pytest.mark.parametrize("devices", [[0], [0, 1]])
@pytest.mark.parametrize("shard_rows", [0, 1, 7, 64])
def test_render_frames_apng_equals_encoding_the_rendered_frames(devices, shard_rows):
    if n_devices() < len(devices):
        pytest.skip("needs two GPUs")
    world = R.scenes.main_hittables()
    cams = R.camera.turntable_cameras(5, 160)
    _, rgb, _ = render.render_frames(world, cams, 8, 20, seed=3, want_linear=False)
    data = render.render_frames_apng(world, cams, 8, 20, seed=3, devices=devices, shard_rows=shard_rows,
                                     delay=(1, 24), plays=2)
    assert data == render.encode_apng(rgb, device=0, delay=(1, 24), plays=2)
    assert np.array_equal(decoded_frames(data), rgb)


def test_cli_apng(tmp_path):
    env = dict(os.environ, PYTHONPATH=ROOT)
    for sub, extra in (("apng", ["--apng"]), ("pngs", [])):
        d = tmp_path / sub
        d.mkdir()
        subprocess.run([sys.executable, "-m", "raytracing_clj_b200.main", "main", "4", "5", "--frames", "8", *extra],
                       cwd=d, env=env, check=True, capture_output=True)
    assert sorted(p.name for p in (tmp_path / "apng").iterdir()) == ["scene.apng"]
    data = (tmp_path / "apng" / "scene.apng").read_bytes()
    im = Image.open(io.BytesIO(data))
    assert im.n_frames == 8 and im.info.get("loop") == 0 and im.info.get("duration") == pytest.approx(1000 / 30)
    frames = decoded_frames(data)
    for k in range(8):
        png = np.array(Image.open(tmp_path / "pngs" / f"scene-{k:04d}.png").convert("RGB"))
        assert np.array_equal(frames[k], png), k
