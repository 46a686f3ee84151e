"""The denoiser on the device (rtclj_ctx_denoise, rtclj_denoise_gpu, rtclj_render_denoised): bit for bit the numpy
model of its definition (tests/denoise_model.py), linear and 8-bit, through every entry point, on every device list,
and on inputs that hold NaN and infinities."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import denoise_model as M
import test_gpu_degenerate_rays as D
import raytracing_clj_b200 as R
from raytracing_clj_b200 import _abi, main, render

pytestmark = pytest.mark.gpu
QL = _abi.F_QUANT_LINEAR


def n_devices():
    n = C.c_int()
    _abi.check(_abi.lib().rtclj_device_count(C.byref(n)))
    return n.value


def same_bits(a, b):
    return np.array_equal(np.asarray(a, np.float64).view(np.int64), np.asarray(b, np.float64).view(np.int64))


def noisy(H, W, seed, specials=True):
    """A piecewise-smooth colour with noise, a guide with an edge, and (specials) NaN / inf / beyond-float32 values."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:H, 0:W]
    G = np.stack([(x > W // 3).astype(float), 0.5 + 0.4 * np.sin(y / 7.0), (x + y) % 29 / 29.0], axis=2)
    Cimg = 0.6 * G + rng.normal(0, 0.15, (H, W, 3))
    if specials and H * W > 8:
        for img, vals in ((Cimg, [np.nan, np.inf, -np.inf, 1e39, -0.0]), (G, [np.nan, np.inf])):
            idx = rng.integers(0, H * W, size=len(vals))
            for i, v in zip(idx, vals):
                img[i // W, i % W, rng.integers(0, 3)] = v
    return np.ascontiguousarray(Cimg), np.ascontiguousarray(G)


def check(Cimg, G, levels, sc=0.8, sg=0.2, flags=0, device=0):
    lin, rgb = render.denoise(Cimg, G, device=device, levels=levels, sigma_color=sc, sigma_guide=sg, flags=flags)
    want_lin, want_rgb = M.denoise(Cimg, G, levels, sc, sg, flags)
    assert same_bits(lin, want_lin), f"L={levels} {Cimg.shape}: linear differs"
    assert np.array_equal(rgb, want_rgb), f"L={levels} {Cimg.shape}: 8-bit differs"


@pytest.mark.parametrize("H,W", [(1, 1), (1, 7), (7, 1), (3, 3), (225, 400)])
@pytest.mark.parametrize("levels", range(1, 9))
def test_equals_the_model(H, W, levels):
    Cimg, G = noisy(H, W, H * 1000 + W + levels)
    for flags in (0, QL):
        check(Cimg, G, levels, flags=flags)


@pytest.mark.parametrize("levels", [1, 5, 8])
def test_equals_the_model_at_1080p(levels):
    Cimg, G = noisy(1080, 1920, levels)
    check(Cimg, G, levels, flags=QL if levels == 8 else 0)


def test_8k_on_row_bands():
    """7680x4320: the model runs on bands plus the filter's reach of 2 (2^L - 1) rows on either side."""
    H, W, L = 4320, 7680, 5
    Cimg, G = noisy(H, W, 8)
    lin, rgb = render.denoise(Cimg, G, levels=L, sigma_color=0.8, sigma_guide=0.2)
    reach = 2 * (2 ** L - 1)
    for y0, y1 in ((0, 40), (2150, 2190), (H - 40, H)):
        a, b = max(0, y0 - reach), min(H, y1 + reach)
        want_lin, want_rgb = M.denoise(Cimg[a:b], G[a:b], L, 0.8, 0.2)
        assert same_bits(lin[y0:y1], want_lin[y0 - a:y1 - a]), (y0, y1)
        assert np.array_equal(rgb[y0:y1], want_rgb[y0 - a:y1 - a]), (y0, y1)


@pytest.mark.parametrize("levels", [1, 3])
def test_context_entry_point_in_place_and_without_outputs(levels):
    H, W = 61, 83
    Cimg, G = noisy(H, W, levels)
    want_lin, want_rgb = M.denoise(Cimg, G, levels, 0.8, 0.2, QL)
    ctx = render.Context(0)
    try:
        s = torch.cuda.current_stream().cuda_stream
        lin, gd = torch.from_numpy(Cimg).cuda(), torch.from_numpy(G).cuda()
        out, rgb = torch.empty_like(lin), torch.zeros(lin.shape, dtype=torch.uint8, device="cuda")
        kw = dict(levels=levels, sigma_color=0.8, sigma_guide=0.2, flags=QL, stream=s)
        ctx.denoise(lin.data_ptr(), gd.data_ptr(), W, H, d_out_linear=out.data_ptr(), d_out_rgb8=rgb.data_ptr(), **kw)
        torch.cuda.synchronize()
        assert same_bits(out.cpu().numpy(), want_lin) and np.array_equal(rgb.cpu().numpy(), want_rgb)
        rgb.zero_()
        ctx.denoise(lin.data_ptr(), gd.data_ptr(), W, H, d_out_rgb8=rgb.data_ptr(), **kw)  # no linear output
        torch.cuda.synchronize()
        assert np.array_equal(rgb.cpu().numpy(), want_rgb)
        ctx.denoise(lin.data_ptr(), gd.data_ptr(), W, H, d_out_linear=lin.data_ptr(), **kw)  # in place
        torch.cuda.synchronize()
        assert same_bits(lin.cpu().numpy(), want_lin)
    finally:
        ctx.close()


def test_every_device():
    Cimg, G = noisy(90, 160, 3)
    for dev in range(n_devices()):
        check(Cimg, G, 4, device=dev)


def device_lists():
    n = n_devices()
    return [[0]] + ([list(range(n)), list(range(n))[::-1]] if n > 1 else [])


def test_render_denoised_equals_render_guide_and_filter():
    """The guide is render(flags=FLAGS_I, max_depth=1, spp=guide_samples); the output is identical for every device
    list and shard_rows."""
    world = R.scenes.cover_hittables(7)
    cam = R.camera.main_camera(320, 180, **R.scenes.COVER_CAMERA)
    colour, _, _ = render.render(world, cam, 8, 50, seed=5)
    guide, _, _ = render.render(world, cam, 3, 1, seed=5, flags=_abi.FLAGS_I)
    want_lin, want_rgb = M.denoise(colour, guide, 4, 0.9, 0.15)
    for devs in device_lists():
        for rows in (0, 1, 7, 64):
            lin, rgb, st = render.render_denoised(world, cam, 8, 50, seed=5, devices=devs, shard_rows=rows,
                                                  guide_samples=3, levels=4, sigma_color=0.9, sigma_guide=0.15)
            assert same_bits(lin, want_lin), (devs, rows)
            assert np.array_equal(rgb, want_rgb), (devs, rows)
            assert st["samples"] == 8 * 320 * 180 and st["total_ms"] > 0


def test_render_denoised_with_a_kernel_choice_and_linear_quantisation():
    world, cam = R.scenes.main_hittables(), R.camera.main_camera(200, 112)
    flags = _abi.FLAGS_MAIN | QL | _abi.F_LANE_KERNEL
    colour, _, _ = render.render(world, cam, 6, 20, seed=9, flags=flags)
    guide, _, _ = render.render(world, cam, 2, 1, seed=9, flags=_abi.FLAGS_I | _abi.F_LANE_KERNEL)
    want_lin, want_rgb = M.denoise(colour, guide, 3, 1.0, 0.2, QL)
    lin, rgb, _ = render.render_denoised(world, cam, 6, 20, seed=9, flags=flags, guide_samples=2, levels=3,
                                         sigma_color=1.0, sigma_guide=0.2)
    assert same_bits(lin, want_lin) and np.array_equal(rgb, want_rgb)


@pytest.mark.parametrize("case", ["d0", "huge-1e200"])
def test_nan_inputs_from_degenerate_cameras(case):
    """Renders of the degenerate-camera scenes hold NaN pixels; the filter keeps them and never uses them as taps."""
    scene, cam = D.CAMERA_CASES[case]
    sc = D.world(scene)
    colour, _, _ = render.render(sc, cam, 4, 10, seed=3, flags=_abi.FLAGS_MAIN)
    guide, _, _ = render.render(sc, cam, 2, 1, seed=3, flags=_abi.FLAGS_I)
    nan_in = np.isnan(colour).any() or np.isnan(guide).any()
    # the same pixels spliced into a larger ordinary image, so that finite neighbours surround them
    bigC, bigG = noisy(24, 40, 1, specials=False)
    bigC[10:10 + cam.height, 16:16 + cam.width] = colour
    bigG[10:10 + cam.height, 16:16 + cam.width] = guide
    for L in (1, 3):
        check(colour, guide, L)
        check(bigC, bigG, L, flags=QL)
    assert nan_in, "the case was chosen for its NaN pixels"


def test_quality_on_the_default_scene():
    """main's default scene (400x225): the denoised 8-spp image is closer to a 1024-spp render with another seed than
    a raw 32-spp render is (measured on a B200 at 1000 W: RMSE ratio 0.61, profiles/r3_bench_denoise.json)."""
    world, cam = R.scenes.main_hittables(), R.camera.main_camera()
    ref, _, _ = render.render(world, cam, 1024, 50, seed=2, want_rgb8=False)
    raw32, _, _ = render.render(world, cam, 32, 50, seed=1, want_rgb8=False)
    dn, _, _ = render.render_denoised(world, cam, 8, 50, seed=1)
    rmse = lambda a: float(np.sqrt(np.mean((a - ref) ** 2)))  # noqa: E731
    assert rmse(dn) < rmse(raw32), (rmse(dn), rmse(raw32))


@pytest.mark.parametrize("every", [0, 4])
def test_cli_writes_denoised_images(tmp_path, every):
    """main --denoise (and --every N --denoise): scene-denoised.ppm / .png hold the filter of the render with its guide;
    scene.ppm is the file a run without --denoise writes."""
    out = str(tmp_path / "scene.ppm")
    main.main_variant(12, 10, out=out, every=every, denoise=True)
    lin, rgb8, _ = render.render(R.scenes.main_hittables(), R.camera.main_camera(), 12, 10, seed=1)
    guide, _, _ = render.render(R.scenes.main_hittables(), R.camera.main_camera(), render.DENOISE_GUIDE_SAMPLES, 1,
                                seed=1, flags=_abi.FLAGS_I)
    _, want = M.denoise(lin, guide, render.DENOISE_LEVELS, render.DENOISE_SIGMA_COLOR, render.DENOISE_SIGMA_GUIDE)
    with open(out, "rb") as f:
        assert f.read() == render.encode_ppm(rgb8)
    with open(str(tmp_path / "scene-denoised.ppm"), "rb") as f:
        assert np.array_equal(render.decode_ppm(f.read()), want)
    assert os.path.getsize(str(tmp_path / "scene-denoised.png")) > 0
