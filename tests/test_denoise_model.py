"""The denoiser's definition on the CPU (include/rtclj_b200.h, DESIGN.md section 4.13): the vectorised numpy model
against an independent per-pixel loop, hand-worked cases at the edges of the definition, and the library's refusals,
which it decides before any device call."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import denoise_model as M  # noqa: E402
from raytracing_clj_b200 import _abi, camera, render, scenes  # noqa: E402

F32 = np.float32


def same_bits(a, b):
    """Equal as float64 bit patterns (NaN == NaN, +0 != -0)."""
    return np.array_equal(np.asarray(a, np.float64).view(np.int64), np.asarray(b, np.float64).view(np.int64))


def rand_images(rng, H, W, specials=False):
    C = rng.random((H, W, 3)) * 1.5
    G = rng.random((H, W, 3))
    G[:, : W // 2] *= 0.2  # an edge in the guide
    if specials:
        for img, vals in ((C, [np.nan, np.inf, -np.inf, 1e39]), (G, [np.nan, -np.inf])):
            idx = rng.integers(0, H * W, size=len(vals))
            for i, v in zip(idx, vals):
                img[i // W, i % W, rng.integers(0, 3)] = v
    return C, G


@pytest.mark.parametrize("H,W,levels,specials", [(5, 7, 1, False), (6, 5, 2, True), (9, 4, 3, False),
                                                 (7, 8, 3, True), (3, 3, 8, True), (1, 7, 4, False),
                                                 (7, 1, 4, True)])
def test_model_equals_the_per_pixel_loop(H, W, levels, specials):
    rng = np.random.default_rng(1000 * H + 10 * W + levels)
    C, G = rand_images(rng, H, W, specials)
    lin, _ = M.denoise(C, G, levels, 0.7, 0.15)
    assert same_bits(lin, M.denoise_scalar(C, G, levels, 0.7, 0.15))


def test_the_filter_smooths_and_keeps_edges():
    rng = np.random.default_rng(5)
    H, W = 32, 32
    G = np.zeros((H, W, 3))
    G[:, 16:] = 1.0  # two regions
    truth = np.where(np.arange(W)[None, :, None] >= 16, 0.8, 0.2) * np.ones((H, W, 3))
    C = truth + rng.normal(0, 0.1, (H, W, 3))
    lin, _ = M.denoise(C, G, 4, 1.0, 0.2)
    assert np.sqrt(np.mean((lin - truth) ** 2)) < 0.3 * np.sqrt(np.mean((C - truth) ** 2))
    assert np.all(lin[:, :16] < 0.5) and np.all(lin[:, 16:] > 0.5)  # nothing leaks across the guide's edge


def test_hand_worked_three_pixels_in_tap_order():
    """1x3 at L = 1: the row dy = 0 only (h = 3/8), taps dx = -2 .. 2 in that order, those outside the image skipped."""
    C = np.array([[[0.1, 0.2, 0.3], [0.5, 0.25, 0.0], [0.9, 0.6, 0.3]]])
    G = np.zeros((1, 3, 3))
    sc, sg = 2.0, 1.0
    lin, _ = M.denoise(C, G, 1, sc, sg)
    with np.errstate(over="ignore"):
        c = C.astype(F32)
    sc2 = F32(sc) * F32(sc)
    hy = F32(0.375)

    def w_of(p, q, hx):
        d = c[0, q] - c[0, p]
        dc = (d[0] * d[0] + d[1] * d[1]) + d[2] * d[2]
        t = max(F32(1) - dc / sc2, F32(0))
        return ((hx * hy) * (t * t)) * F32(1)  # the guide is flat: k(0) = 1

    for p in range(3):
        acc, W = np.zeros(3, F32), F32(0)
        for q, hx in zip(range(p - 2, p + 3), (F32(1 / 16), F32(0.25), F32(0.375), F32(0.25), F32(1 / 16))):
            if 0 <= q < 3:
                w = w_of(p, q, hx)
                acc = acc + w * c[0, q]
                W = W + w
        assert same_bits(lin[0, p], (acc / W).astype(np.float64)), p


@pytest.mark.parametrize("H,W", [(1, 1), (1, 7), (7, 1), (3, 3)])
def test_steps_beyond_the_image_clip_to_the_centre(H, W):
    """At steps >= the image size only the centre tap is left: c_(i+1) = (w c) / w with w = 9/64 * k * k."""
    rng = np.random.default_rng(H * 10 + W)
    C, G = rand_images(rng, H, W)
    lin, _ = M.denoise(C, G, 8, 0.5, 0.3)
    c = M.denoise(C, G, 2, 0.5, 0.3)[0].astype(F32)  # levels 0 and 1 (steps 1, 2) still see neighbours
    w = F32(9.0 / 64.0)
    for _ in range(2, 8):
        c = (w * c) / w
    assert same_bits(lin, c.astype(np.float64))
    assert same_bits(lin, M.denoise_scalar(C, G, 8, 0.5, 0.3))


def test_non_finite_centres_keep_their_input_and_are_never_taps():
    rng = np.random.default_rng(7)
    C, G = rand_images(rng, 6, 6)
    C[2, 3] = [np.nan, 0.5, 0.5]
    C[4, 1] = [0.1, np.inf, 0.2]
    C[0, 0] = [1e39, 0.0, 0.0]  # finite in f64, inf in float32
    G[5, 5] = [-np.inf, 0.0, 0.0]
    lin, rgb = M.denoise(C, G, 3, 0.8, 0.3)
    for y, x in ((2, 3), (4, 1), (0, 0), (5, 5)):
        assert same_bits(lin[y, x], C[y, x])  # the input double, not its float32
    # never a tap: the other pixels are those of an image where the four hold values so far off that k gives them
    # weight 0 -- and not those of one where they hold ordinary values
    keep = np.ones((6, 6), bool)
    keep[[2, 4, 0, 5], [3, 1, 0, 5]] = False
    far, near = C.copy(), C.copy()
    for y, x in ((2, 3), (4, 1), (0, 0)):
        far[y, x], near[y, x] = [123.0, -5.0, 7.0], [0.6, 0.6, 0.6]
    G_far = G.copy()
    G_far[5, 5] = [50.0, 0.0, 0.0]
    assert np.all(np.isfinite(lin[keep]))
    assert same_bits(lin[keep], M.denoise(far, G_far, 3, 0.8, 0.3)[0][keep])
    assert not same_bits(lin[keep], M.denoise(near, G, 3, 0.8, 0.3)[0][keep])
    assert rgb[2, 3, 0] == 0  # write-color! of NaN


def test_squared_differences_that_overflow_give_zero_weight():
    """3e38 next to -3e38: the difference is inf in float32, k(inf) = fmax(-inf, 0)^2 = 0, so each pixel sees only
    itself and keeps (w c) / w."""
    C = np.array([[[3e38, 0, 0], [-3e38, 0, 0]]])
    G = np.zeros((1, 2, 3))
    lin, _ = M.denoise(C, G, 1, 1.0, 1.0)
    w = F32(9.0 / 64.0)
    assert same_bits(lin[0, :, 0], ((w * C[0, :, 0].astype(F32)) / w).astype(np.float64))
    assert same_bits(lin, M.denoise_scalar(C, G, 1, 1.0, 1.0))


def test_float32_sums_that_overflow_become_non_finite_floats():
    """Two neighbours at 3.4e38 sum past the float32 range: the pixel is filtered into inf and kept so."""
    C = np.full((1, 3, 3), 3.4e38)
    G = np.zeros((1, 3, 3))
    lin, _ = M.denoise(C, G, 2, 1e19, 1.0)
    assert same_bits(lin, M.denoise_scalar(C, G, 2, 1e19, 1.0))
    assert np.all(np.isfinite(lin)) or np.any(np.isinf(lin))


def test_signed_zeros():
    C = np.full((2, 2, 3), -0.0)
    G = np.zeros((2, 2, 3))
    lin, rgb = M.denoise(C, G, 2, 1.0, 1.0)
    assert same_bits(lin, np.zeros((2, 2, 3)))  # 0 + w * -0 = +0
    assert np.all(rgb == 0)


def test_quantise_matches_the_library_write_color():
    rng = np.random.default_rng(3)
    v = np.concatenate([rng.random(1000) * 1.2 - 0.1, [0.0, -0.0, 1.0, 0.999 ** 2, 1 / 255.999, np.nan]])
    for flags in (0, _abi.F_QUANT_LINEAR):
        assert np.array_equal(M.quantise(v, bool(flags)), render.quantise_rgb8(v, flags))


# ---- refusals: decided on the host before any device call (RTCLJ_E_INVALID), else the call goes on to the device
FLT_MIN = float(np.finfo(np.float32).tiny)
EDGE = float(np.sqrt(np.float64(FLT_MIN))) * 128  # (EDGE 2^-7)^2 ~ FLT_MIN

REFUSALS = [  # width, height, levels, sigma_color, sigma_guide
    (0, 4, 3, 1.0, 0.2), (4, -1, 3, 1.0, 0.2), (4, 4, 0, 1.0, 0.2), (4, 4, 9, 1.0, 0.2), (4, 4, -3, 1.0, 0.2),
    (4, 4, 3, 0.0, 0.2), (4, 4, 3, -1.0, 0.2), (4, 4, 3, np.nan, 0.2), (4, 4, 3, np.inf, 0.2),
    (4, 4, 3, 1.0, 0.0), (4, 4, 3, 1.0, -0.5), (4, 4, 3, 1.0, np.nan), (4, 4, 3, 1.0, np.inf),
    (4, 4, 3, 1e-300, 0.2),   # float32(sigma) = 0
    (4, 4, 3, 1e20, 0.2),     # sigma^2 overflows float32 at level 0
    (4, 4, 8, 1e-18, 0.2),    # (sigma 2^-7)^2 subnormal
    (4, 4, 8, EDGE * 0.99, 0.2),
    (4, 4, 3, 1.0, 1e-20),    # sigma_guide^2 subnormal
    (4, 4, 3, 1.0, 2e19),     # sigma_guide^2 = inf
]
ACCEPTED = [(4, 4, 1, 1.0, 0.2), (4, 4, 8, 1.0, 0.2), (4, 4, 8, EDGE * 1.01, 0.2), (4, 4, 1, 2e-19, 2e-19),
            (4, 4, 3, 1e19, 1e19), (1, 1, 8, 3.0, 3.0)]


def call_gpu(W, H, levels, sc, sg):
    lin = np.zeros((max(H, 1), max(W, 1), 3))
    sig = (C.c_double * 2)(sc, sg)
    return _abi.lib().rtclj_denoise_gpu(0, lin.ctypes.data, lin.ctypes.data, W, H, levels, sig, 0, lin.ctypes.data, None)


@pytest.mark.parametrize("args", REFUSALS)
def test_refusals(args):
    assert M.check(*args) is not None
    assert call_gpu(*args) == _abi.E_INVALID, _abi.lib().rtclj_last_error()


@pytest.mark.parametrize("args", ACCEPTED)
def test_accepted_arguments_reach_the_device(args):
    assert M.check(*args) is None
    assert call_gpu(*args) in (_abi.OK, _abi.E_NO_DEVICE), _abi.lib().rtclj_last_error()


def test_null_pointers_are_refused():
    lib = _abi.lib()
    img = np.zeros((2, 2, 3))
    sig = (C.c_double * 2)(1.0, 0.2)
    assert lib.rtclj_denoise_gpu(0, None, img.ctypes.data, 2, 2, 3, sig, 0, None, None) == _abi.E_INVALID
    assert lib.rtclj_denoise_gpu(0, img.ctypes.data, None, 2, 2, 3, sig, 0, None, None) == _abi.E_INVALID
    assert lib.rtclj_denoise_gpu(0, img.ctypes.data, img.ctypes.data, 2, 2, 3, None, 0, None, None) == _abi.E_INVALID
    assert lib.rtclj_ctx_denoise(None, img.ctypes.data, img.ctypes.data, 2, 2, 3, sig, 0, None, None, None) == _abi.E_INVALID


def test_render_denoised_refuses_before_rendering():
    world, cam = scenes.main_hittables(), camera.main_camera(16, 9)
    for kw in (dict(guide_samples=0), dict(levels=9), dict(sigma_color=0.0), dict(sigma_guide=np.inf)):
        with pytest.raises(_abi.RtcljError) as e:
            render.render_denoised(world, cam, 4, 4, **kw)
        assert e.value.code == _abi.E_INVALID, kw
    with pytest.raises(ValueError):
        render.denoise(np.zeros((2, 2, 3)), np.zeros((2, 3, 3)))
