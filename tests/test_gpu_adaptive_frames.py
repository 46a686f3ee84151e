"""Accumulations over frames on the GPU (rtclj_ctx_accum_begin_frames, rtclj_progressive_create_frames): after every
step, every frame's linear image, 8-bit image, sample-count map and noise estimate are BIT-identical to a single-camera
accumulation of that frame's camera with the same params, tolerance and min_samples, stepped with the same passes."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib as O
import raytracing_clj_b200 as R
from raytracing_clj_b200 import _abi, render
from test_gpu_adaptive import CASES, median_tolerance
from test_gpu_progressive import assert_bits, context, device_count

pytestmark = pytest.mark.gpu
S, CAM = R.scenes, R.camera
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def moved(cam, k, defocus=None):
    """Frame k of a small fly-by: the camera and its image plane moved along x; defocus: the frame's angle."""
    c = _abi.Camera.from_buffer_copy(render._camera_struct(cam))
    c.center[0] += 0.13 * k
    c.pixel00[0] += 0.13 * k
    if defocus is not None:
        c.defocus_angle = defocus
    return c


class Images:
    """Device images of K frames (linear, 8-bit, sample counts, noise) and their host copies."""

    def __init__(self, cam, k):
        import torch
        H, W = cam.height, cam.width
        self.lin = torch.zeros((k, H, W, 3), dtype=torch.float64, device="cuda:0")
        self.rgb = torch.zeros((k, H, W, 3), dtype=torch.uint8, device="cuda:0")
        self.samples = torch.zeros((k, H, W), dtype=torch.int32, device="cuda:0")
        self.stderr = torch.zeros((k, H, W, 3), dtype=torch.float64, device="cuda:0")
        self.stream = torch.cuda.current_stream().cuda_stream

    def step(self, ctx, n, adaptive):
        d = ctx.accum_step(n, d_out_linear=self.lin.data_ptr(), d_out_rgb8=self.rgb.data_ptr(), stream=self.stream)
        active = ctx.accum_noise(self.samples.data_ptr(), self.stderr.data_ptr(), stream=self.stream) if adaptive else 0
        st = ctx.stats(self.stream)
        out = [t.cpu().numpy().copy() for t in (self.lin, self.rgb, self.samples, self.stderr)]
        return d, out, active, st


def run(world, cams, passes, depth, seed, flags, unit, tol, least, shard=None, frames=True):
    """The passes of one accumulation; frames=True: one accumulation of all cameras, else one per camera (stacked).
    Returns per step (d, [lin, rgb, samples, stderr] of [K, ...], active pixels, samples traced)."""
    steps = [[d, [[], [], [], []], 0, 0] for d in np.cumsum(passes)]
    for group in ([cams] if frames else [[c] for c in cams]):
        ctx = context(world)
        img = Images(cams[0], len(group))
        kw = dict(seed=seed, flags=flags, samples_per_unit=unit, shard=shard, stream=img.stream, tolerance=tol,
                  min_samples=least)
        if frames:
            ctx.accum_begin_frames(group, sum(passes), depth, **kw)
        else:
            ctx.accum_begin(group[0], sum(passes), depth, **kw)
        for s, n in zip(steps, passes):
            d, out, active, st = img.step(ctx, n, tol is not None)
            assert d == s[0]
            for a, b in zip(s[1], out):
                a.append(b)
            s[2] += active
            s[3] += st["samples"]
        ctx.close()
    for s in steps:
        s[1] = [np.concatenate(a) for a in s[1]]
    return steps


def assert_frames_equal(got, want, what, rows=None):
    for (d, g, ga, gs), (_, w, wa, ws) in zip(got, want):
        sel = (slice(None), slice(None) if rows is None else rows)
        assert_bits((g[0][sel], g[1][sel]), (w[0][sel], w[1][sel]), f"{what}: images after {d}")
        assert np.array_equal(g[2][sel], w[2][sel]), f"{what}: sample counts after {d}"
        assert np.array_equal(g[3][sel].view(np.uint64), w[3][sel].view(np.uint64)), f"{what}: noise after {d}"
        if rows is None:
            assert ga == wa and gs == ws, (what, d, ga, wa, gs, ws)


@pytest.mark.parametrize("order", ["chunked", "strict"])
@pytest.mark.parametrize("name,world,cam,flags,depth", CASES, ids=[c[0] for c in CASES])
def test_every_frame_equals_its_own_accumulation(name, world, cam, flags, depth, order):
    """Every kernel family, chunked and strict, irregular passes, a tolerance that stops some pixels; frame 1 has no
    defocus disk where the others have one."""
    strict = order == "strict"
    passes, unit, least = ((3, 5, 2, 7, 11), 28, 4) if strict else ((8, 4, 8, 4, 3), 4, 8)
    cams = [moved(cam, 0), moved(cam, 1, defocus=0.0), moved(cam, 2), moved(cam, 3)]
    tol = median_tolerance(world, cam, passes, depth, 5, flags, unit, least)
    got = run(world, cams, passes, depth, 5, flags, unit, tol, least)
    want = run(world, cams, passes, depth, 5, flags, unit, tol, least, frames=False)
    assert_frames_equal(got, want, name)
    assert len(np.unique(got[-1][1][2])) >= 2 and got[-1][2] < got[0][2]


@pytest.mark.parametrize("order", ["chunked", "strict"])
def test_plain_accumulation_over_frames(order):
    world, cam = S.main_hittables(), CAM.main_camera(40)
    cams = [CAM.main_camera(40, look_from=CAM.turntable_look_from(k, 5)) for k in range(5)]
    unit = 40 if order == "strict" else 6
    got = run(world, cams, (6, 12, 18, 4), 50, 3, O.FLAGS_MAIN, unit, None, 0)
    want = run(world, cams, (6, 12, 18, 4), 50, 3, O.FLAGS_MAIN, unit, None, 0, frames=False)
    assert_frames_equal(got, want, f"plain {order}")


@pytest.mark.parametrize("flags,depth", [(O.FLAGS_MAIN, 50), (O.FLAGS_I, 50)], ids=["lane", "primary"])
def test_more_frames_than_one_launch_takes(flags, depth):
    """130 frames: two launch groups (128 + 2), each with its own list."""
    lane = flags == O.FLAGS_MAIN
    world = S.main_hittables() if lane else S.i_hittables()
    base = CAM.main_camera(12, 7) if lane else CAM.i_camera(12)
    cams = [moved(base, k * 0.05) for k in range(130)]
    unit, least = (4, 8) if lane else (0, 2)  # the primary-ray render: strict order, pass unit 1
    tol = median_tolerance(world, base, (8, 4, 4), depth, 2, flags, unit, least)
    got = run(world, cams, (8, 4, 4), depth, 2, flags, unit, tol, least)
    pick = [0, 1, 64, 127, 128, 129]
    want = run(world, [cams[k] for k in pick], (8, 4, 4), depth, 2, flags, unit, tol, least, frames=False)
    sub = [(d, [a[pick] for a in imgs], 0, 0) for d, imgs, _, _ in got]
    assert_frames_equal(sub, [(d, imgs, 0, 0) for d, imgs, _, _ in want], "130 frames")


@pytest.mark.parametrize("strict", [False, True], ids=["chunked", "strict"])
def test_shards_and_device_lists(strict):
    """Context shards (the rows of one shard) and host-buffer handles over every device list (the whole image)."""
    world = S.cover_hittables(7)
    cam = CAM.main_camera(48, 27, **S.COVER_CAMERA)
    cams = [moved(cam, k) for k in range(3)]
    passes, unit, least = ((8, 4, 4, 5), 21, 4) if strict else ((8, 4, 4, 5), 4, 8)
    tol = median_tolerance(world, cam, passes, 50, 6, O.FLAGS_MAIN, unit, least)
    for shard in ((0, 2, 3), (1, 2, 3), (2, 3, 1)):
        rows = np.array(render.shard_rows(cam.height, *shard))
        got = run(world, cams, passes, 50, 6, O.FLAGS_MAIN, unit, tol, least, shard=shard)
        want = run(world, cams, passes, 50, 6, O.FLAGS_MAIN, unit, tol, least, shard=shard, frames=False)
        assert_frames_equal(got, want, f"shard {shard}", rows=rows)
    want = run(world, cams, passes, 50, 6, O.FLAGS_MAIN, unit, tol, least, frames=False)
    lists = [[0]] + ([list(range(min(device_count(), 3)))] if device_count() > 1 else [])
    for devs in lists:
        with render.ProgressiveFrames(world, cams, sum(passes), 50, seed=6, samples_per_unit=unit, devices=devs,
                                      tolerance=tol, min_samples=least) as p:
            assert p.pass_unit == (1 if strict else unit)
            for n, (d, w, wa, _) in zip(passes, want):
                lin, rgb, _ = p.step(n)
                samples, stderr, active = p.noise()
                assert p.samples_done == d and active == wa
                assert_bits((lin, rgb), (w[0], w[1]), f"devices {devs} after {d}")
                assert np.array_equal(samples, w[2]) and np.array_equal(stderr.view(np.uint64), w[3].view(np.uint64))


def test_min_samples_at_the_target_is_the_sequence_render():
    """min_samples >= spp: no pixel stops early, so the last step is rtclj_render_frames of the target."""
    world = S.main_hittables()
    cams = [CAM.main_camera(40, look_from=CAM.turntable_look_from(k, 4)) for k in range(4)]
    for unit, passes in ((5, (10, 5, 5, 3)), (23, (1, 2, 20))):
        got = run(world, cams, passes, 50, 8, O.FLAGS_MAIN, unit, (0.0, 0.0), sum(passes))
        lin, rgb, _ = render.render_frames(world, cams, sum(passes), 50, seed=8, samples_per_unit=unit)
        assert_bits((got[-1][1][0], got[-1][1][1]), (lin, rgb), f"unit {unit}")
        assert (got[-1][1][2] == sum(passes)).all() and got[-1][2] == 0


def test_strict_frames_split_into_sub_passes():
    """Two 1920x1080 frames in strict order: one sample of both is 133 MB of colours, so a pass of 24 samples runs as
    sub-passes of 16 where a single frame's runs whole -- the same bits."""
    world = S.main_hittables()
    cams = [CAM.main_camera(1920, 1080), CAM.main_camera(1920, 1080, look_from=CAM.turntable_look_from(1, 6))]
    got = run(world, cams, (24, 8), 6, 4, O.FLAGS_MAIN | _abi.F_LANE_KERNEL, 32, (0.02, 0.1), 16)
    want = run(world, cams, (24, 8), 6, 4, O.FLAGS_MAIN | _abi.F_LANE_KERNEL, 32, (0.02, 0.1), 16, frames=False)
    assert_frames_equal(got, want, "1080p strict")
    assert got[0][3] == 2 * 1920 * 1080 * 24


def test_cli_writes_the_adaptive_turntable(tmp_path):
    """main 64 4 --frames 3 --tolerance ... --every 8: three PNGs, frame 0 with the pixels of the single-image run;
    with --apng the same frames in one animation."""
    from PIL import Image
    env = dict(os.environ, PYTHONPATH=ROOT)
    args = ["64", "4", "--tolerance", "0.02,0.1", "--every", "8"]
    for extra in (["--frames", "3"], ["--frames", "3", "--apng"], []):
        subprocess.run([sys.executable, "-m", "raytracing_clj_b200.main", "main", *args, *extra], cwd=tmp_path, env=env,
                       check=True, capture_output=True, text=True)
    frame0 = np.asarray(Image.open(tmp_path / "scene-0000.png").convert("RGB"))
    single = np.asarray(Image.open(tmp_path / "scene.png").convert("RGB"))
    assert np.array_equal(frame0, single)
    anim = Image.open(tmp_path / "scene.apng")
    assert anim.n_frames == 3
    for k in range(3):
        anim.seek(k)
        assert np.array_equal(np.asarray(anim.convert("RGB")),
                              np.asarray(Image.open(tmp_path / f"scene-{k:04d}.png").convert("RGB")))
