"""Progressive rendering on the GPU (rtclj_ctx_accum_*, rtclj_progressive_*): an accumulation over passes
performs the additions of a one-shot render in the same order, so after passes totalling d samples its images
are BIT-identical to rtclj_ctx_render with spp = d in the same summation order -- for every kernel that
accumulates, in strict and in chunked order, sharded or not, on any device list."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib as O
import raytracing_clj_b200 as R
from raytracing_clj_b200 import _abi, render

pytestmark = pytest.mark.gpu
S, CAM = R.scenes, R.camera
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def device_count():
    n = C.c_int()
    _abi.check(_abi.lib().rtclj_device_count(C.byref(n)))
    return n.value


class Bufs:
    """Device images for a camera, and their host copies."""

    def __init__(self, cam):
        import torch
        self.lin = torch.zeros((cam.height, cam.width, 3), dtype=torch.float64, device="cuda:0")
        self.rgb = torch.zeros((cam.height, cam.width, 3), dtype=torch.uint8, device="cuda:0")
        self.stream = torch.cuda.current_stream().cuda_stream

    def ptrs(self):
        return dict(d_out_linear=self.lin.data_ptr(), d_out_rgb8=self.rgb.data_ptr(), stream=self.stream)

    def host(self):
        import torch
        torch.cuda.synchronize()
        return self.lin.cpu().numpy().copy(), self.rgb.cpu().numpy().copy()


def context(world):
    ctx = render.Context(0)
    ctx.set_scene(world)
    return ctx


def oneshot(ctx, cam, spp, depth, seed, flags, unit, shard=None):
    b = Bufs(cam)
    ctx.render(cam, spp, depth, seed=seed, flags=flags, samples_per_unit=unit, shard=shard, **b.ptrs())
    ctx.stats(b.stream)
    return b.host()


def assert_bits(a, b, what):
    lin_a, rgb_a = a
    lin_b, rgb_b = b
    # bit patterns, so that signed zeros count too
    bad = np.argwhere(lin_a.view(np.uint64) != lin_b.view(np.uint64))
    assert bad.size == 0, f"{what}: {len(bad)} linear values differ, first {bad[0]}"
    assert np.array_equal(rgb_a, rgb_b), what


def accumulate_and_check(world, cam, passes, depth, seed, flags, unit, strict, shard=None):
    """Runs the passes on one context; after every pass compares with a one-shot render on another.
    Returns the last images."""
    acc, ref = context(world), context(world)
    target = sum(passes)
    b = Bufs(cam)
    pass_unit = acc.accum_begin(cam, target, depth, seed=seed, flags=flags, samples_per_unit=unit, shard=shard,
                                stream=b.stream)
    assert pass_unit == (1 if strict else unit), pass_unit
    d = 0
    for n in passes:
        d = acc.accum_step(n, **b.ptrs())
        got = b.host()
        st = acc.stats(b.stream)
        assert st["samples_per_unit"] == (d if strict else unit)
        want = oneshot(ref, cam, d, depth, seed, flags, d if strict else unit, shard=shard)
        assert_bits(got, want, f"after {d} samples")
    assert d == target
    acc.close(), ref.close()
    return got


# (name, world, camera, flags, depth); strict order: each kernel over the main / realm / -i variants, with and
# without the defocus disk
STRICT_CASES = [
    ("lane-main-defocus", S.main_hittables(), CAM.main_camera(48), O.FLAGS_MAIN | _abi.F_LANE_KERNEL, 50),
    ("lane-main", S.main_hittables(), CAM.main_camera(48, defocus_angle=0.0), O.FLAGS_MAIN | _abi.F_LANE_KERNEL, 50),
    ("lane-realm", S.realm_hittables(), CAM.realm_camera(40), O.FLAGS_REALM | _abi.F_LANE_KERNEL, 50),
    ("lane-i", S.i_hittables(), CAM.i_camera(40), O.FLAGS_I | _abi.F_LANE_KERNEL, 50),
    ("lane2-main-defocus", S.cover_hittables(7), CAM.main_camera(48, 27, **S.COVER_CAMERA), O.FLAGS_MAIN | _abi.F_LANE2_KERNEL, 50),
    ("lane2-realm", S.cover_hittables(7), CAM.realm_camera(40, 22, look_from=(13.0, 2.0, 3.0), look_at=(0.0, 0.0, 0.0)),
     O.FLAGS_REALM | _abi.F_LANE2_KERNEL, 50),
    ("lane2-i", S.cover_hittables(7), CAM.i_camera(40), O.FLAGS_I | _abi.F_LANE2_KERNEL, 50),
    ("smem-main-defocus", S.main_hittables(), CAM.main_camera(48), O.FLAGS_MAIN | _abi.F_SMEM_TABLE, 50),
    ("smem-realm", S.realm_hittables(), CAM.realm_camera(40), O.FLAGS_REALM | _abi.F_SMEM_TABLE, 50),
    ("smem-i", S.i_hittables(), CAM.i_camera(40), O.FLAGS_I | _abi.F_SMEM_TABLE, 50),
    ("primary-i", S.i_hittables(), CAM.i_camera(40), O.FLAGS_I, 50),
    ("primary-main-depth1-defocus", S.main_hittables(), CAM.main_camera(48), O.FLAGS_MAIN, 1),
    ("primary-main-depth1", S.main_hittables(), CAM.main_camera(48, defocus_angle=0.0), O.FLAGS_MAIN, 1),
    ("primary-realm-depth1", S.realm_hittables(), CAM.realm_camera(40), O.FLAGS_REALM, 1),
]


@pytest.mark.parametrize("name,world,cam,flags,depth", STRICT_CASES, ids=[c[0] for c in STRICT_CASES])
def test_strict_passes_equal_one_shot_strict_renders(name, world, cam, flags, depth):
    """Uneven passes (1, 7, 16, 40): after every pass the images are those of the strict one-shot render of the
    samples so far; the last one is also the CPU oracle's strict render (first rows)."""
    passes = (1, 7, 16, 40)
    unit = 0 if name.startswith("primary") else sum(passes)  # primary-ray renders are strict by default
    lin, rgb = accumulate_and_check(world, cam, passes, depth, 9, flags, unit, strict=True)
    rows = (0, 6)
    lin_o, rgb_o, _ = O.render(S.to_soa(world), cam, sum(passes), depth, seed=9, flags=flags & 0xffff, threads=8,
                               samples_per_unit=sum(passes), rows=rows)
    assert np.array_equal(lin[rows[0]:rows[1]], lin_o[rows[0]:rows[1]]), name
    assert np.array_equal(rgb[rows[0]:rows[1]], rgb_o[rows[0]:rows[1]]), name


CHUNK_CASES = [
    ("lane-main", S.main_hittables(), CAM.main_camera(48), O.FLAGS_MAIN, 50),
    ("lane2-realm", S.cover_hittables(7), CAM.realm_camera(40, 22, look_from=(13.0, 2.0, 3.0), look_at=(0.0, 0.0, 0.0)),
     O.FLAGS_REALM | _abi.F_LANE2_KERNEL, 50),
    ("smem-main", S.main_hittables(), CAM.main_camera(48), O.FLAGS_MAIN | _abi.F_SMEM_TABLE, 50),
    ("primary-i", S.i_hittables(), CAM.i_camera(40), O.FLAGS_I, 50),
    ("large-scene", S.field_hittables(7, half=14), CAM.main_camera(32, 18, **S.COVER_CAMERA), O.FLAGS_MAIN, 50),
]


@pytest.mark.parametrize("name,world,cam,flags,depth", CHUNK_CASES, ids=[c[0] for c in CHUNK_CASES])
def test_chunked_passes_equal_one_shot_chunked_renders(name, world, cam, flags, depth):
    """samples_per_unit = 8, passes 8, 24, 16 and a last one of 5 (target 53): after every pass the images equal
    rtclj_ctx_render(spp = d, samples_per_unit = 8); the last one is the one-shot render of the target."""
    lin, rgb = accumulate_and_check(world, cam, (8, 24, 16, 5), depth, 4, flags, 8, strict=False)
    ctx = context(world)
    assert_bits((lin, rgb), oneshot(ctx, cam, 53, depth, 4, flags, 8), name)
    ctx.close()


def test_default_unit_is_the_one_shot_default():
    """samples_per_unit 0 on a full-depth render: the pass unit is the library's own choice, and the last image
    is the image of the default one-shot render."""
    world, cam = S.main_hittables(), CAM.main_camera(64)
    ctx = context(world)
    b = Bufs(cam)
    unit = ctx.accum_begin(cam, 40, 50, seed=3, stream=b.stream)
    assert unit > 1
    done = 0
    while done < 40:
        done = ctx.accum_step(min(unit, 40 - done), **b.ptrs())
    lin, rgb, st = render.render(world, cam, 40, 50, seed=3)
    assert st["samples_per_unit"] == unit
    assert_bits(b.host(), (lin, rgb), "default unit")
    ctx.close()


def test_strict_pass_larger_than_the_buffer_runs_in_sub_passes():
    """1920x1080, one strict pass of 64 samples: 4.2 GB of per-sample colours, beyond the accumulation's 2 GiB, so
    the pass runs as sub-passes, each folded in sample order -- the same bits as the one-shot strict render."""
    world, cam = S.main_hittables(), CAM.main_camera(1920, 1080)
    ctx = context(world)
    b = Bufs(cam)
    assert ctx.accum_begin(cam, 64, 50, seed=2, samples_per_unit=64, stream=b.stream) == 1
    assert ctx.accum_step(64, **b.ptrs()) == 64
    got = b.host()
    st = ctx.stats(b.stream)
    assert st["samples"] == 1920 * 1080 * 64  # the counters add up over the sub-passes
    want = oneshot(ctx, cam, 64, 50, 2, O.FLAGS_MAIN, 64)
    assert_bits(got, want, "1920x1080 strict")
    ctx.close()


def test_errors_and_a_render_between_steps():
    world, cam = S.main_hittables(), CAM.main_camera(32)
    lib = _abi.lib()
    ctx = context(world)
    b = Bufs(cam)

    def code(fn):
        with pytest.raises(_abi.RtcljError) as e:
            fn()
        return e.value.code, str(e.value)

    # a step before any begin
    assert code(lambda: ctx.accum_step(1, **b.ptrs()))[0] == _abi.E_INVALID
    # the wavefront and split kernels do not accumulate
    for f in (_abi.F_WAVE_KERNEL, _abi.F_SPLIT_KERNEL):
        assert code(lambda: ctx.accum_begin(cam, 16, 50, flags=O.FLAGS_MAIN | f))[0] == _abi.E_INVALID
    assert ctx.accum_begin(cam, 53, 50, seed=5, samples_per_unit=8, stream=b.stream) == 8
    rc, msg = code(lambda: ctx.accum_step(5, **b.ptrs()))  # not a multiple of the pass unit, not the last pass
    assert rc == _abi.E_INVALID and "pass_unit = 8" in msg
    assert code(lambda: ctx.accum_step(0, **b.ptrs()))[0] == _abi.E_INVALID
    assert code(lambda: ctx.accum_step(56, **b.ptrs()))[0] == _abi.E_INVALID  # beyond the target
    assert ctx.accum_step(8, **b.ptrs()) == 8
    # a plain render of something else on the same context leaves the accumulation as it was
    other = Bufs(CAM.main_camera(20))
    ctx.render(CAM.main_camera(20), 12, 7, seed=99, flags=O.FLAGS_REALM, samples_per_unit=12, **other.ptrs())
    assert ctx.accum_step(16, **b.ptrs()) == 24
    ref = context(world)
    assert_bits(b.host(), oneshot(ref, cam, 24, 50, 5, O.FLAGS_MAIN, 8), "render between steps")
    assert ctx.accum_step(24, **b.ptrs()) == 48
    assert ctx.accum_step(5, **b.ptrs()) == 53  # the last pass may be any size
    assert code(lambda: ctx.accum_step(1, **b.ptrs()))[0] == _abi.E_INVALID  # the target is reached
    # rtclj_ctx_set_scene ends the accumulation
    ctx.accum_begin(cam, 16, 50, samples_per_unit=8, stream=b.stream)
    ctx.set_scene(world)
    assert code(lambda: ctx.accum_step(8, **b.ptrs()))[0] == _abi.E_INVALID
    # null handles
    unit, done = C.c_int32(), C.c_int32()
    prm = _abi.Params(16, 50, 1, O.FLAGS_MAIN, 0, 0, 0, 0, 0, 0)
    cm = render._camera_struct(cam)
    assert lib.rtclj_ctx_accum_begin(None, C.byref(cm), C.byref(prm), C.byref(unit), None) == _abi.E_INVALID
    assert lib.rtclj_ctx_accum_step(None, 8, None, None, C.byref(done), None) == _abi.E_INVALID
    assert lib.rtclj_progressive_step(None, 8, None, None, C.byref(done), None) == _abi.E_INVALID
    assert lib.rtclj_last_error() != b""
    # device lists
    for bad in ([-1], [0, 0], [device_count()]):
        assert code(lambda: render.Progressive(world, cam, 8, 50, devices=bad))[0] == _abi.E_INVALID
    with render.Progressive(world, cam, 16, 50, samples_per_unit=8) as p:
        assert code(lambda: p.step(3))[0] == _abi.E_INVALID
        assert code(lambda: p.step(24))[0] == _abi.E_INVALID
        p.step(8)
        assert p.samples_done == 8
    ref.close(), ctx.close()


def test_max_depth_zero_accumulates_black():
    world, cam = S.main_hittables(), CAM.main_camera(32)
    for unit in (0, 4):
        ctx = context(world)
        b = Bufs(cam)
        pass_unit = ctx.accum_begin(cam, 12, 0, samples_per_unit=unit, stream=b.stream)
        d = ctx.accum_step(pass_unit, **b.ptrs())
        lin, rgb = b.host()
        assert not lin.any() and not np.signbit(lin).any()
        assert_bits((lin, rgb), oneshot(ctx, cam, d, 0, 1, O.FLAGS_MAIN, pass_unit), f"black, unit {unit}")
        ctx.close()


def test_sharded_accumulations_cover_the_image():
    """Three contexts accumulating a shard each: the union of their rows is the whole accumulation, and the
    one-shot image."""
    world, cam = S.cover_hittables(7), CAM.main_camera(64, 36, **S.COVER_CAMERA)
    b = Bufs(cam)
    ctxs = [context(world) for _ in range(3)]
    for i, c in enumerate(ctxs):
        c.accum_begin(cam, 20, 50, seed=6, samples_per_unit=4, shard=(i, 3, 2), stream=b.stream)
    for n in (4, 8, 8):
        for c in ctxs:
            c.accum_step(n, **b.ptrs())
    assert_bits(b.host(), oneshot(ctxs[0], cam, 20, 50, 6, O.FLAGS_MAIN, 4), "shards")
    for c in ctxs:
        c.close()


def test_progressive_host_buffers_one_and_several_devices():
    """render.Progressive (rtclj_progressive_*): every step writes the whole image of the samples so far, the
    same for one device and for several."""
    world, cam = S.cover_hittables(7), CAM.main_camera(96, 54, **S.COVER_CAMERA)
    with render.Progressive(world, cam, 30, 50, seed=8, samples_per_unit=6, devices=[0]) as p:
        assert p.pass_unit == 6
        steps = [p.step(n) for n in (6, 12, 12)]
        assert p.samples_done == 30
    for (lin, rgb, st), n, d in zip(steps, (6, 12, 12), (6, 18, 30)):
        lin_r, rgb_r, _ = render.render(world, cam, d, 50, seed=8, samples_per_unit=6)
        assert_bits((lin, rgb), (lin_r, rgb_r), f"one device, {d} samples")
        assert st["n_devices"] == 1 and st["samples"] == 96 * 54 * n
    if device_count() < 2:
        pytest.skip("one GPU on this box")
    with render.Progressive(world, cam, 30, 50, seed=8, samples_per_unit=6, devices=[0, 1]) as p:
        got = [p.step(n) for n in (6, 12, 12)]
    for (lin, rgb, st), (lin1, rgb1, _) in zip(got, steps):
        assert_bits((lin, rgb), (lin1, rgb1), "two devices")
        assert st["n_devices"] == 2


def test_cli_every_writes_the_same_file(tmp_path):
    """`main 32 50 --every 9` rewrites scene.ppm after every pass; its last scene.ppm / scene.png are byte for
    byte those of `main 32 50`."""
    env = dict(os.environ, PYTHONPATH=ROOT)
    for sub, extra in (("once", []), ("every", ["--every", "9"])):
        d = tmp_path / sub
        d.mkdir()
        subprocess.run([sys.executable, "-m", "raytracing_clj_b200.main", "main", "32", "50", *extra], cwd=d, env=env,
                       check=True, capture_output=True)
    for f in ("scene.ppm", "scene.png"):
        assert (tmp_path / "once" / f).read_bytes() == (tmp_path / "every" / f).read_bytes(), f
    assert not list((tmp_path / "every").glob("*.tmp"))
