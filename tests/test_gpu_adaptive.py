"""Adaptive sampling on the GPU (rtclj_ctx_accum_begin_adaptive, rtclj_progressive_*_adaptive): passes trace only
the pixels whose noise estimate is still above the tolerance, and after every pass each pixel's images are
BIT-identical to a one-shot rtclj_ctx_render at the pixel's own sample count; the stopping rule is the header's,
recomputed here in numpy from the CPU oracle's per-sample colours."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib as O
import oracle_samples as OS
import raytracing_clj_b200 as R
from raytracing_clj_b200 import _abi, render
from test_gpu_progressive import Bufs, assert_bits, context, device_count, oneshot

pytestmark = pytest.mark.gpu
S, CAM = R.scenes, R.camera
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HUGE = 1e300  # a tolerance no estimate exceeds: every pixel stops at min_samples


class Noise:
    """Device buffers for the sample-count map and the noise estimate."""

    def __init__(self, cam):
        import torch
        self.samples = torch.zeros((cam.height, cam.width), dtype=torch.int32, device="cuda:0")
        self.stderr = torch.zeros((cam.height, cam.width, 3), dtype=torch.float64, device="cuda:0")

    def read(self, ctx, stream):
        active = ctx.accum_noise(self.samples.data_ptr(), self.stderr.data_ptr(), stream=stream)
        return self.samples.cpu().numpy().copy(), self.stderr.cpu().numpy().copy(), active


def adaptive_run(world, cam, passes, depth, seed, flags, unit, tol, least, shard=None):
    """Runs the passes of one adaptive accumulation; returns [(d, lin, rgb, samples, stderr, active, stats)]."""
    ctx = context(world)
    b, nz = Bufs(cam), Noise(cam)
    ctx.accum_begin(cam, sum(passes), depth, seed=seed, flags=flags, samples_per_unit=unit, shard=shard,
                    stream=b.stream, tolerance=tol, min_samples=least)
    out = []
    for n in passes:
        d = ctx.accum_step(n, **b.ptrs())
        samples, stderr, active = nz.read(ctx, b.stream)
        lin, rgb = b.host()
        out.append((d, lin, rgb, samples, stderr, active, ctx.stats(b.stream)))
    ctx.close()
    return out


def median_tolerance(world, cam, passes, depth, seed, flags, unit, least):
    """An absolute tolerance that stops about half of the pixels at min_samples: the median of the estimates there
    (a run that stops every pixel at min_samples sees the same sums)."""
    run = adaptive_run(world, cam, passes, depth, seed, flags, unit, (HUGE, 0.0), least)
    at = next(r for r in run if r[0] >= least)
    return (float(np.median(at[4].max(axis=2))), 0.0)


def check_groups(ref, cam, d, lin, rgb, samples, depth, seed, flags, unit, strict, shard=None):
    """Every pixel against the one-shot render at its own count (only the rows of `shard`, if given)."""
    rows = np.arange(cam.height) if shard is None else np.array(render.shard_rows(cam.height, *shard))
    counts = np.unique(samples[rows])
    for n in counts:
        assert 0 < n <= d, (n, d)
        want_lin, want_rgb = oneshot(ref, cam, int(n), depth, seed, flags, int(n) if strict else unit)
        m = np.zeros(samples.shape, dtype=bool)
        m[rows] = samples[rows] == n
        assert_bits((lin[m], rgb[m]), (want_lin[m], want_rgb[m]), f"after {d}: the {m.sum()} pixels of {n} samples")
    return counts


# (name, world, camera, flags, depth, strict); strict order runs through sample_buf (lane, lane2, smem) or through
# the seeded primary-ray kernel (primary-*)
CASES = [
    ("lane-main-defocus", S.main_hittables(), CAM.main_camera(40), O.FLAGS_MAIN | _abi.F_LANE_KERNEL, 50),
    ("lane-main", S.main_hittables(), CAM.main_camera(40, defocus_angle=0.0), O.FLAGS_MAIN | _abi.F_LANE_KERNEL, 50),
    ("lane-realm", S.realm_hittables(), CAM.realm_camera(32), O.FLAGS_REALM | _abi.F_LANE_KERNEL, 50),
    ("lane-i", S.i_hittables(), CAM.i_camera(32), O.FLAGS_I | _abi.F_LANE_KERNEL, 50),
    ("lane2-main-defocus", S.cover_hittables(7), CAM.main_camera(40, 22, **S.COVER_CAMERA), O.FLAGS_MAIN | _abi.F_LANE2_KERNEL, 50),
    ("lane2-realm", S.cover_hittables(7), CAM.realm_camera(32, 18, look_from=(13.0, 2.0, 3.0), look_at=(0.0, 0.0, 0.0)),
     O.FLAGS_REALM | _abi.F_LANE2_KERNEL, 50),
    ("lane2-i", S.cover_hittables(7), CAM.i_camera(32), O.FLAGS_I | _abi.F_LANE2_KERNEL, 50),
    ("smem-main-defocus", S.main_hittables(), CAM.main_camera(40), O.FLAGS_MAIN | _abi.F_SMEM_TABLE, 50),
    ("smem-realm", S.realm_hittables(), CAM.realm_camera(32), O.FLAGS_REALM | _abi.F_SMEM_TABLE, 50),
    ("smem-i", S.i_hittables(), CAM.i_camera(32), O.FLAGS_I | _abi.F_SMEM_TABLE, 50),
    ("primary-i", S.i_hittables(), CAM.i_camera(32), O.FLAGS_I, 50),
    # (at max-depth 1 a hit is black: cameras that also see the sky, so that some pixels are noisy)
    ("primary-main-depth1-defocus", S.main_hittables(), CAM.main_camera(40, 22, **S.COVER_CAMERA), O.FLAGS_MAIN, 1),
    ("primary-realm-depth1", S.realm_hittables(), CAM.realm_camera(32, 18, look_from=(13.0, 2.0, 3.0), look_at=(0.0, 0.0, 0.0)),
     O.FLAGS_REALM, 1),
]


@pytest.mark.parametrize("order", ["chunked", "strict"])
@pytest.mark.parametrize("name,world,cam,flags,depth", CASES, ids=[c[0] for c in CASES])
def test_every_pixel_equals_the_one_shot_render_of_its_count(name, world, cam, flags, depth, order):
    """Uneven passes; a tolerance that stops some pixels but not all.  After every pass, the pixels of each sample
    count carry the bits of the one-shot render at that count."""
    strict = order == "strict"
    if strict:
        passes, unit, least = (3, 5, 2, 7, 11), sum((3, 5, 2, 7, 11)), 4
    else:
        passes, unit, least = (8, 4, 8, 4, 3), 4, 8
    tol = median_tolerance(world, cam, passes, depth, 5, flags, unit, least)
    run = adaptive_run(world, cam, passes, depth, 5, flags, unit, tol, least)
    ref = context(world)
    for d, lin, rgb, samples, _, _, _ in run:
        counts = check_groups(ref, cam, d, lin, rgb, samples, depth, 5, flags, unit, strict)
    assert len(counts) >= 2, counts
    ref.close()


def test_sharded_adaptive_accumulations_are_exact_and_cover_the_image():
    world, cam = S.cover_hittables(7), CAM.main_camera(48, 27, **S.COVER_CAMERA)
    passes, unit, least = (8, 4, 4, 5), 4, 8
    tol = median_tolerance(world, cam, passes, 50, 6, O.FLAGS_MAIN, unit, least)
    whole = adaptive_run(world, cam, passes, 50, 6, O.FLAGS_MAIN, unit, tol, least)
    ref = context(world)
    for i in range(3):
        part = adaptive_run(world, cam, passes, 50, 6, O.FLAGS_MAIN, unit, tol, least, shard=(i, 3, 2))
        rows = render.shard_rows(cam.height, i, 3, 2)
        for (d, lin, rgb, samples, stderr, _, _), w in zip(part, whole):
            check_groups(ref, cam, d, lin, rgb, samples, 50, 6, O.FLAGS_MAIN, unit, False, shard=(i, 3, 2))
            for a, b in zip((lin, rgb, samples, stderr), w[1:5]):
                assert np.array_equal(a[rows].view(np.uint8), b[rows].view(np.uint8))
    ref.close()


def replay(colors, passes, unit, target, least, tol, strict, mean_divide):
    """The header's rule in numpy from per-sample colours [P, spp, 3]: (samples [P], stderr [P,3], mean [P,3]) after
    every pass.  Sums are formed sequentially (np.add.accumulate would do as well; np.sum would not: pairwise)."""
    npix = colors.shape[0]
    s1, s2 = np.zeros((npix, 3)), np.zeros((npix, 3))
    n, live = np.zeros(npix, dtype=np.int64), np.ones(npix, dtype=bool)
    d, out = 0, []
    for p in passes:
        idx = np.nonzero(live)[0]
        for u0 in range(d, d + p, unit):   # the units of the pass, in order
            U = np.zeros((len(idx), 3))
            for k in range(u0, min(u0 + unit, d + p)):
                U = U + colors[idx, k]
            s1[idx] = s1[idx] + U
            s2[idx] = s2[idx] + U * U
        d += p
        n[idx] = d
        m = np.ceil(n / unit).astype(np.float64)[:, None]
        with np.errstate(divide="ignore", invalid="ignore"):
            q = s1 * s1
            q = q / m
            v = s2 - q
            v = v / (m * (m - 1.0))
            v = v / (float(unit) * float(unit))
            v = np.fmax(v, 0.0)
            se = np.sqrt(v)
        num = (0.0 + s1) if strict else s1
        mean = num / n[:, None] if mean_divide else num * (1.0 / n[:, None])
        with np.errstate(over="ignore", invalid="ignore"):
            t = tol[0] + tol[1] * np.abs(mean)
            overflow = ~(np.isfinite(s1 * s1) & np.isfinite(s2))  # moments that overflowed count as noisy
        keep = (n < target) & ((n < least) | (se > t).any(axis=1) | overflow.any(axis=1))
        live[idx] = keep[idx]
        out.append((n.copy(), se.copy(), mean.copy()))
    return out


@pytest.mark.parametrize("order", ["chunked", "strict"])
def test_rule_against_the_oracle(order):
    """The device's sample map equals numpy's exactly, its noise estimate and linear image bit for bit."""
    world, cam = S.main_hittables(), CAM.main_camera(24)
    strict = order == "strict"
    passes = (4, 2, 3, 5) if strict else (8, 4, 4, 3)
    unit = 1 if strict else 4
    least, target = (4 if strict else 8), sum(passes)
    colors = OS.sample_colors(S.to_soa(world), cam, target, 50, seed=2, flags=O.FLAGS_MAIN)
    colors = colors.reshape(-1, target, 3)
    # a tolerance between the estimates of the pixels at min_samples (numpy's own), so that both outcomes occur
    probe = replay(colors, passes, unit, target, least, (HUGE, 0.0), strict, True)
    at = next(r for r, d in zip(probe, np.cumsum(passes)) if d >= least)
    tol = (float(np.median(at[1].max(axis=1))), 0.02)
    want = replay(colors, passes, unit, target, least, tol, strict, True)
    got = adaptive_run(world, cam, passes, 50, 2, O.FLAGS_MAIN, target if strict else unit, tol, least)
    H, W = cam.height, cam.width
    for (d, lin, _, samples, stderr, active, _), (n, se, mean) in zip(got, want):
        assert np.array_equal(samples.reshape(-1), n), d
        assert np.array_equal(stderr.reshape(-1, 3).view(np.uint64), se.view(np.uint64)), d
        assert np.array_equal(lin.reshape(-1, 3).view(np.uint64), mean.view(np.uint64)), d
    assert len(np.unique(got[-1][3])) >= 2


def test_decisions_are_the_same_on_every_kernel_and_shard_layout():
    world, cam = S.cover_hittables(7), CAM.main_camera(48, 27, **S.COVER_CAMERA)
    passes, unit, least = (8, 4, 8, 4), 4, 8
    tol = median_tolerance(world, cam, passes, 50, 4, O.FLAGS_MAIN, unit, least)
    base = adaptive_run(world, cam, passes, 50, 4, O.FLAGS_MAIN | _abi.F_LANE_KERNEL, unit, tol, least)
    for extra in (_abi.F_LANE2_KERNEL, _abi.F_SMEM_TABLE):
        other = adaptive_run(world, cam, passes, 50, 4, O.FLAGS_MAIN | extra, unit, tol, least)
        for a, b in zip(base, other):
            for x, y in zip(a[1:5], b[1:5]):
                assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), extra
            assert a[5] == b[5], extra
    flat = [r[1:5] for r in base]
    for rows in (1, 3):
        got = [None] * len(passes)
        for i in range(2):
            part = adaptive_run(world, cam, passes, 50, 4, O.FLAGS_MAIN, unit, tol, least, shard=(i, 2, rows))
            mine = render.shard_rows(cam.height, i, 2, rows)
            for k, r in enumerate(part):
                if got[k] is None:
                    got[k] = [np.zeros_like(x) for x in r[1:5]]
                for g, x in zip(got[k], r[1:5]):
                    g[mine] = x[mine]
        for g, f in zip(got, flat):
            for x, y in zip(g, f):
                assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), rows
    # host buffers on devices [0] and [0, 1]
    outs = []
    for devs in ([0], [0, 1]):
        if len(devs) > device_count():
            pytest.skip("one GPU on this box")
        with render.Progressive(world, cam, sum(passes), 50, seed=4, samples_per_unit=unit, devices=devs,
                                tolerance=tol, min_samples=least) as p:
            outs.append([p.step(n)[:2] + p.noise()[:2] for n in passes])
    for a, b in zip(*outs):
        for x, y in zip(a, b):
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8))


def test_limits():
    world, cam = S.main_hittables(), CAM.main_camera(40)
    passes, unit = (8, 4, 8, 5), 4
    target = sum(passes)
    # min_samples >= spp: nothing stops early, the plain accumulation bit for bit after every pass
    run = adaptive_run(world, cam, passes, 50, 3, O.FLAGS_MAIN, unit, (0.0, 0.0), target)
    plain = context(world)
    b = Bufs(cam)
    plain.accum_begin(cam, target, 50, seed=3, samples_per_unit=unit, stream=b.stream)
    for (d, lin, rgb, samples, _, active, st), n in zip(run, passes):
        assert plain.accum_step(n, **b.ptrs()) == d
        assert_bits((lin, rgb), b.host(), f"min_samples = spp, after {d}")
        assert (samples == d).all() and st["samples"] == n * cam.width * cam.height
    assert run[-1][5] == 0
    plain.close()
    # a huge tolerance: every pixel stops at the first pass boundary at or above min_samples (12), later passes
    # trace nothing and leave the images as they were
    run = adaptive_run(world, cam, passes, 50, 3, O.FLAGS_MAIN, unit, (HUGE, HUGE), 12)
    assert run[0][5] == cam.width * cam.height and run[1][5] == 0
    for d, lin, rgb, samples, _, active, st in run[2:]:
        assert (samples == 12).all() and st["samples"] == 0 and active == 0
        assert_bits((lin, rgb), run[1][1:3], f"stopped, after {d}")
    # the counters count what was traced: active pixels x pass samples
    tol = median_tolerance(world, cam, passes, 50, 3, O.FLAGS_MAIN, unit, 8)
    run = adaptive_run(world, cam, passes, 50, 3, O.FLAGS_MAIN, unit, tol, 8)
    active = cam.width * cam.height
    for (d, _, _, samples, _, now_active, st), n in zip(run, passes):
        assert st["samples"] == active * n, d
        assert (samples == d).sum() >= now_active
        active = now_active


def test_host_api_end_to_end():
    """render.Progressive with a tolerance, into host buffers on every device present: the images, map and noise
    of the device-resident context; noise() counts the pixels the next pass traces."""
    world, cam = S.cover_hittables(7), CAM.main_camera(64, 36, **S.COVER_CAMERA)
    passes, unit, least = (6, 6, 12, 6), 6, 12
    tol = median_tolerance(world, cam, passes, 50, 8, O.FLAGS_MAIN, unit, least)
    want = adaptive_run(world, cam, passes, 50, 8, O.FLAGS_MAIN, unit, tol, least)
    devs = list(range(device_count()))
    with render.Progressive(world, cam, sum(passes), 50, seed=8, samples_per_unit=unit, devices=devs, tolerance=tol,
                            min_samples=least) as p:
        assert p.pass_unit == unit
        prev_active = None
        for n, w in zip(passes, want):
            lin, rgb, st = p.step(n)
            samples, stderr, active = p.noise()
            for x, y in zip((lin, rgb, samples, stderr), w[1:5]):
                assert np.array_equal(x.view(np.uint8), y.view(np.uint8))
            assert active == w[5] and st["n_devices"] == len(devs)
            if prev_active is not None:
                assert (samples == p.samples_done).sum() == prev_active  # exactly the active pixels were traced
            prev_active = active


def test_cli_tolerance_writes_the_image_and_the_sample_map(tmp_path):
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-m", "raytracing_clj_b200.main", "main", "24", "10", "--every", "4",
                        "--tolerance", "0.01,0.05"], cwd=tmp_path, env=env, check=True, capture_output=True, text=True)
    for f in ("scene.ppm", "scene.png", "scene-samples.png"):
        assert (tmp_path / f).stat().st_size > 0, f
    assert "samples traced:" in r.stdout
