"""Adaptive sampling at the sizes it is used at, through the public API: a strict pass cut into sub-passes at
1920x1080, a compaction whose scan takes several rounds at 3840x2160, late passes that trace a handful of pixels out
of two million, a scene of more than 512 spheres, albedo outside [0, 1], moments that overflow, and a context that
serves other renders between and after adaptive accumulations.  Exact means what tests/test_gpu_adaptive.py means:
every pixel carries the bits of the one-shot rtclj_ctx_render at its own sample count, signed zeros included."""
import os
import re

import numpy as np
import pytest

import oracle_lib as O
import oracle_samples as OS
import raytracing_clj_b200 as R
from raytracing_clj_b200 import _abi, render
from test_gpu_adaptive import HUGE, adaptive_run, check_groups, median_tolerance, replay
from test_gpu_progressive import Bufs, assert_bits, context, device_count, oneshot

pytestmark = pytest.mark.gpu
S, CAM = R.scenes, R.camera
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "raytracing-clj_b200", "csrc")


def constant(name, path):
    """A size constant of the library's source, so that a test notices when its case no longer reaches the path it
    was written for."""
    text = open(os.path.join(CSRC, path)).read()
    if name == "kAccumSampleBufBytes":
        m = re.search(r"kAccumSampleBufBytes = \(size_t\)(\d+) << (\d+);", text)
        return int(m.group(1)) << int(m.group(2))
    m = re.search(r"kListThreads = (\d+), kListPer = (\d+), kListTile = kListThreads \* kListPer;", text)
    return int(m.group(1)) * int(m.group(2))


def same_bits(a, b, what):
    assert np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8)), what


def estimates(world, cam, passes, depth, seed, flags, unit, least):
    """Each pixel's largest channel estimate at the first decision (passes up to min_samples), from a run that
    stops every pixel there: a pixel's decision depends on its own sums only."""
    upto = []
    for n in passes:
        upto.append(n)
        if sum(upto) >= least:
            break
    at = adaptive_run(world, cam, tuple(upto), depth, seed, flags, unit, (HUGE, 0.0), least)[-1]
    return at[4].max(axis=2)


def replay_rows(world, cam, rows, passes, depth, seed, flags, unit, tol, least, strict, run):
    """The header's rule in numpy on rows [r0, r1) from the CPU oracle's per-sample colours, against the run."""
    target = sum(passes)
    colors = OS.sample_colors(S.to_soa(world), cam, target, depth, seed=seed, flags=flags, rows=rows)
    want = replay(colors.reshape(-1, target, 3), passes, unit, target, least, tol, strict,
                  bool(flags & O.F_MEAN_DIVIDE))
    r0, r1 = rows
    for (d, lin, _, samples, stderr, _, _), (n, se, mean) in zip(run, want):
        same_bits(samples[r0:r1].reshape(-1), n.astype(np.int32), f"samples, rows {rows}, after {d}")
        same_bits(stderr[r0:r1].reshape(-1, 3), se, f"stderr, rows {rows}, after {d}")
        same_bits(lin[r0:r1].reshape(-1, 3), mean, f"linear, rows {rows}, after {d}")
    return want


def check_run(world, cam, run, depth, seed, flags, unit, strict):
    ref = context(world)
    counts = None
    for d, lin, rgb, samples, _, _, _ in run:
        counts = check_groups(ref, cam, d, lin, rgb, samples, depth, seed, flags, unit, strict)
    ref.close()
    return counts


# ---------------------------------------------------------------- 1. strict passes cut into sub-passes

SUBPASS = [("lane", S.main_hittables(), CAM.main_camera(1920, defocus_angle=0.0), O.FLAGS_MAIN | _abi.F_LANE_KERNEL),
           ("lane2", S.cover_hittables(7), CAM.main_camera(1920, 1080, **S.COVER_CAMERA), O.FLAGS_MAIN | _abi.F_LANE2_KERNEL),
           ("smem", S.main_hittables(), CAM.main_camera(1920, defocus_angle=0.0), O.FLAGS_MAIN | _abi.F_SMEM_TABLE)]


@pytest.mark.parametrize("name,world,cam,flags", SUBPASS, ids=[c[0] for c in SUBPASS])
def test_strict_passes_cut_into_sub_passes_are_exact(name, world, cam, flags):
    """Passes of 40 samples at 1920x1080 in strict order: each is cut into sub-passes of 32 + 8 by the sample
    buffer's size, the first of which folds without deciding.  About half of the pixels stop at 40, so the second
    pass runs with the list half empty."""
    passes, depth, seed = (40, 40), 50, 11
    pixels = cam.width * cam.height
    per = constant("kAccumSampleBufBytes", "rtclj_abi.cu") // (pixels * 32)
    assert per < passes[0] and passes[0] % per != 0, per  # the pass really is cut, with a short last sub-pass
    target, least = sum(passes), 40
    est = estimates(world, cam, passes, depth, seed, flags, target, least)
    tol = (float(np.median(est)), 0.0)
    run = adaptive_run(world, cam, passes, depth, seed, flags, target, tol, least)
    (_, _, _, s1, _, a1, st1), (_, _, _, s2, _, a2, st2) = run
    assert st1["samples"] == pixels * 40 and (s1 == 40).all()
    assert a1 == int((est > tol[0]).sum()) and 0.3 * pixels < a1 < 0.7 * pixels, a1
    assert st2["samples"] == a1 * 40 and a2 == 0 and (s2 == 80).sum() == a1  # counters add up over sub-passes
    counts = check_run(world, cam, run, depth, seed, flags, target, True)
    assert list(counts) == [40, 80]
    if name != "lane":
        return
    # two shards of 64 samples per sub-pass (no cut) make the same images, sample map and noise
    got = [[np.zeros_like(x) for x in r[1:5]] for r in run]
    for i in range(2):
        rows = render.shard_rows(cam.height, i, 2, 1)
        assert constant("kAccumSampleBufBytes", "rtclj_abi.cu") // (len(rows) * cam.width * 32) >= passes[0]
        part = adaptive_run(world, cam, passes, depth, seed, flags, target, tol, least, shard=(i, 2, 1))
        for g, r in zip(got, part):
            for x, y in zip(g, r[1:5]):
                x[rows] = y[rows]
    for g, r in zip(got, run):
        for x, y in zip(g, r[1:5]):
            same_bits(x, y, "two shards against the whole frame")
    for rows in ((0, 2), (cam.height - 1, cam.height)):
        replay_rows(world, cam, rows, passes, depth, seed, flags, 1, tol, least, True, run)


# ---------------------------------------------------------------- 2. compaction rounds


@pytest.mark.parametrize("order", ["chunked", "strict"])
@pytest.mark.parametrize("W,H", [(3840, 2160), (2049, 1024), (2048, 1024)])
def test_compaction_over_several_scan_rounds_is_exact(W, H, order):
    """The -i scene (the primary-ray kernels, seeded in strict order) at sizes of 1024 tiles, 1025 tiles and, at
    3840x2160, 4050 tiles: the scan of the tile counts takes 1, 2 and 4 rounds of 1024."""
    tile = constant("kListTile", "rtclj_adaptive.cuh")
    tiles = -(-W * H // tile)
    assert tiles == {(3840, 2160): 4050, (2049, 1024): 1025, (2048, 1024): 1024}[(W, H)]
    world, cam, flags, depth, seed = S.i_hittables(), CAM.i_camera(W, H), O.FLAGS_I, 50, 13
    strict = order == "strict"
    passes, unit, least = ((4, 4, 4), 12, 4) if strict else ((8, 4, 4), 4, 8)
    tol = median_tolerance(world, cam, passes, depth, seed, flags, unit, least)
    run = adaptive_run(world, cam, passes, depth, seed, flags, unit, tol, least)
    assert 0 < run[0][5] < W * H
    counts = check_run(world, cam, run, depth, seed, flags, unit, strict)
    assert len(counts) >= 2
    if (W, H) != (3840, 2160):
        return
    # 4 shards of 540 rows (1013 tiles: one round) and 3 of 720 (1350 tiles: two rounds) make the whole frame
    for count in (4, 3):
        got = [[np.zeros_like(x) for x in r[1:5]] for r in run]
        for i in range(count):
            rows = render.shard_rows(H, i, count, 1)
            assert -(-len(rows) * W // tile) == {4: 1013, 3: 1350}[count]
            part = adaptive_run(world, cam, passes, depth, seed, flags, unit, tol, least, shard=(i, count, 1))
            for g, r in zip(got, part):
                for x, y in zip(g, r[1:5]):
                    x[rows] = y[rows]
        for g, r in zip(got, run):
            for x, y in zip(g, r[1:5]):
                same_bits(x, y, f"{count} shards against the whole frame")
    # the rows that hold the round boundaries: position 1024 k * tile of the descending order is local pixel
    # W H - 1 - 1024 k tile
    for k, row in ((1, 1613), (2, 1067), (3, 521)):
        assert (W * H - 1 - 1024 * k * tile) // W == row
        replay_rows(world, cam, (row, row + 1), passes, depth, seed, flags, 1 if strict else unit, tol, least, strict,
                    run)


# ---------------------------------------------------------------- 3. sparse late passes

SPARSE = [("lane", S.main_hittables(), CAM.main_camera(1920, defocus_angle=0.0), O.FLAGS_MAIN | _abi.F_LANE_KERNEL, 50),
          ("lane2", S.cover_hittables(7), CAM.main_camera(1920, 1080, **S.COVER_CAMERA), O.FLAGS_MAIN | _abi.F_LANE2_KERNEL, 50),
          ("smem", S.main_hittables(), CAM.main_camera(1920, defocus_angle=0.0), O.FLAGS_MAIN | _abi.F_SMEM_TABLE, 50),
          ("primary", S.main_hittables(), CAM.main_camera(1920, 1080, **S.COVER_CAMERA), O.FLAGS_MAIN, 1)]


@pytest.mark.parametrize("name,world,cam,flags,depth", SPARSE, ids=[c[0] for c in SPARSE])
def test_sparse_late_passes_are_exact(name, world, cam, flags, depth):
    """Tolerances from the estimates at the first decision that leave exactly k pixels of 1920x1080 active, then
    two more passes: the listed kernels' persistent grids run with a few tickets, or with lanes that take a second
    and later ticket from a list of 94 721 pixels."""
    passes, unit, least, seed = (8, 8, 8), 4, 8, 17
    pixels = cam.width * cam.height
    est = estimates(world, cam, passes, depth, seed, flags, unit, least).reshape(-1)
    # the achievable active counts: a pixel stays iff its estimate exceeds the absolute tolerance
    levels = np.unique(est)
    above = est.size - np.searchsorted(np.sort(est), levels, side="right")
    refs = {}
    ref = context(world)
    for n in (8, 16, 24):
        refs[n] = oneshot(ref, cam, n, depth, seed, flags, unit)
    ref.close()
    for k in (1, 32, 33, 94721):
        # k, or the nearest count above 0 if estimates tie at the threshold
        at = int(np.argmin(np.where(above > 0, np.abs(above - k), np.iinfo(np.int64).max)))
        tol, want_active = (float(levels[at]), 0.0), int(above[at])
        assert want_active == int((est > tol[0]).sum()) and want_active > 0
        run = adaptive_run(world, cam, passes, depth, seed, flags, unit, tol, least)
        first, late = run[0], run[1:]
        assert first[5] == want_active, (k, first[5], want_active)
        active = want_active
        for d, lin, rgb, samples, _, now, st in late:
            assert st["samples"] == active * 8, (k, d)
            stopped = samples.reshape(-1) == 8
            assert stopped.sum() == pixels - want_active
            active = now
        # the stopped pixels keep the bits of the first pass; every pixel is exact at its own count
        for d, lin, rgb, samples, _, _, _ in run:
            for n in np.unique(samples):
                m = samples == n
                assert_bits((lin[m], rgb[m]), (refs[n][0][m], refs[n][1][m]), f"k = {k}, after {d}, {n} samples")
        m = run[-1][3] == 8
        assert_bits((run[-1][1][m], run[-1][2][m]), (run[0][1][m], run[0][2][m]), f"k = {k}: stopped pixels")


# ---------------------------------------------------------------- 4.-6. scenes


def exact_case(world, cam, flags, depth, seed, order):
    strict = order == "strict"
    passes, unit, least = ((3, 5, 4), 12, 4) if strict else ((8, 4, 4), 4, 8)
    tol = median_tolerance(world, cam, passes, depth, seed, flags, unit, least)
    run = adaptive_run(world, cam, passes, depth, seed, flags, unit, tol, least)
    assert len(check_run(world, cam, run, depth, seed, flags, unit, strict)) >= 2
    return passes, unit, tol, least, run


@pytest.mark.parametrize("order", ["chunked", "strict"])
def test_scene_of_more_than_512_spheres(order):
    """784 spheres: the table is staged through shared memory (render_listed_kernel<false, ...>)."""
    world = S.field_hittables(7, half=14)
    assert len(world) > 512
    exact_case(world, CAM.main_camera(480, 270, **S.COVER_CAMERA), O.FLAGS_MAIN, 50, 19, order)


def outside_world():
    sp, mat = R.hittable.sphere, R.material
    return [S.body(sp((0, -100.5, -1), 100.0), mat.lambertian((0.8, 0.8, 0.0))),
            S.body(sp((-1.0, 0, -1), 0.5), mat.dielectric(1.5)),
            S.body(sp((-1.0, 0, -1), -0.4), mat.dielectric(1.5)),
            S.body(sp((0.0, 0, -1.2), 0.5), mat.metal((1.3, 0.6, -0.1), 1.7)),
            S.body(sp((1.0, 0, -1), 0.5), mat.dielectric(1.0)),
            S.body(sp((1.0, 0.9, -1), 0.3), mat.dielectric(0.4)),
            S.body(sp((0.3, 0.1, -0.4), 0.0), mat.lambertian((0.5, 0.5, 0.5))),
            S.body(sp((0.0, 0.8, -1.2), -0.25), mat.lambertian((0.2, 0.9, 0.4))),
            S.body(sp((0.0, 0.8, -1.2), 0.1), mat.metal((0.9, 0.9, 0.9), 0.0))]


@pytest.mark.parametrize("order", ["chunked", "strict"])
def test_albedo_outside_the_unit_interval(order):
    """Negative albedo: colours and sums can be negative or -0.0, and |mean| enters the tolerance."""
    world, cam, seed = outside_world(), CAM.main_camera(96), 23
    passes, unit, tol, least, run = exact_case(world, cam, O.FLAGS_MAIN, 50, seed, order)
    strict = order == "strict"
    assert (run[-1][1] < 0).any()
    for rows in ((0, 2), (30, 33)):
        replay_rows(world, cam, rows, passes, 50, seed, O.FLAGS_MAIN, 1 if strict else unit, tol, least, strict, run)


@pytest.mark.parametrize("order", ["chunked", "strict"])
def test_overflowing_moments_keep_a_pixel_active(order):
    """A ground of albedo 1e100: paths with two or more bounces on it carry colours above sqrt(DBL_MAX), so S1^2 and
    S2 overflow.  Under a tolerance nothing finite exceeds, those pixels still trace to the target (the variance
    is not finite, so they count as noisy); the others stop at min_samples."""
    sp, mat = R.hittable.sphere, R.material
    world = [S.body(sp((0, -100.5, -1), 100.0), mat.lambertian((1e100, 1e100, 1e100))),
             S.body(sp((0.0, 0, -1), 0.5), mat.lambertian((0.1, 0.2, 0.5))),
             S.body(sp((-1.0, 0, -1), 0.5), mat.metal((0.8, 0.8, 0.8), 0.0)),
             S.body(sp((1.0, 0, -1), 0.5), mat.dielectric(1.5))]
    cam, seed, depth = CAM.main_camera(64), 29, 50
    strict = order == "strict"
    passes, unit, least = ((4, 4, 4), 12, 4) if strict else ((8, 4, 4), 4, 8)
    target = sum(passes)
    tol = (HUGE, 0.0)
    run = adaptive_run(world, cam, passes, depth, seed, O.FLAGS_MAIN, unit, tol, least)
    want = replay_rows(world, cam, (0, cam.height), passes, depth, seed, O.FLAGS_MAIN, 1 if strict else unit, tol,
                       least, strict, run)
    samples = run[-1][3]
    assert set(np.unique(samples)) == {least, target}, np.unique(samples)
    assert (samples == target).sum() >= 10
    # the pixels that went on are those whose moments overflowed
    assert np.array_equal(samples.reshape(-1) == target, want[-1][0] == target)
    check_run(world, cam, run, depth, seed, O.FLAGS_MAIN, unit, strict)


# ---------------------------------------------------------------- 7. context reuse


def test_context_serves_other_renders_between_and_after_adaptive_accumulations():
    """One-shot renders between adaptive steps (strict, which needs the sample buffer; chunked; another shard), then
    a second adaptive accumulation smaller and one larger than the first, then a plain accumulation: every result
    equals the same call on a fresh context bit for bit."""
    world, flags, depth, seed = S.main_hittables(), O.FLAGS_MAIN | _abi.F_LANE_KERNEL, 50, 31
    cam = CAM.main_camera(480, 270)
    passes, unit, least = (8, 4, 4), 4, 8
    tol = median_tolerance(world, cam, passes, depth, seed, flags, unit, least)
    fresh = adaptive_run(world, cam, passes, depth, seed, flags, unit, tol, least)
    big, small = CAM.main_camera(960, 540), CAM.main_camera(240, 135)
    others = [(big, 24, 24, None), (cam, 12, 4, None), (cam, 8, 4, (1, 2, 1))]  # (camera, spp, unit, shard)
    ref = context(world)
    want_others = [oneshot(ref, c, spp, depth, seed, flags, u, shard=sh) for c, spp, u, sh in others]
    ref.close()

    from test_gpu_adaptive import Noise
    ctx = context(world)
    b, nz = Bufs(cam), Noise(cam)
    ctx.accum_begin(cam, sum(passes), depth, seed=seed, flags=flags, samples_per_unit=unit, stream=b.stream,
                    tolerance=tol, min_samples=least)
    for n, w, (c, spp, u, sh), wo in zip(passes, fresh, others, want_others):
        d = ctx.accum_step(n, **b.ptrs())
        samples, stderr, active = nz.read(ctx, b.stream)
        lin, rgb = b.host()
        for x, y in zip((lin, rgb, samples, stderr), w[1:5]):
            same_bits(x, y, f"adaptive step after {d}")
        assert active == w[5] and ctx.stats(b.stream)["samples"] == w[6]["samples"]
        got = oneshot(ctx, c, spp, depth, seed, flags, u, shard=sh)
        rows = slice(None) if sh is None else render.shard_rows(c.height, *sh)
        assert_bits((got[0][rows], got[1][rows]), (wo[0][rows], wo[1][rows]), f"one-shot {spp} spp between steps")
    # a second adaptive accumulation, smaller then larger than the first, and a plain one after them
    for c in (small, big):
        t = median_tolerance(world, c, passes, depth, seed, flags, unit, least)
        want = adaptive_run(world, c, passes, depth, seed, flags, unit, t, least)
        bc, nc = Bufs(c), Noise(c)
        ctx.accum_begin(c, sum(passes), depth, seed=seed, flags=flags, samples_per_unit=unit, stream=bc.stream,
                        tolerance=t, min_samples=least)
        for n, w in zip(passes, want):
            ctx.accum_step(n, **bc.ptrs())
            samples, stderr, active = nc.read(ctx, bc.stream)
            for x, y in zip(bc.host() + (samples, stderr), w[1:5]):
                same_bits(x, y, f"second accumulation at {c.width}x{c.height}")
            assert active == w[5]
    ctx.accum_begin(cam, sum(passes), depth, seed=seed, flags=flags, samples_per_unit=unit, stream=b.stream)
    d = 0
    for n in passes:
        d = ctx.accum_step(n, **b.ptrs())
    ref = context(world)
    assert_bits(b.host(), oneshot(ref, cam, d, depth, seed, flags, unit), "plain accumulation after adaptive ones")
    ref.close()
    ctx.close()


# ---------------------------------------------------------------- 8. several devices


def test_full_frame_on_two_devices_equals_one():
    if device_count() < 2:
        pytest.skip("one GPU on this box")
    world, cam = S.cover_hittables(7), CAM.main_camera(1920, 1080, **S.COVER_CAMERA)
    passes, unit, least = (8, 8, 8), 8, 16
    tol = (0.02, 0.05)
    outs = []
    for devs in ([0], [0, 1]):
        with render.Progressive(world, cam, sum(passes), 50, seed=37, samples_per_unit=unit, devices=devs,
                                tolerance=tol, min_samples=least) as p:
            outs.append([p.step(n)[:2] + p.noise() for n in passes])
    for a, b in zip(*outs):
        for x, y in zip(a[:4], b[:4]):
            same_bits(x, y, "devices [0, 1] against [0]")
        assert a[4] == b[4]


def test_one_row_image_leaves_a_device_without_rows():
    if device_count() < 2:
        pytest.skip("one GPU on this box")
    world, cam = S.main_hittables(), CAM.i_camera(64, 1)
    outs = []
    for devs in ([0], [0, 1]):
        with render.Progressive(world, cam, 16, 50, seed=41, samples_per_unit=4, devices=devs, tolerance=(0.05, 0.0),
                                min_samples=8) as p:
            steps = []
            for n in (8, 4, 4):
                lin, rgb, st = p.step(n)
                samples, stderr, active = p.noise()
                steps.append((lin, rgb, samples, stderr, active, st["samples"]))
            outs.append(steps)
    for a, b in zip(*outs):
        for x, y in zip(a[:4], b[:4]):
            same_bits(x, y, "one row on two devices")
        assert a[4:] == b[4:]
