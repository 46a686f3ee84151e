"""The six variant switches in every combination, seeds across the whole 64-bit Philox key, and an image past 2^31
pixels -- on every kernel family, against the CPU oracle, bit for bit.

The reference's three programs differ by six bits of rtclj_params.flags, and the kernels read them at run time in four
shading implementations and three finalize paths.  The rest of the suite renders three combinations only, in which
SCHLICK, REVERSE_PRODUCT and MEAN_DIVIDE are always set together, and NORMAL_SHADING always comes with QUANT_LINEAR;
it uses seeds below 2^32 (the key's high word k1 = 0), and images of at most 33 M pixels.  Here:

- all 64 combinations on the one-shot kernels, in chunked and strict order (one unit per pixel, and through the
  per-sample buffer), on scenes in which every switch changes the image (tests/variant_matrix.py and the liveness
  check of tests/test_variant_matrix.py);
- a pairwise covering array of the switches (plus the three programs) on the shared-table kernel, camera sequences,
  accumulations and adaptive accumulations;
- ten seeds that set either word of the key, or make a round key wrap, on every kernel family, the twins and the
  host-buffer entry points;
- a 65536 x 33280 image (2^31 + 2^25 pixels): Philox pixel counters at or above 2^31, output offsets above 2^32 bytes,
  and a sample count above 2^32."""
import numpy as np
import pytest

import oracle_lib as O
import oracle_samples as OS
import raytracing_clj_b200 as R
import variant_matrix as V
from raytracing_clj_b200 import _abi, render
from test_gpu_adaptive import adaptive_run, check_groups, median_tolerance
from test_gpu_frames import LIN_SENTINEL, RGB_SENTINEL, check, cover_cams
from test_gpu_progressive import accumulate_and_check, assert_bits, context

pytestmark = pytest.mark.gpu
S, CAM = R.scenes, R.camera


def differs(got, want, depth):
    """None if the GPU render (linear, rgb8, stats) equals the oracle's (linear, rgb8, segments, samples), else why.
    At depth 0 the library traces nothing and counts no samples; the oracle counts its black samples."""
    lin, rgb, st = got
    want = want[:3] + (want[3] if depth > 0 else 0,)
    bad = np.argwhere(lin.view(np.uint64) != want[0].view(np.uint64))
    if bad.size:
        return f"{len(bad)} linear values differ, first {bad[0].tolist()}: oracle {want[0][tuple(bad[0])]!r} gpu {lin[tuple(bad[0])]!r}"
    if not np.array_equal(rgb, want[1]):
        return f"{int((rgb != want[1]).sum())} 8-bit values differ"
    if (st["segments"], st["samples"]) != want[2:]:
        return f"segments / samples {st['segments']} / {st['samples']}, oracle {want[2]} / {want[3]}"
    return None


def report(failed, what):
    assert not failed, f"{what}: {len(failed)} renders differ from the oracle:\n" + "\n".join(failed[:12])


# ---------------------------------------------------------------- all 64 combinations on the one-shot kernels

PATH_SCENES = ["mixed", "mixed-depth2", "mixed-depth1", "mixed-depth0", "guard"]
# family -> (scenes, flags that select it); "lane-packed" is the constant-table kernel of < 64 spheres, "lane-unpacked"
# that of 64 .. 512; "primary" the primary-ray kernel (<= 6 spheres, depth 1 or NORMAL_SHADING: on "small", at depth
# 50, the combinations without NORMAL_SHADING run the library's path kernel)
FAMILIES = {
    "auto": (PATH_SCENES + ["cover"], 0),
    "lane-packed": (PATH_SCENES, _abi.F_LANE_KERNEL),
    "lane-unpacked": (["cover"], _abi.F_LANE_KERNEL),
    "lane2": (PATH_SCENES + ["cover"], _abi.F_LANE2_KERNEL),
    "wave": (PATH_SCENES + ["cover"], _abi.F_WAVE_KERNEL),
    "split": (PATH_SCENES + ["cover"], _abi.F_SPLIT_KERNEL),
    "smem-table": (PATH_SCENES + ["cover"], _abi.F_SMEM_TABLE),
    "no-cull": (["mixed", "guard", "cover"], _abi.F_NO_CULL),
    "primary": (["small-depth1", "small-depth1-pinhole", "small"], 0),
}
# order -> (spp, samples_per_unit) for a scene of spp s: chunks of 3 samples; one unit per pixel (spp < 64); one unit
# per pixel through the per-sample buffer (spp >= 64, first scene of the family only)
ORDERS = {"chunked": lambda s: (s, 3), "strict": lambda s: (s, s), "strict-sample-buf": lambda s: (65, 65)}


@pytest.mark.parametrize("order", list(ORDERS))
@pytest.mark.parametrize("family", list(FAMILIES))
def test_every_combination_on_every_kernel(family, order):
    names, extra = FAMILIES[family]
    if order == "strict-sample-buf":
        names = names[:1]
    failed = []
    for name in names:
        scene, cam, spp0, depth, seed = V.SCENES[name]
        spp, unit = ORDERS[order](spp0)
        for f in V.ALL_COMBOS:
            got = render.render(scene, cam, spp, depth, seed=seed, flags=f | extra, samples_per_unit=unit)
            why = differs(got, V.oracle(name, f, spp=spp, unit=unit), depth)
            if why:
                failed.append(f"{name} flags {f:#08b}: {why}")
    report(failed, f"{family} {order}")


# ---------------------------------------------------------------- the covering array on the larger regimes


def smem_blocks():
    import torch
    import cull_walk_model as M
    return M.smem_table_blocks(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)


@pytest.mark.parametrize("which", ["field-780", "boundary"])
def test_pairwise_on_the_shared_table_kernel(which):
    """More than 512 spheres: the shared-memory-table kernel; "boundary": 32 S + 16 spheres, the last blocks of the
    table read from global memory (the size of test_gpu_large_scenes.boundary_scene)."""
    if which == "field-780":
        bodies = S.field_hittables(7, half=14)
        cam, spp, units = CAM.main_camera(32, 18, **S.COVER_CAMERA), 6, (0, 4)
    else:
        field = S._random_field(1, -80, 80)
        n = 32 * smem_blocks() + 16
        assert n + 3 < len(field), n
        bodies = field[:n - 3] + field[-3:]   # the ground, ~n grid spheres and the three big ones
        cam = CAM.main_camera(32, 18, vfov=40.0, look_from=(-20.0, 10.0, 30.0), look_at=(-55.0, 0.0, 0.0),
                              defocus_angle=0.3, focus_dist=40.0)
        spp, units = 3, (0,)
    scene = V.garble(S.to_soa(bodies))
    assert len(scene[1]) > 512
    failed = []
    for f in V.PAIRWISE:
        for unit in units:
            lin, rgb, st = O.render(scene, cam, spp, 50, seed=31 + f, flags=f, threads=8, samples_per_unit=unit or spp)
            got = render.render(scene, cam, spp, 50, seed=31 + f, flags=f, samples_per_unit=unit or spp)
            why = differs(got, (lin, rgb, st.segments, st.samples), 50)
            if why:
                failed.append(f"flags {f:#08b} unit {unit}: {why}")
    report(failed, which)


def turntable(n=3, w=40, h=22, defocus=10.0):
    return [CAM.main_camera(w, h, vfov=40.0, look_from=CAM.turntable_look_from(k, n, (-2.0, 1.0, 1.0), (0.0, 0.0, -1.0)),
                            look_at=(0.0, 0.0, -1.0), defocus_angle=defocus, focus_dist=3.0) for k in range(n)]


# family -> (scene, cameras, depth, flags that select it)
TWIN_FAMILIES = {
    "lane-packed": (V.soa(V.MIXED), turntable(), 50, _abi.F_LANE_KERNEL),
    "lane-unpacked": (V.cover_slice(), cover_cams(3, 40, 22), 50, _abi.F_LANE_KERNEL),
    "lane2": (V.soa(V.MIXED), turntable(), 50, _abi.F_LANE2_KERNEL),
    "smem-table": (V.soa(V.MIXED), turntable(), 50, _abi.F_SMEM_TABLE),
    "primary": (V.soa(V.SMALL), turntable(), 1, 0),
}


@pytest.mark.parametrize("family", list(TWIN_FAMILIES))
def test_pairwise_camera_sequences(family):
    """Each frame of a sequence equals its single render: chunked, strict, and strict through the sample buffer."""
    world, cams, depth, extra = TWIN_FAMILIES[family]
    for f in V.PAIRWISE:
        for spp, unit in ((7, 3), (7, 7), (65, 65)):
            check(world, cams, spp, depth, f | extra, f"{family} flags {f:#08b} spp {spp} unit {unit}", unit=unit, seed=f)


@pytest.mark.parametrize("order", ["chunked", "strict"])
@pytest.mark.parametrize("family", list(TWIN_FAMILIES))
def test_pairwise_accumulations(family, order):
    """After every pass, the one-shot render of the samples so far; strict order on the primary kernel runs its
    seeded variant."""
    world, cams, depth, extra = TWIN_FAMILIES[family]
    strict = order == "strict"
    passes = (1, 6, 5) if strict else (3, 6, 2)
    unit = (0 if family == "primary" else sum(passes)) if strict else 3
    for f in V.PAIRWISE:
        accumulate_and_check(world, cams[0], passes, depth, 40 + f, f | extra, unit, strict)


@pytest.mark.parametrize("order", ["chunked", "strict"])
@pytest.mark.parametrize("family", list(TWIN_FAMILIES))
def test_pairwise_adaptive_accumulations(family, order):
    """Every pixel equal to the one-shot render at its own count (finalize_adaptive_kernel reads MEAN_DIVIDE and
    QUANT_LINEAR)."""
    world, cams, depth, extra = TWIN_FAMILIES[family]
    strict = order == "strict"
    passes, unit, least = ((3, 5, 2, 7), 17, 4) if strict else ((6, 3, 6, 3), 3, 6)
    mixed = 0
    for f in V.PAIRWISE:
        flags = f | extra
        tol = median_tolerance(world, cams[0], passes, depth, 50 + f, flags, unit, least)
        ref = context(world)
        for d, lin, rgb, samples, _, _, _ in adaptive_run(world, cams[0], passes, depth, 50 + f, flags, unit, tol, least):
            counts = check_groups(ref, cams[0], d, lin, rgb, samples, depth, 50 + f, flags, unit, strict)
        ref.close()
        mixed += len(counts) >= 2
    assert mixed >= len(V.PAIRWISE) // 2, "too few combinations stop some pixels early"


# ---------------------------------------------------------------- seeds across the 64-bit key

SEED_KERNELS = {"auto": 0, "lane": _abi.F_LANE_KERNEL, "lane2": _abi.F_LANE2_KERNEL, "wave": _abi.F_WAVE_KERNEL,
                "split": _abi.F_SPLIT_KERNEL, "smem-table": _abi.F_SMEM_TABLE, "no-cull": _abi.F_NO_CULL}


@pytest.mark.parametrize("seed", V.SEEDS, ids=[f"{s:#x}" for s in V.SEEDS])
def test_seed_on_every_kernel_family(seed):
    """A defocus camera and glass (FLAGS_MAIN: Schlick draws), so that the rarely taken Philox call sites run: the disk
    rejection loop, unit-vector retries and the first sample of each chunk."""
    failed = []
    runs = [("mixed", extra, k) for k, extra in SEED_KERNELS.items()] + \
           [("cover", _abi.F_LANE_KERNEL, "lane-unpacked"), ("small-depth1", 0, "primary"), ("small", 0, "primary-i")]
    for name, extra, kernel in runs:
        scene, cam, spp, depth, _ = V.SCENES[name]
        flags = O.FLAGS_I if kernel == "primary-i" else O.FLAGS_MAIN
        for unit in (3, spp):
            got = render.render(scene, cam, spp, depth, seed=seed, flags=flags | extra, samples_per_unit=unit)
            why = differs(got, V.oracle(name, flags, unit=unit, seed=seed), depth)
            if why:
                failed.append(f"{kernel} unit {unit}: {why}")
    report(failed, f"seed {seed:#x}")
    # the high word is part of the key: s and s + 2^32 give different images, on the GPU and in the oracle
    scene, cam, spp, depth, _ = V.SCENES["mixed"]
    other = (seed + (1 << 32)) % (1 << 64)
    a = render.render(scene, cam, spp, depth, seed=seed, flags=O.FLAGS_MAIN, samples_per_unit=spp)[0]
    b = render.render(scene, cam, spp, depth, seed=other, flags=O.FLAGS_MAIN, samples_per_unit=spp)[0]
    assert not np.array_equal(a, b)
    assert not np.array_equal(V.oracle("mixed", O.FLAGS_MAIN, seed=seed)[0], V.oracle("mixed", O.FLAGS_MAIN, seed=other)[0])


@pytest.mark.parametrize("seed", V.SEEDS, ids=[f"{s:#x}" for s in V.SEEDS])
def test_seed_on_the_twins(seed):
    """Camera sequences, accumulations (strict on the seeded primary kernel) and adaptive accumulations."""
    for family in ("lane-packed", "lane2", "primary"):
        world, cams, depth, extra = TWIN_FAMILIES[family]
        check(world, cams, 7, depth, O.FLAGS_MAIN | extra, f"frames {family}", unit=3, seed=seed)
    for family, strict in (("lane-packed", True), ("lane2", False), ("primary", True)):
        world, cams, depth, extra = TWIN_FAMILIES[family]
        passes = (1, 6, 5) if strict else (3, 6, 2)
        unit = (0 if family == "primary" else sum(passes)) if strict else 3
        accumulate_and_check(world, cams[0], passes, depth, seed, O.FLAGS_MAIN | extra, unit, strict)
    for family, strict in (("lane2", False), ("primary", True)):
        world, cams, depth, extra = TWIN_FAMILIES[family]
        passes, unit, least = ((3, 5, 2, 7), 17, 4) if strict else ((6, 3, 6, 3), 3, 6)
        flags = O.FLAGS_MAIN | extra
        tol = median_tolerance(world, cams[0], passes, depth, seed, flags, unit, least)
        ref = context(world)
        for d, lin, rgb, samples, _, _, _ in adaptive_run(world, cams[0], passes, depth, seed, flags, unit, tol, least):
            check_groups(ref, cams[0], d, lin, rgb, samples, depth, seed, flags, unit, strict)
        ref.close()


@pytest.mark.parametrize("seed", V.SEEDS, ids=[f"{s:#x}" for s in V.SEEDS])
def test_seed_on_the_host_buffer_entry_points(seed):
    """render.render, render_ppm, render_png, the host Progressive and host render_frames, against the oracle."""
    name = "mixed"
    scene, cam, spp, depth, _ = V.SCENES[name]
    lin_o, rgb_o, segments, _ = V.oracle(name, O.FLAGS_MAIN, unit=3, seed=seed)
    lin, rgb, st = render.render(scene, cam, spp, depth, seed=seed, flags=O.FLAGS_MAIN, samples_per_unit=3)
    assert_bits((lin, rgb), (lin_o, rgb_o), "render")
    assert st["segments"] == segments
    ppm, _ = render.render_ppm(scene, cam, spp, depth, seed=seed, flags=O.FLAGS_MAIN, samples_per_unit=3)
    assert ppm == render.encode_ppm(rgb_o)
    png, _ = render.render_png(scene, cam, spp, depth, seed=seed, flags=O.FLAGS_MAIN, samples_per_unit=3)
    assert png == render.encode_png(rgb_o, device=0)
    with render.Progressive(scene, cam, spp, depth, seed=seed, flags=O.FLAGS_MAIN, samples_per_unit=3) as p:
        for n in (3, 3, 1):
            lin, rgb, _ = p.step(n)
    assert_bits((lin, rgb), (lin_o, rgb_o), "Progressive")
    cams = turntable(3, 32, 18)
    lin, rgb, st = render.render_frames(scene, cams, spp, depth, seed=seed, flags=O.FLAGS_MAIN, samples_per_unit=3)
    for f, c in enumerate(cams):
        want = O.render(scene, c, spp, depth, seed=seed, flags=O.FLAGS_MAIN, threads=8, samples_per_unit=3)
        assert_bits((lin[f], rgb[f]), want[:2], f"render_frames, frame {f}")


# ---------------------------------------------------------------- past 2^31 pixels

W_BIG, H_BIG = 65536, 33280        # 2^31 + 2^25 pixels; row 32768 starts at pixel 2^31
GIB = 1 << 30


def free_device_bytes():
    import torch
    return torch.cuda.mem_get_info(0)[0]


def need(nbytes, what):
    free = free_device_bytes()
    if free < nbytes:
        pytest.skip(f"{what} needs {nbytes / GIB:.1f} GiB of device memory, {free / GIB:.1f} GiB free")


def reference_rows(scene, cam, spp, depth, seed, flags, rows):
    """{row: (linear [W,3], rgb8 [W,3])} from the oracle's per-sample colours: each pixel's samples summed in sample
    order (one unit per pixel), the mean rule, rto_quantise -- without the full image on the host."""
    quantise = np.vectorize(lambda c, linear: O.lib().rto_quantise(float(c), int(linear)), otypes=[np.uint8])
    out = {}
    for r in rows:
        colors = OS.sample_colors(scene, cam, spp, depth, seed=seed, flags=flags, rows=(r, r + 1))[0]
        acc = np.zeros((cam.width, 3))
        for k in range(spp):
            acc = acc + colors[:, k]
        lin = acc / float(spp) if flags & O.F_MEAN_DIVIDE else acc * (1.0 / float(spp))
        out[r] = (lin, quantise(lin, bool(flags & O.F_QUANT_LINEAR)))
    return out


BIG_KERNELS = {"lane": (V.MIXED, 50, _abi.F_LANE_KERNEL), "lane2": (V.MIXED, 50, _abi.F_LANE2_KERNEL),
               "primary": (V.SMALL, 1, 0)}


@pytest.mark.parametrize("outputs", ["rgb8", "linear"])
@pytest.mark.parametrize("kernel", list(BIG_KERNELS))
def test_shard_past_two_to_the_31_pixels(kernel, outputs):
    """shard (1, 2, 32768): rows 32768 .. 33279 only, into full-size images.  Their Philox pixel indices are at least
    2^31 and their output offsets above 2^32 bytes; every other row keeps the sentinel."""
    import torch
    spheres, depth, extra = BIG_KERNELS[kernel]
    scene, cam, seed, flags = V.soa(spheres), V.mixed_camera(W_BIG, H_BIG), 0x9E3779B97F4A7C15, O.FLAGS_MAIN
    npix = W_BIG * H_BIG
    want_lin = outputs == "linear"
    need(npix * 3 * (9 if want_lin else 1) + 4 * GIB, f"{W_BIG} x {H_BIG} {outputs}")
    ctx = context(scene)
    try:
        d_rgb = torch.full((H_BIG, W_BIG, 3), RGB_SENTINEL, dtype=torch.uint8, device="cuda:0")
        d_lin = torch.full((H_BIG, W_BIG, 3), LIN_SENTINEL, dtype=torch.float64, device="cuda:0") if want_lin else None
        stream = torch.cuda.current_stream().cuda_stream
        ctx.render(cam, 2, depth, seed=seed, flags=flags | extra, samples_per_unit=2, shard=(1, 2, 32768),
                   d_out_linear=d_lin.data_ptr() if want_lin else 0, d_out_rgb8=d_rgb.data_ptr(), stream=stream)
        st = ctx.stats(stream)
        assert st["samples"] == (H_BIG - 32768) * W_BIG * 2
        want = reference_rows(scene, cam, 2, depth, seed, flags, (32768, 32769, H_BIG - 1))
        for r, (lin_o, rgb_o) in want.items():
            assert np.array_equal(d_rgb[r].cpu().numpy(), rgb_o), f"row {r}: 8-bit image differs"
            if want_lin:
                assert_bits((d_lin[r].cpu().numpy(), rgb_o), (lin_o, rgb_o), f"row {r}")
        for r in (0, 1, 32767):
            assert (d_rgb[r] == RGB_SENTINEL).all(), f"row {r} is not in the shard"
            if want_lin:
                assert (d_lin[r] == LIN_SENTINEL).all(), f"row {r} is not in the shard"
    finally:
        ctx.close()
        d_rgb = d_lin = None
        torch.cuda.empty_cache()


def test_whole_image_past_two_to_the_31_pixels():
    """The whole 65536 x 33280 image on the primary-ray kernel, 8-bit only: 4.4 G samples, a count above 2^32.  Its
    unit sums take 52 GB of scratch."""
    import torch
    scene, cam, seed, flags = V.soa(V.SMALL), V.mixed_camera(W_BIG, H_BIG), (1 << 64) - 1, O.FLAGS_MAIN
    npix = W_BIG * H_BIG
    need(npix * (3 + 24) + 4 * GIB, f"a whole {W_BIG} x {H_BIG} render")
    ctx = context(scene)
    try:
        d_rgb = torch.full((H_BIG, W_BIG, 3), RGB_SENTINEL, dtype=torch.uint8, device="cuda:0")
        stream = torch.cuda.current_stream().cuda_stream
        ctx.render(cam, 2, 1, seed=seed, flags=flags, d_out_rgb8=d_rgb.data_ptr(), stream=stream)
        st = ctx.stats(stream)
        assert st["samples"] == npix * 2 and st["samples"] > 1 << 32 and st["segments"] == st["samples"]
        want = reference_rows(scene, cam, 2, 1, seed, flags, (0, 32767, 32768, 32769, H_BIG - 1))
        for r, (_, rgb_o) in want.items():
            assert np.array_equal(d_rgb[r].cpu().numpy(), rgb_o), f"row {r}: 8-bit image differs"
    finally:
        ctx.close()
        d_rgb = None
        torch.cuda.empty_cache()
