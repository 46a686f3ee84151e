"""The shared-memory-table kernel (render_kernel<false>, every scene of more than 512 spheres) at its edges: survivor
lists that fill up and are resolved in several rounds ("flushes"), the boundary between the part of the table staged
in shared memory and the part read from global memory, the largest scene the 16-bit list entries allow, and the
prefilter candidate pushed out of its three slots.  Every render is compared with the CPU oracle (linear bits, 8-bit
image, segment count) and with the same render under RTCLJ_F_NO_CULL.

Bead scenes make the survivor set of every primary ray known exactly, so that tests/cull_walk_model.py can show which
rounds a ray takes and where each starts."""
import os

import numpy as np
import pytest

import cull_walk_model as M
import oracle_lib as O
import raytracing_clj_b200 as R
from raytracing_clj_b200 import _abi, render
from test_gpu_adaptive import adaptive_run, check_groups, median_tolerance
from test_gpu_progressive import context

pytestmark = pytest.mark.gpu
S_, CAM = R.scenes, R.camera


@pytest.fixture(scope="module")
def S():
    """Blocks of 32 spheres staged in shared memory, from this device's opt-in limit and the library's formula."""
    import torch
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    s = M.smem_table_blocks(optin)
    print(f"\nshared-memory opt-in {optin} B: S = {s} blocks ({32 * s} spheres)")
    # the cases below need a global part well below the largest scene, and room for 8 blocks before it
    assert 16 <= s and 32 * s + 48 < M.C["max_spheres"] - 64, s
    return s


# ---------------------------------------------------------------- helpers


def soa(center, radius, albedo, kind=None, ior=None):
    n = len(radius)
    kind = np.zeros(n, np.int32) if kind is None else np.asarray(kind, np.int32)
    ior = np.ones(n) if ior is None else np.asarray(ior, np.float64)
    return tuple(np.ascontiguousarray(a) for a in (np.asarray(center, np.float64).reshape(n, 3),
                                                   np.asarray(radius, np.float64), kind,
                                                   np.asarray(albedo, np.float64).reshape(n, 3), np.zeros(n), ior))


def assert_exact(scene, cam, spp, depth, seed, flags, unit=0):
    """The render against the oracle (bits of the linear image, 8-bit image, segments) and against the exhaustive
    fp64 scan (RTCLJ_F_NO_CULL).  Returns the stats of the culled render."""
    unit = unit or spp
    lin_o, rgb_o, st_o = O.render(scene, cam, spp, depth, seed=seed, flags=flags & 0xffff, threads=8,
                                  samples_per_unit=unit)
    lin, rgb, st = render.render(scene, cam, spp, depth, seed=seed, flags=flags, samples_per_unit=unit)
    bad = np.argwhere(lin.view(np.uint64) != lin_o.view(np.uint64))
    assert bad.size == 0, (f"{len(bad)} of {lin.size} linear values differ from the oracle; first {bad[0]}: "
                           f"oracle {lin_o[tuple(bad[0])]!r} gpu {lin[tuple(bad[0])]!r}")
    assert np.array_equal(rgb, rgb_o) and st["segments"] == st_o.segments
    lin_x, rgb_x, st_x = render.render(scene, cam, spp, depth, seed=seed, flags=flags | _abi.F_NO_CULL,
                                       samples_per_unit=unit)
    assert np.array_equal(lin.view(np.uint64), lin_x.view(np.uint64)) and np.array_equal(rgb, rgb_x)
    assert st_x["segments"] == st["segments"] and st_x["exact_tests"] == st_x["segments"] * len(scene[1])
    return st


# ---------------------------------------------------------------- bead scenes
#
# The camera sits at the origin and looks down -z, without defocus, with a vertical field of 2 degrees.  At 32 x 16
# pixels (or narrower) every primary direction, pixel jitter included, is within atan(sqrt(tan^2 2 + tan^2 1)) < 2.3
# degrees of the axis: sin < 0.04.
#
# Beads are spheres centred on the axis at depth Z = 100, of radius 20 to 60.  A primary ray's line passes within
# 100 * 0.04 = 4 of their centre, so it crosses every bead with a margin of at least 16 in distance (and it is hit
# from outside: the camera is 100 from the centre).  Being crossed, a bead survives the conservative cull whatever its
# rounding.  The stale ray of an idle lane (origin 0, direction +z) lies on the axis and crosses them too.
#
# Decoys sit on a ring of radius 1000 around the axis at the same depth, with radius 2: every primary line stays
# more than 990 away from their centres, so their true discriminant r^2 - dist^2 is below -9.8e5.  The cull inflates
# it by less than 76 eps (|c|^2 + |o|^2) + 5 eps r^2 (DESIGN.md, "cull error bound") with |c|, |o| < 2200 after the
# host's shift: below 25, four orders of magnitude short.  So a primary ray's survivors are exactly the beads, which
# the test asserts through the prefilter counter.
#
# All beads share a centre, so the nearest hit is the bead of the largest radius (60); the others have distinct radii
# below it.  Each sphere has its own lambertian albedo, so a wrong winner changes the pixel.

Z, R_NEAR, RING = 100.0, 60.0, 1000.0


def bead_camera(w=32, h=16):
    return CAM.main_camera(w, h, vfov=2.0, look_from=(0.0, 0.0, 0.0), look_at=(0.0, 0.0, -1.0), defocus_angle=0.0,
                           focus_dist=1.0)


def bead_index(n, half):
    """The bead of half block `half`: a different bit position from block to block."""
    return min(16 * half + half % 16, n - 1)


def bead_scene(n, halves, nearest, tie=None, extra=()):
    """Decoys everywhere, a bead in each half block of `halves` and at the indices `extra`; the bead of half block
    `nearest` is the nearest.  With `tie`, the bead of that half block is the same sphere as the nearest one, with
    another albedo."""
    idx = np.arange(n)
    phi = idx * 2.399963229728653  # golden angle: the decoys spread evenly over the ring
    center = np.stack([RING * np.cos(phi), RING * np.sin(phi), np.full(n, -Z)], axis=1)
    radius = np.full(n, 2.0)
    albedo = 0.1 + 0.8 * np.modf(np.outer(idx + 1, [0.6180339887, 0.4142135623, 0.7320508075]))[0]
    beads = sorted({bead_index(n, h) for h in halves} | set(extra))
    assert all(i // 16 in halves for i in extra)
    center[beads] = (0.0, 0.0, -Z)
    radius[beads] = 20.0 + 38.0 * (1 + np.arange(len(beads))[::-1]) / (len(beads) + 1)  # (20, 58], distinct
    radius[bead_index(n, nearest)] = R_NEAR
    if tie is not None:
        radius[bead_index(n, tie)] = R_NEAR
    return soa(center, radius, albedo), len(beads)


# Sizes: just above 512 (the smallest scenes of this kernel, tails of 1 and 16 spheres), and around the shared-memory
# boundary 32 S: the tail in shared memory, no global part, the tail as the only global read (1 or 16 spheres), a
# global block (17 spheres past 32 S), a global block and a global tail.  Then the largest scenes.
SIZES = {"513": lambda s: 513, "560": lambda s: 560, "32S-16": lambda s: 32 * s - 16, "32S": lambda s: 32 * s,
         "32S+1": lambda s: 32 * s + 1, "32S+16": lambda s: 32 * s + 16, "32S+17": lambda s: 32 * s + 17,
         "32S+48": lambda s: 32 * s + 48, "65520": lambda s: 65520, "65532": lambda s: 65532}


def case_layout(case, n, s):
    """(surviving half blocks, half block of the nearest bead, half block of its tie or None)."""
    nb, tail = M.layout(n)
    nh = 2 * nb + tail
    if case == "nearest-last":
        return list(range(nh)), nh - 1, None
    if case == "nearest-first":
        return list(range(nh)), 0, None
    if case == "tie":
        return list(range(nh)), 0, nh - 1
    if case == "round-at-S":  # 8 full blocks just before S, then survivors everywhere past it
        e = min(s, nb)
        return list(range(2 * e - 16, nh)), 2 * e, None
    if case == "tail-pending":  # 8 full blocks at the end fill the list before the tail
        return list(range(2 * nb - 16, nh)), nh - 1, None
    if case == "many-rounds":  # one entry per block: 14 blocks per round
        return list(range(0, nh, 2)), 2 * (nb // 2), None
    if case == "max-index":  # survivors decode from half block 4095
        return [0, 4095], 4095, None
    raise KeyError(case)


def reaches(case, rounds, n, s, nearest, tie):
    """The path each case is for, shown on the model's rounds."""
    nb, tail = M.layout(n)
    where = M.round_of_half(rounds, nearest)
    if case == "nearest-last":
        return len(rounds) >= 2 and where == len(rounds) - 1
    if case == "nearest-first":
        return len(rounds) >= 2 and where == 0
    if case == "tie":
        return where < M.round_of_half(rounds, tie)
    if case == "round-at-S":
        k = next((k for k, r in enumerate(rounds) if k and r.start == s), None)
        return k is not None and (nb > s or M.tail_is_global(n, s)) and where == k
    if case == "tail-pending":
        return len(rounds) >= 2 and rounds[-1] == M.Round(nb, nb, (2 * nb,), True, ()) and where == len(rounds) - 1
    if case == "many-rounds":
        return len(rounds) > 16 and 0 < where < len(rounds) - 1
    if case == "max-index":
        return n == M.C["max_spheres"] and nearest == (n - 1) // 16 == 4095
    raise KeyError(case)


def _bead_params():
    out = []
    for size in SIZES:
        cases = ["nearest-last", "nearest-first", "tie"]
        if size in ("513", "560", "32S-16", "32S+1", "32S+16", "32S+48", "65520"):
            cases.append("tail-pending")
        if size in ("32S+1", "32S+16", "32S+17", "32S+48"):
            cases.append("round-at-S")
        if size.startswith("32S"):
            cases.append("many-rounds")
        if size == "65520":
            cases = ["nearest-last", "tail-pending"]
        if size == "65532":
            cases = ["nearest-last", "max-index"]
        out += [(size, case) for case in cases]
    return out


BEAD_PARAMS = _bead_params()


@pytest.mark.parametrize("size,case", BEAD_PARAMS, ids=[f"{s}-{c}" for s, c in BEAD_PARAMS])
def test_bead_scene(size, case, S):
    n = SIZES[size](S)
    halves, nearest, tie = case_layout(case, n, S)
    extra = ()
    if case == "max-index":  # beads at 65 520 and 65 531, both in the last half block; the latter is nearest
        extra = (65520,)
        assert bead_index(n, 4095) == n - 1 == 65531
    rounds = M.walk(n, S, halves)
    assert reaches(case, rounds, n, S, nearest, tie), [(r.start, r.stop, len(r.halves), r.tail) for r in rounds]
    scene, nbeads = bead_scene(n, halves, nearest, tie, extra)
    small = n > 60000  # the oracle's cost grows with n
    cam = bead_camera(16, 8) if small else bead_camera()
    spp = 1 if small else 2
    k = BEAD_PARAMS.index((size, case))
    flags, depth = (O.FLAGS_MAIN, O.FLAGS_REALM)[k % 2], 2 + k % 4
    st = assert_exact(scene, cam, spp, depth, 100 + k, flags)
    assert st["exact_tests"] < st["segments"] * n // 8, st
    # primary rays only: every segment's survivors are the beads, so the model's rounds are every segment's rounds
    st = assert_exact(scene, cam, spp, 1, 200 + k, O.FLAGS_I)
    segs = cam.width * cam.height * spp
    assert st["segments"] == segs
    assert st["prefilter_tests"] == segs * nbeads, (st["prefilter_tests"], segs, nbeads)
    assert segs <= st["exact_tests"] <= segs * nbeads
    # a lower bound: idle lanes of a warp cull their stale rays as well, and count
    assert st["list_overflows"] >= segs * (len(rounds) - 1), (st["list_overflows"], segs, len(rounds))
    print(f"\n{size} {case}: n = {n}, model rounds {len(rounds)}, segments {segs}, "
          f"list_overflows {st['list_overflows']} (>= {segs * (len(rounds) - 1)})")


def test_more_than_the_largest_scene_is_refused():
    n = M.C["max_spheres"] + 1
    scene = soa(np.zeros((n, 3)) + (0.0, 0.0, -5.0), np.ones(n), np.full((n, 3), 0.5))
    with pytest.raises(_abi.RtcljError) as e:
        render.render(scene, bead_camera(4, 2), 1, 1, flags=O.FLAGS_I)
    assert e.value.code == _abi.E_TOO_LARGE


# ---------------------------------------------------------------- the displaced prefilter candidate
#
# Three glass spheres of index of refraction 1 (transparent) centred on the camera contain it and everything else.
# Their near root is negative, so their lower bound is below that of any sphere in front: they take the prefilter's
# three slots, and the bead in front -- the winner -- is pushed out and tested on the spot.

SMALL_KERNELS = {"lane": _abi.F_LANE_KERNEL, "lane2": _abi.F_LANE2_KERNEL, "wave": _abi.F_WAVE_KERNEL,
                 "split": _abi.F_SPLIT_KERNEL, "smem": _abi.F_SMEM_TABLE}
DISPLACED = [(k, n, order) for k in SMALL_KERNELS for n in (40, 300) for order in ("bead-first", "bead-last")]
DISPLACED += [("smem", 600, "bead-first"), ("smem", 600, "bead-last")]


@pytest.mark.parametrize("kernel,n,order", DISPLACED, ids=[f"{k}-{n}-{o}" for k, n, o in DISPLACED])
def test_displaced_candidate_wins(kernel, n, order):
    idx = np.arange(n)
    phi = idx * 2.399963229728653
    center = np.stack([RING * np.cos(phi), RING * np.sin(phi), np.full(n, -Z)], axis=1)
    radius = np.full(n, 2.0)
    albedo = 0.1 + 0.8 * np.modf(np.outer(idx + 1, [0.6180339887, 0.4142135623, 0.7320508075]))[0]
    kind, ior = np.zeros(n, np.int32), np.ones(n)
    bead, shells = (0, [1, n // 2, n - 1]) if order == "bead-first" else (n - 1, [0, 1, n // 2])
    center[bead], radius[bead] = (0.0, 0.0, -Z), 30.0
    for j, i in enumerate(shells):
        center[i], radius[i], kind[i] = (0.0, 0.0, 0.0), 4 * RING + j, _abi.DIELECTRIC
    scene = soa(center, radius, albedo, kind, ior)
    cam = bead_camera(24, 12)
    st = assert_exact(scene, cam, 2, 1, 7, O.FLAGS_I | SMALL_KERNELS[kernel])
    segs = cam.width * cam.height * 2
    # four survivors per ray; with three slots, one of the four exact tests is the on-the-spot one
    assert st["segments"] == segs and st["prefilter_tests"] == 4 * segs and st["exact_tests"] == 4 * segs, st
    # paths through the bead and out through the three shells to the sky
    assert_exact(scene, cam, 2, 6, 8, O.FLAGS_REALM | SMALL_KERNELS[kernel])


# ---------------------------------------------------------------- fuzz past 513 spheres


def fuzz_world(rng, n, case):
    """test_gpu_parity.test_cull_fuzz_against_exhaustive_scan's scenes and cameras, at n spheres."""
    sp, mat = R.hittable.sphere, R.material
    scale = 10.0 ** rng.uniform(-3, 9)
    spread = scale * 10.0 ** rng.uniform(-2, 2)
    offset = rng.normal(size=3) * scale * (0 if case % 3 else 1e3)
    world = []
    for i in range(n):
        c = offset + rng.normal(size=3) * spread * (0.01 if rng.random() < 0.2 else 1.0)
        if world and rng.random() < 0.1:
            c = np.array(world[-1]["hittable/center"])
        r = scale * 10.0 ** rng.uniform(-3, 1) * (-1 if rng.random() < 0.05 else 1)
        kind = rng.integers(0, 3)
        m = (mat.lambertian(tuple(rng.random(3))) if kind == 0 else
             mat.metal(tuple(rng.random(3)), float(rng.random() * 1.2)) if kind == 1 else
             mat.dielectric(float(rng.uniform(0.5, 2.5))))
        world.append(S_.body(sp(tuple(float(x) for x in c), float(r)), m))
    pick = np.array(world[int(rng.integers(0, n))]["hittable/center"])
    where = rng.integers(0, 3)
    look_from = (pick + rng.normal(size=3) * scale * 1e-4 if where == 0 else
                 pick + rng.normal(size=3) * spread * 3 if where == 1 else
                 offset + rng.normal(size=3) * spread * 10.0 ** rng.uniform(1, 4))
    cam = CAM.main_camera(48, 27, vfov=float(rng.uniform(1, 120)), look_from=tuple(float(x) for x in look_from),
                          look_at=tuple(float(x) for x in pick), defocus_angle=float(rng.choice([0.0, 2.0])),
                          focus_dist=float(np.linalg.norm(look_from - pick) + 1e-9 * scale))
    return S_.to_soa(world), cam, scale


def test_cull_fuzz_past_513_spheres(S):
    """The fuzz of test_gpu_parity at 600, 2 000, about 32 S and 20 000 spheres: against RTCLJ_F_NO_CULL every time,
    against the oracle on every fourth case.  RTCLJ_FUZZ_CASES scales it as it scales that fuzz (a third of it)."""
    rng = np.random.default_rng(20261020)
    cases = max(4, int(os.environ.get("RTCLJ_FUZZ_CASES", "48")) // 3)
    for case in range(cases):
        n = (600, 2000, 32 * S + int(rng.integers(-32, 49)), 20000)[case % 4]
        scene, cam, scale = fuzz_world(rng, n, case)
        variant = O.FLAGS_REALM if case % 2 else O.FLAGS_MAIN
        a, ra, sa = render.render(scene, cam, 4, 12, seed=case, flags=variant, samples_per_unit=4)
        b, rb, sb = render.render(scene, cam, 4, 12, seed=case, flags=variant | _abi.F_NO_CULL, samples_per_unit=4)
        assert sa["segments"] == sb["segments"] and np.array_equal(a, b, equal_nan=True), (case, n, scale)
        assert np.array_equal(ra, rb), (case, n, scale)
        if case % 4 == case // 4 % 4:  # a quarter of the cases, every size in turn
            lo, ro, so = O.render(scene, cam, 4, 12, seed=case, flags=variant, threads=8, samples_per_unit=4)
            assert so.segments == sa["segments"] and np.array_equal(lo, a, equal_nan=True) and np.array_equal(ro, ra), \
                (case, n, scale)


# ---------------------------------------------------------------- the twins at the boundary


def boundary_scene(s):
    n = 32 * s + 16  # S blocks in shared memory, the tail global; a round starts at block S
    halves, nearest, _ = case_layout("round-at-S", n, s)
    rounds = M.walk(n, s, halves)
    assert reaches("round-at-S", rounds, n, s, nearest, None)
    return bead_scene(n, halves, nearest)[0]


def test_strict_order_at_the_boundary(S):
    """64 samples per pixel in one unit: the strict order, traced through the sample buffer
    (render_kernel<false, true>) and added in sample order, against the oracle's strict sum."""
    assert_exact(boundary_scene(S), bead_camera(16, 8), 64, 3, 41, O.FLAGS_MAIN)


def test_adaptive_accumulation_at_the_boundary(S):
    """An adaptive accumulation (render_listed_kernel<false>): every pixel exact at its own count."""
    scene, cam = boundary_scene(S), bead_camera()
    passes, unit, least, depth, seed, flags = (8, 4, 4), 4, 8, 3, 43, O.FLAGS_MAIN
    tol = median_tolerance(scene, cam, passes, depth, seed, flags, unit, least)
    run = adaptive_run(scene, cam, passes, depth, seed, flags, unit, tol, least)
    ref = context(scene)
    counts = None
    for d, lin, rgb, samples, _, _, _ in run:
        counts = check_groups(ref, cam, d, lin, rgb, samples, depth, seed, flags, unit, False)
    ref.close()
    assert len(counts) >= 2, counts
    # and the one-shot render of the full count against the oracle
    assert_exact(scene, cam, sum(passes), depth, seed, flags, unit=unit)
