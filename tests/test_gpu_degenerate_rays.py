"""Degenerate and non-finite rays on every kernel, against the CPU oracle.

A ray whose fp32 |d|^2 lies outside [1e-30, 1e30] skips the cull and scans every sphere in fp64, in list order, with
the reference's acceptance rule (hittable.clj:15-21): `root <= t_min || t_max <= root` is false for a NaN root, so a
NaN root is accepted and every later body then wins (DESIGN.md section 4.1).  The camera's directions are not range
limited (DESIGN.md section 4.8), and scattering makes such rays from ordinary cameras: a metal reflection keeps |d| and
adds fuzz * U, and a dielectric of tiny ior refracting at normal incidence scales the direction's tangential part by
1 / ior.  The lambertian near-zero guard (material.clj:17) fires when U + N is below 1e-8 in every component; the
counter-based stream essentially never draws that, so one case places a sphere where it must.

tests/oracle_probe.py counts, in the oracle's own arithmetic, the scans of each case that take a degenerate direction
and those that accept a NaN root; every case asserts the counts it exists for, so that it cannot silently stop
covering its path.

Every render is compared with the oracle: the same NaN positions, identical bits everywhere else, the same 8-bit image
and the same segment and sample counts.  The sign and payload of a NaN are not compared."""
from types import SimpleNamespace

import numpy as np
import pytest

import oracle_lib as O
import oracle_probe as OP
from raytracing_clj_b200 import _abi, render
from test_gpu_adaptive import adaptive_run

pytestmark = pytest.mark.gpu
LAMB, METAL, DIEL = _abi.LAMBERTIAN, _abi.METAL, _abi.DIELECTRIC
HUGE = 1e300  # a tolerance no estimate exceeds: every pixel with a finite estimate stops at min_samples

# ---------------------------------------------------------------- helpers


def camera(p00, du=(0.0, 0.0, 0.0), dv=(0.0, 0.0, 0.0), w=8, h=4, center=(0.0, 0.0, 0.0)):
    """An rtclj_camera built field by field (oracle_lib.make_camera reads the same fields), without defocus."""
    z = (0.0, 0.0, 0.0)
    return SimpleNamespace(pixel00=tuple(p00), pixel_du=tuple(du), pixel_dv=tuple(dv), center=tuple(center),
                           defocus_u=z, defocus_v=z, defocus_angle=0.0, width=w, height=h)


def world(spheres, pad=0):
    """spheres: [(center, radius, kind, albedo, fuzz, ior)], in list order.  With `pad`, decoys behind the camera (on a
    ring at z = +60, which no camera ray of these cases comes near) come FIRST, up to `pad` spheres in all, so that the
    case's own spheres keep their order at the end of the list."""
    n_dec = max(0, pad - len(spheres))
    k = np.arange(n_dec)
    phi = k * 2.399963229728653
    decoys = [((20.0 * np.cos(p), 20.0 * np.sin(p), 60.0), 1.0, LAMB,
               tuple(0.1 + 0.8 * np.modf((i + 1) * np.array([0.618, 0.414, 0.732]))[0]), 0.0, 1.0)
              for i, p in zip(k, phi)]
    body = decoys + list(spheres)
    n = len(body)
    center = np.ascontiguousarray(np.array([b[0] for b in body], np.float64).reshape(n, 3))
    radius = np.array([b[1] for b in body], np.float64)
    kind = np.array([b[2] for b in body], np.int32)
    albedo = np.ascontiguousarray(np.array([b[3] for b in body], np.float64).reshape(n, 3))
    fuzz = np.array([b[4] for b in body], np.float64)
    ior = np.array([b[5] for b in body], np.float64)
    return center, radius, kind, albedo, fuzz, ior


def compare(got, want, what):
    """NaN-aware equality: the same NaN positions, identical bits elsewhere, the same 8-bit image and counters.
    got = (linear, rgb8, segments, samples), want likewise.  Returns the number of NaN values."""
    lin_g, rgb_g, seg_g, smp_g = got
    lin_w, rgb_w, seg_w, smp_w = want
    nan_g, nan_w = np.isnan(lin_g), np.isnan(lin_w)
    assert np.array_equal(nan_g, nan_w), f"{what}: NaN at {np.argwhere(nan_g != nan_w)[:4].tolist()} differs"
    bad = np.argwhere((lin_g.view(np.uint64) != lin_w.view(np.uint64)) & ~nan_w)
    assert bad.size == 0, (f"{what}: {len(bad)} linear values differ, first {bad[0].tolist()}: "
                           f"oracle {lin_w[tuple(bad[0])]!r} gpu {lin_g[tuple(bad[0])]!r}")
    assert np.array_equal(rgb_g, rgb_w), f"{what}: 8-bit image differs"
    assert (seg_g, smp_g) == (seg_w, smp_w), f"{what}: segments / samples {seg_g} / {smp_g}, oracle {seg_w} / {smp_w}"
    return int(nan_w.sum())


def oracle(scene, cam, spp, depth, seed, flags, unit=0):
    lin, rgb, st = O.render(scene, cam, spp, depth, seed=seed, flags=flags & 0xffff, threads=4,
                            samples_per_unit=unit or spp)
    return lin, rgb, st.segments, st.samples


def gpu(scene, cam, spp, depth, seed, flags, unit=0):
    lin, rgb, st = render.render(scene, cam, spp, depth, seed=seed, flags=flags, samples_per_unit=unit or spp)
    return lin, rgb, st["segments"], st["samples"]


# ---------------------------------------------------------------- the cases
#
# The camera sits at the origin.  The base scene is two spheres on the -z axis, the nearer first: a lambertian and,
# behind it, a metal.  An ordinary ray hits the lambertian; a ray whose scan meets a NaN root ends on the metal (the
# later body wins), which absorbs the NaN reflection at once -- a different colour and segment count.

BASE = [((0.0, 0.0, -1.0), 0.5, LAMB, (0.9, 0.3, 0.2), 0.0, 1.5),
        ((0.0, 0.0, -1.1), 0.5, METAL, (0.3, 0.5, 0.9), 0.2, 1.5)]
# A root is accepted above t_min = 1e-3 in units of |d|: a direction of length 1e16 reaches only bodies more than 1e13
# away.  The same pair, far down the axis, for the camera cases (at 1e100 and more every finite root is below t_min).
FAR = [((0.0, 0.0, -5e14), 2e14, LAMB, (0.7, 0.6, 0.2), 0.0, 1.5),
       ((0.0, 0.0, -6e14), 2e14, METAL, (0.2, 0.6, 0.7), 0.2, 1.5)]
GROUND = ((0.0, -100.5, -1.0), 100.0, LAMB, (0.5, 0.6, 0.4), 0.0, 1.5)


def view(s):
    """p00 - center = (0, 0, -s) and pixel steps of s / 1000: every primary direction has length about s."""
    return camera((0.0, 0.0, -s), (s * 1e-3, 0.0, 0.0), (0.0, -s * 1e-3, 0.0))


CAMERA_CASES = {
    "d0": (BASE + FAR, camera((0.0, 0.0, 0.0))),  # d = 0: every root is 0 / 0
    "tiny-1e-20": (BASE + FAR, view(1e-20)),      # fp32 |d|^2 underflows, a = 1e-40 is inside the division window
    "tiny-1e-80": (BASE + FAR, view(1e-80)),      # a = 1e-160: div_by / divs_by divide
    "huge-1e16": (BASE + FAR, view(1e16)),        # degenerate, everything finite
    "huge-1e100": (BASE + FAR, view(1e100)),      # a = 1e200 outside the division window, roots finite: sky
    "huge-1e200": (BASE + FAR, view(1e200)),      # a = inf: NaN roots
}
# (spheres, camera, depth, variants, NaN roots expected)
SCATTER_CASES = {
    # reflections of length ~1e200 after the first bounce, then a = inf: NaN roots
    "metal-fuzz-1e200": ([((0.0, 0.0, -1.0), 0.5, METAL, (0.8, 0.8, 0.8), 1e200, 1.5), GROUND] + BASE, view(1.0), 10,
                         ("main", "realm"), True),
    # a camera inside a metal sphere: the first reflection that is not absorbed has |d| ~ 1e16 (degenerate, finite)
    "inside-metal-fuzz-1e16": ([((0.0, 0.0, 0.0), 10.0, METAL, (0.9, 0.8, 0.7), 1e16, 1.5),
                                ((0.0, 0.0, -3.0), 1.0, LAMB, (0.2, 0.7, 0.3), 0.0, 1.5)] + BASE, view(1.0), 50,
                               ("main", "realm"), False),
    # Within ~1e-8 rad of the normal, cos_theta rounds to 1 and sin_theta to 0, so even ri = 1 / ior = 1e300 refracts:
    # the tangential part, ~1e-12, times 1e300 overflows |perp|^2, and the next direction has |d|^2 = inf.  Realm only:
    # main's Schlick term is r0 = 1 at normal incidence for this ior, so main always reflects.
    "dielectric-ior-1e-300": ([((0.0, 0.0, -1.0), 0.5, DIEL, (1.0, 1.0, 1.0), 0.0, 1e-300), GROUND] + BASE,
                              camera((0.0, 0.0, -1.0), (1e-12, 0.0, 0.0), (0.0, -1e-12, 0.0)), 10, ("realm",), True),
}
VARIANTS = {"main": (O.FLAGS_MAIN, 10), "realm": (O.FLAGS_REALM, 10), "i": (O.FLAGS_I, 10), "main-depth1": (O.FLAGS_MAIN, 1)}
KERNELS = {"auto": 0, "lane": _abi.F_LANE_KERNEL, "lane2": _abi.F_LANE2_KERNEL, "wave": _abi.F_WAVE_KERNEL,
           "split": _abi.F_SPLIT_KERNEL, "smem": _abi.F_SMEM_TABLE, "nocull": _abi.F_NO_CULL}
PADS = (0, 64, 600)


def kernels_for(n):
    """Above 512 spheres every kernel flag selects the shared-table kernel: run it and the exhaustive scan."""
    return {k: KERNELS[k] for k in ("auto", "nocull")} if n > 512 else KERNELS


def check_kernels(scene, cam, spp, depth, seed, flags, what):
    """Every kernel against the oracle; reports every kernel that differs.  Returns (oracle result, NaN count)."""
    want = oracle(scene, cam, spp, depth, seed, flags)
    failed, nans = [], 0
    for name, extra in kernels_for(len(scene[1])).items():
        try:
            nans = compare(gpu(scene, cam, spp, depth, seed, flags | extra), want, f"{what} [{name}]")
        except AssertionError as e:
            failed.append(str(e))
    assert not failed, "\n".join(failed)
    return want, nans


# (case, variant) pairs whose oracle image must contain NaN: the tests fail instead of silently losing it
MUST_NAN = {("d0", "i"), ("huge-1e200", "i")}
# camera cases whose scans accept NaN roots (in the oracle's arithmetic)
NAN_ROOTS = {"d0", "huge-1e200"}


def assert_reaches(scene, cam, spp, depth, seed, flags, degenerate, nan_roots):
    """The oracle's scans of this render: `degenerate` = the least number that take a degenerate direction,
    `nan_roots` = whether some accept a NaN root (None: either)."""
    p = OP.scans(scene, cam, spp, depth, seed, flags)
    assert p["degenerate"] >= degenerate, p
    if nan_roots is not None:
        assert (p["nan_roots"] > 0) == nan_roots, p
    return p


@pytest.mark.parametrize("pad", PADS)
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("case", list(CAMERA_CASES))
def test_degenerate_camera_directions(case, variant, pad):
    spheres, cam = CAMERA_CASES[case]
    flags, depth = VARIANTS[variant]
    scene = world(spheres, pad)
    seed = 11 + PADS.index(pad)
    # every camera ray is degenerate
    assert_reaches(scene, cam, 4, depth, seed, flags, cam.width * cam.height * 4, case in NAN_ROOTS)
    _, nans = check_kernels(scene, cam, 4, depth, seed, flags, f"{case} {variant} pad {pad}")
    if (case, variant) in MUST_NAN:
        assert nans > 0, "the case no longer produces a NaN root"


SCATTER_PARAMS = [(c, v) for c, case in SCATTER_CASES.items() for v in case[3]]


@pytest.mark.parametrize("pad", PADS)
@pytest.mark.parametrize("case,variant", SCATTER_PARAMS, ids=[f"{c}-{v}" for c, v in SCATTER_PARAMS])
def test_directions_made_by_scattering(case, variant, pad):
    spheres, cam, depth, _, nan_roots = SCATTER_CASES[case]
    flags = VARIANTS[variant][0]
    scene = world(spheres, pad)
    seed = 21 + PADS.index(pad)
    assert_reaches(scene, cam, 4, depth, seed, flags, 1, nan_roots)
    check_kernels(scene, cam, 4, depth, seed, flags, f"{case} {variant} pad {pad}")


# ---------------------------------------------------------------- the near-zero guard, engineered
#
# All camera rays of the guard camera share the direction U = the lambertian unit vector the oracle draws for
# (pixel 0, sample 0, stage 1), and the first sphere is placed so that the ray meets it at normal N = -U.  At that
# scatter U + N cancels to rounding error: main's guard replaces it by N; realm traces it, a direction of length
# ~1e-16, which takes the degenerate scan.


def unit_vector(seed, pixel, sample, stage):
    """vec3a/random-unit-vec3 with the kernels' rejection rule (rtclj_render_body.cuh, oracle random_unit)."""
    block = 0
    while True:
        w = O.philox((pixel, sample, stage, block), (seed & 0xffffffff, seed >> 32))
        for half in range(2):
            bits = w[2 * half] | (w[2 * half + 1] << 32)
            x, y, z = (-1.0 + 2.0 * (float((bits >> s) & 0x1FFFFF) * (1.0 / 2097152.0)) for s in (0, 21, 42))
            l2 = x * x + y * y + z * z
            if 1e-160 < l2 <= 1.0:
                q = np.sqrt(l2)
                return (x / q, y / q, z / q)
        block += 1


GUARD_SEED, T0, RAD = 5, 1.25, 0.75  # (at t0 = r = 1 the sum cancels to exactly 0, which "d0" covers)


def guard_case():
    """The scene's spheres and camera, and (U + N) of pixel 0, sample 0's first scatter, replayed in float64 with
    the oracle's operations (hittable.clj:9-31)."""
    U = unit_vector(GUARD_SEED, 0, 0, 1)
    C = tuple((T0 + RAD) * u for u in U)
    spheres = [(C, RAD, LAMB, (0.8, 0.4, 0.2), 0.0, 1.5),
               (tuple(-3.0 * u for u in U), 1.0, LAMB, (0.2, 0.4, 0.8), 0.0, 1.5)]  # behind the camera, later in the list
    d, oc = np.array(U), np.array(C)
    a = d[0] * d[0] + d[1] * d[1] + d[2] * d[2]
    h = d[0] * oc[0] + d[1] * oc[1] + d[2] * oc[2]
    c = (oc[0] * oc[0] + oc[1] * oc[1] + oc[2] * oc[2]) - RAD * RAD
    root = (h - np.sqrt(h * h - a * c)) / a
    assert root > 1e-3
    P = d * root
    outward = (P - oc) / RAD
    front = (d[0] * outward[0] + d[1] * outward[1] + d[2] * outward[2]) < 0.0
    N = outward if front else -outward
    return spheres, camera(U), d + N


@pytest.mark.parametrize("pad", PADS)
@pytest.mark.parametrize("variant", ["main", "realm"])
def test_near_zero_guard(variant, pad):
    spheres, cam, _ = guard_case()
    flags, depth = VARIANTS[variant]
    scene = world(spheres, pad)
    # realm traces U + N (degenerate); main's guard replaces it by N, so no scan of main is degenerate
    p = assert_reaches(scene, cam, 4, depth, GUARD_SEED, flags, 1 if variant == "realm" else 0, None)
    assert variant == "realm" or p["degenerate"] == 0, p
    check_kernels(scene, cam, 4, depth, GUARD_SEED, flags, f"guard {variant} pad {pad}")
    if variant == "main":
        # the guard decides pixel 0: without it the pixel differs (and still equals the oracle's unguarded render)
        flags_off = flags & ~O.F_NEAR_ZERO_GUARD
        with_guard = gpu(scene, cam, 4, depth, GUARD_SEED, flags)
        without = gpu(scene, cam, 4, depth, GUARD_SEED, flags_off)
        compare(without, oracle(scene, cam, 4, depth, GUARD_SEED, flags_off), "guard off")
        assert not np.array_equal(with_guard[0][0, 0].view(np.uint64), without[0][0, 0].view(np.uint64))
        assert np.array_equal(with_guard[0][1:].view(np.uint64), without[0][1:].view(np.uint64))


# ---------------------------------------------------------------- strict order through the sample buffer

STRICT = [("d0", "realm"), ("huge-1e200", "main"), ("metal-fuzz-1e200", "main"), ("guard", "realm")]


@pytest.mark.parametrize("case,variant", STRICT, ids=[f"{c}-{v}" for c, v in STRICT])
def test_strict_order(case, variant):
    """64 samples per pixel in one unit: every sample's colour through the sample buffer, added in sample order."""
    if case == "guard":
        spheres, cam, _ = guard_case()
        depth = 10
    elif case in CAMERA_CASES:
        spheres, cam = CAMERA_CASES[case]
        depth = 10
    else:
        spheres, cam, depth = SCATTER_CASES[case][:3]
    flags = VARIANTS[variant][0]
    for pad in (0, 64):
        scene = world(spheres, pad)
        want = oracle(scene, cam, 64, depth, 31, flags)
        for name in ("auto", "lane", "lane2", "split", "smem"):
            compare(gpu(scene, cam, 64, depth, 31, flags | KERNELS[name]), want, f"strict {case} pad {pad} [{name}]")


# ---------------------------------------------------------------- adaptive accumulation: the listed kernels
#
# Columns of the mixed camera: |d| ~ 1e154 * x, so column 0 keeps a finite |d|^2 (a sky pixel on the -i scene), from
# column 2 on |d|^2 = inf and every sphere's root is NaN; in column 1 it depends on the jitter.  A pixel whose sums are
# NaN counts as noisy (DESIGN.md section 4.10): it runs to spp while the others stop at min_samples.  (Decoys would
# make every column NaN: their |oc| of ~60 puts h^2 over the fp64 range already in column 0.)

MIXED = ([((1.0, 0.0, -5.0), 0.5, LAMB, (0.9, 0.3, 0.2), 0.0, 1.5),
          ((1.0, 0.3, -5.5), 0.5, METAL, (0.3, 0.5, 0.9), 0.2, 1.5)],
         camera((0.0, 0.0, -1.0), (1e154, 0.0, 0.0), (0.0, -0.05, 0.0)))
ADAPTIVE = [("i-primary", O.FLAGS_I, 0), ("i-lane", O.FLAGS_I | _abi.F_LANE_KERNEL, 0),
            ("i-lane2", O.FLAGS_I | _abi.F_LANE2_KERNEL, 0), ("i-smem", O.FLAGS_I | _abi.F_SMEM_TABLE, 0),
            ("main-depth1-primary", O.FLAGS_MAIN, 0), ("realm-pad64", O.FLAGS_REALM, 64),
            ("realm-pad600", O.FLAGS_REALM, 600)]


@pytest.mark.parametrize("order", ["chunked", "strict"])
@pytest.mark.parametrize("name,flags,pad", ADAPTIVE, ids=[a[0] for a in ADAPTIVE])
def test_adaptive_accumulation(name, flags, pad, order):
    """Every pixel exact at its own count after every pass; NaN pixels run to spp, the others stop at min_samples
    (a tolerance no finite estimate exceeds)."""
    spheres, cam = MIXED
    scene = world(spheres, pad)
    passes = (4, 4, 4, 4)
    spp = sum(passes)
    depth = 1 if "depth1" in name else 10
    strict = order == "strict"
    unit, least = (spp, 4) if strict else (4, 8)  # (chunked: an estimate needs two units)
    run = adaptive_run(scene, cam, passes, depth, 41, flags, unit, (HUGE, 0.0), least)
    for d, lin, rgb, samples, _, active, _ in run:
        for n in np.unique(samples):
            assert 0 < n <= d, (n, d)
            m = samples == n
            want = oracle(scene, cam, int(n), depth, 41, flags, int(n) if strict else unit)
            compare((lin[m], rgb[m], 0, 0), (want[0][m], want[1][m], 0, 0), f"{name} after {d}: {m.sum()} pixels of {n}")
        nan_px = np.isnan(lin).any(axis=2)  # a NaN pixel stays NaN: it never stopped
        assert (samples[nan_px] == d).all(), (d, samples)
        assert (samples[~nan_px] == min(d, least)).all(), (d, samples)
        assert active == (0 if d == spp else cam.width * cam.height if d < least else int(nan_px.sum())), (d, active)
    if flags & O.F_NORMAL_SHADING:
        assert nan_px.any() and not nan_px.all(), nan_px
