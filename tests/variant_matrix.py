"""Scenes, flag combinations and seeds for the variant-switch matrix (tests/test_variant_matrix.py on the CPU,
tests/test_gpu_variant_matrix.py on the GPU).

The six switches of rtclj_params.flags are independent: the oracle implements each one separately
(oracle/rt_oracle.c), and so must every kernel.  The scenes here are built so that each switch changes the image:
an spp that is not a power of two (MEAN_DIVIDE: sum / spp and sum * (1 / spp) round differently), paths of several
attenuating hits of different albedo (REVERSE_PRODUCT), glass at grazing angles and an ior < 1 sphere
(SCHLICK), and the engineered near-zero scatter of test_gpu_degenerate_rays.guard_case (NEAR_ZERO_GUARD).  The
material fields a kind ignores hold large finite garbage: a dielectric's albedo, a lambertian's fuzz and a metal's
ior.  A kernel that reads one of them changes the image."""
from __future__ import annotations

import functools

import numpy as np

import oracle_lib as O
import raytracing_clj_b200 as R
from raytracing_clj_b200 import _abi
from test_gpu_degenerate_rays import GUARD_SEED, guard_case

CAM = R.camera
LAMB, METAL, DIEL = _abi.LAMBERTIAN, _abi.METAL, _abi.DIELECTRIC
BITS = {"NEAR_ZERO_GUARD": O.F_NEAR_ZERO_GUARD, "SCHLICK": O.F_SCHLICK, "REVERSE_PRODUCT": O.F_REVERSE_PRODUCT,
        "MEAN_DIVIDE": O.F_MEAN_DIVIDE, "NORMAL_SHADING": O.F_NORMAL_SHADING, "QUANT_LINEAR": O.F_QUANT_LINEAR}
ALL_COMBOS = list(range(64))

# A strength-2 covering array of the six switches: the columns a, b, c, a^b, a^c, b^c of the 2^3 full factorial
# (row r: a, b, c = bits 0, 1, 2 of r).  Any two columns are independent over GF(2), so every pair of switches takes
# each of its four value pairs (twice).
COVERING = [sum(bit << k for k, bit in enumerate((a, b, c, a ^ b, a ^ c, b ^ c)))
            for a, b, c in ((r & 1, (r >> 1) & 1, (r >> 2) & 1) for r in range(8))]
# the rows of the larger regimes: the covering array and the reference's three programs
PAIRWISE = COVERING + [O.FLAGS_MAIN, O.FLAGS_REALM, O.FLAGS_I]

# Seeds across the 64-bit Philox key: k0 = the low word, k1 = the high word.  The rounds add 0x9E3779B9 to k0 and
# 0xBB67AE85 to k1; K0_WRAP and K1_WRAP make the round key of the last round (r = 9) wrap to 0 in one word.
K0_WRAP = (0x12345678 << 32) | ((-9 * 0x9E3779B9) & 0xFFFFFFFF)
K1_WRAP = (((-9 * 0xBB67AE85) & 0xFFFFFFFF) << 32) | 0x0BADF00D
SEEDS = [0, 1, 0xFFFFFFFF, 1 << 32, (1 << 32) + 1, 0x9E3779B97F4A7C15, 1 << 63, (1 << 64) - 1, K0_WRAP, K1_WRAP]

GARBAGE_ALBEDO, GARBAGE_FUZZ, GARBAGE_IOR = (3.0e7, -4.5e5, 9.0e9), 7.5e8, -6.0e12


def soa(spheres):
    """spheres: [(center, radius, kind, albedo, fuzz, ior)] -> the rtclj_scene arrays, with the fields each kind
    ignores overwritten by garbage."""
    n = len(spheres)
    center = np.array([s[0] for s in spheres], np.float64).reshape(n, 3)
    radius = np.array([s[1] for s in spheres], np.float64)
    kind = np.array([s[2] for s in spheres], np.int32)
    albedo = np.array([s[3] for s in spheres], np.float64).reshape(n, 3)
    fuzz = np.array([s[4] for s in spheres], np.float64)
    ior = np.array([s[5] for s in spheres], np.float64)
    return garble((center, radius, kind, albedo, fuzz, ior))


def garble(scene):
    center, radius, kind, albedo, fuzz, ior = (np.array(a) for a in scene)
    albedo[kind == DIEL] = GARBAGE_ALBEDO
    fuzz[kind == LAMB] = GARBAGE_FUZZ
    ior[kind == METAL] = GARBAGE_IOR
    return tuple(np.ascontiguousarray(a) for a in (center, radius, kind, albedo, fuzz, ior))


# Seven spheres: lambertians and metals of different albedo (one with fuzz > 1: absorption), glass, a hollow
# ior < 1 bubble and a small ior 0.6 sphere, which refracts from the outside with ri = 1 / 0.6 and so reflects
# totally at grazing incidence.
MIXED = [((0.0, -100.5, -1.0), 100.0, LAMB, (0.8, 0.8, 0.0), 0.0, 1.0),
         ((0.0, 0.0, -1.2), 0.5, LAMB, (0.1, 0.2, 0.5), 0.0, 1.0),
         ((-1.0, 0.0, -1.0), 0.5, DIEL, (1.0, 1.0, 1.0), 0.0, 1.5),
         ((-1.0, 0.0, -1.0), 0.4, DIEL, (1.0, 1.0, 1.0), 0.0, 1.0 / 1.5),
         ((1.0, 0.0, -1.0), 0.5, METAL, (0.8, 0.6, 0.2), 0.3, 1.0),
         ((0.3, 0.75, -1.6), 0.3, METAL, (0.9, 0.5, 0.7), 1.7, 1.0),
         ((-0.2, -0.3, -0.5), 0.15, DIEL, (1.0, 1.0, 1.0), 0.0, 0.6)]
# Six of them, for the primary-ray kernel (<= 6 spheres)
SMALL = MIXED[:3] + MIXED[4:]


def mixed_camera(w=48, h=27, defocus=10.0):
    return CAM.main_camera(w, h, vfov=40.0, look_from=(-2.0, 1.0, 1.0), look_at=(0.0, 0.0, -1.0),
                           defocus_angle=defocus, focus_dist=3.0)


def cover_slice():
    """120 spheres of the cover scene (64 .. 512: the unpacked constant-table kernel), ground first, with glass."""
    bodies = R.scenes.cover_hittables(7)
    return garble(R.scenes.to_soa(bodies[:117] + bodies[-3:]))


def cover_camera(w=48, h=27):
    return CAM.main_camera(w, h, **R.scenes.COVER_CAMERA)


def guard_scene():
    spheres, cam, _ = guard_case()
    return soa(spheres), cam


# name -> (scene, camera, spp, depth, seed); the scenes of the liveness check and of the full matrix
def scenes():
    guard, guard_cam = guard_scene()
    return {
        "mixed": (soa(MIXED), mixed_camera(), 7, 50, 3),
        "mixed-depth2": (soa(MIXED), mixed_camera(), 6, 2, 4),
        "mixed-depth1": (soa(MIXED), mixed_camera(), 12, 1, 5),
        "mixed-depth0": (soa(MIXED), mixed_camera(), 3, 0, 6),
        "guard": (guard, guard_cam, 6, 10, GUARD_SEED),
        "cover": (cover_slice(), cover_camera(), 6, 50, 7),
        "small-depth1": (soa(SMALL), mixed_camera(), 12, 1, 8),
        "small-depth1-pinhole": (soa(SMALL), mixed_camera(defocus=0.0), 12, 1, 9),
        "small": (soa(SMALL), mixed_camera(), 6, 50, 10),
    }


SCENES = scenes()


@functools.lru_cache(maxsize=None)
def oracle(name, flags, spp=None, unit=0, seed=None):
    """The oracle's render of SCENES[name] (linear, rgb8, segments, samples); spp / seed default to the scene's."""
    scene, cam, spp0, depth, seed0 = SCENES[name]
    spp = spp or spp0
    lin, rgb, st = O.render(scene, cam, spp, depth, seed=seed0 if seed is None else seed, flags=flags, threads=8,
                            samples_per_unit=unit or spp)
    lin.flags.writeable = rgb.flags.writeable = False
    return lin, rgb, st.segments, st.samples
