"""The two-level cull of render_lane2_kernel (DESIGN.md 4.2, "group bound") keeps exactly the survivors of the flat
cull: on random scenes of 64 ... 512 spheres it renders the same image as render_kernel<true>, which culls every
sphere against every ray, with the same number of prefilter tests (one per cull survivor).  Run with `pytest -m gpu`."""
import numpy as np
import pytest

import raytracing_clj_b200 as R
from raytracing_clj_b200 import _abi, render

pytestmark = pytest.mark.gpu
S, CAM = R.scenes, R.camera


def random_scene(rng, n):
    """A field of small spheres in a slab (the cover scene's shape) at a random scale and offset, a few huge
    ground-like spheres, coincident centres and negative radii."""
    sp, mat = R.hittable.sphere, R.material
    scale = 10.0 ** rng.uniform(-2, 6)
    offset = rng.normal(size=3) * scale * (1e3 if rng.random() < 0.3 else 1.0)
    world = []
    for i in range(n):
        if i < int(rng.integers(0, 4)):
            c, r = offset + np.array([0.0, -1e3 * scale, 0.0]) * rng.uniform(0.5, 1.5), 1e3 * scale
        elif world and rng.random() < 0.05:
            c, r = np.array(world[-1]["hittable/center"]), scale * rng.uniform(0.05, 0.3)
        else:
            c = offset + np.array([rng.uniform(-11, 11), rng.uniform(0.0, 0.4), rng.uniform(-11, 11)]) * scale
            r = scale * 10.0 ** rng.uniform(-1.5, -0.3) * (-1 if rng.random() < 0.03 else 1)
        kind = rng.integers(0, 3)
        m = (mat.lambertian(tuple(rng.random(3))) if kind == 0 else
             mat.metal(tuple(rng.random(3)), float(rng.random() * 0.5)) if kind == 1 else
             mat.dielectric(1.5))
        world.append(S.body(sp(tuple(float(x) for x in c), float(r)), m))
    where = rng.integers(0, 3)
    look_from = offset + scale * (np.array([13.0, 2.0, 3.0]) if where == 0 else            # the cover camera
                                  np.array([rng.uniform(-11, 11), 0.2, rng.uniform(-11, 11)]) if where == 1 else  # in the slab
                                  rng.normal(size=3) * 10.0 ** rng.uniform(1, 3))          # far away
    look_at = offset + scale * np.array([rng.uniform(-3, 3), 0.0, rng.uniform(-3, 3)])
    cam = CAM.main_camera(64, 36, vfov=float(rng.uniform(10, 90)), look_from=tuple(float(x) for x in look_from),
                          look_at=tuple(float(x) for x in look_at), defocus_angle=0.0,
                          focus_dist=float(np.linalg.norm(look_from - look_at)))
    return world, cam


@pytest.mark.parametrize("n", [64, 100, 257, 484, 512])
def test_two_level_cull_keeps_the_flat_cull_survivors(n):
    rng = np.random.default_rng(1000 + n)
    for case in range(6):
        world, cam = random_scene(rng, n)
        for flags in (_abi.FLAGS_MAIN, _abi.FLAGS_REALM):
            a, ra, sa = render.render(world, cam, 4, 12, seed=case, flags=flags | _abi.F_LANE2_KERNEL, samples_per_unit=4)
            b, rb, sb = render.render(world, cam, 4, 12, seed=case, flags=flags | _abi.F_LANE_KERNEL, samples_per_unit=4)
            assert np.array_equal(a, b, equal_nan=True) and np.array_equal(ra, rb), (n, case)
            assert sa["segments"] == sb["segments"] and sa["prefilter_tests"] == sb["prefilter_tests"], (n, case, sa, sb)


def test_cover_scene_frame_keeps_the_flat_cull_survivors():
    world = S.cover_hittables(7)
    cam = CAM.main_camera(320, 180, **S.COVER_CAMERA)
    a, ra, sa = render.render(world, cam, 16, 50, seed=1, flags=_abi.FLAGS_MAIN | _abi.F_LANE2_KERNEL)
    b, rb, sb = render.render(world, cam, 16, 50, seed=1, flags=_abi.FLAGS_MAIN | _abi.F_LANE_KERNEL)
    assert np.array_equal(a, b) and np.array_equal(ra, rb)
    assert sa["segments"] == sb["segments"] and sa["prefilter_tests"] == sb["prefilter_tests"], (sa, sb)
