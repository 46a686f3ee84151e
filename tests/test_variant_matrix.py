"""The variant-switch matrix on the CPU: every switch is live in the matrix's scenes (a matrix over a switch that
changes nothing proves nothing), the covering array covers every pair, the wrap seeds wrap, and the Python layer
refuses a seed the 64-bit key cannot hold instead of truncating it."""
import itertools

import numpy as np
import pytest

import oracle_lib as O
import raytracing_clj_b200 as R
import variant_matrix as V
from raytracing_clj_b200 import _abi, render


def test_covering_array_covers_every_pair_of_switches():
    assert len(V.COVERING) == 8 and len(set(V.COVERING)) == 8
    for (_, a), (_, b) in itertools.combinations(V.BITS.items(), 2):
        pairs = {(bool(f & a), bool(f & b)) for f in V.COVERING}
        assert pairs == {(False, False), (False, True), (True, False), (True, True)}, (a, b)
    assert all(0 <= f < 64 for f in V.PAIRWISE)


def test_every_switch_changes_the_image():
    """For every switch b, some scene of the matrix and some combination f give oracle(f) != oracle(f ^ b): in the bits
    of the linear image, or for QUANT_LINEAR, which changes only the quantisation, in the 8-bit image."""
    live = {name: set() for name in V.BITS}
    for scene in ("mixed", "mixed-depth2", "guard", "small-depth1"):
        for f in V.ALL_COMBOS:
            lin, rgb = V.oracle(scene, f)[:2]
            for name, bit in V.BITS.items():
                if f & bit:
                    continue
                lin_b, rgb_b = V.oracle(scene, f | bit)[:2]
                if (lin.view(np.uint64) != lin_b.view(np.uint64)).any() or (rgb != rgb_b).any():
                    live[name].add((scene, f))
    dead = [name for name, where in live.items() if not where]
    assert not dead, f"switches that change no image of the matrix: {dead}"
    # the guard fires only in its engineered scene; the others in the path-traced scene itself
    assert {s for s, _ in live["NEAR_ZERO_GUARD"]} == {"guard"}
    for name in ("SCHLICK", "REVERSE_PRODUCT", "MEAN_DIVIDE", "NORMAL_SHADING", "QUANT_LINEAR"):
        assert any(s == "mixed" for s, _ in live[name]), name
    # QUANT_LINEAR changes the 8-bit image only
    lin0, rgb0 = V.oracle("mixed", 0)[:2]
    lin1, rgb1 = V.oracle("mixed", O.F_QUANT_LINEAR)[:2]
    assert np.array_equal(lin0.view(np.uint64), lin1.view(np.uint64)) and not np.array_equal(rgb0, rgb1)


def test_depth_zero_is_black_under_every_combination():
    for f in V.ALL_COMBOS:
        lin, rgb, segments, samples = V.oracle("mixed-depth0", f)
        assert not lin.any() and not rgb.any() and segments == 0, f


def test_the_wrap_seeds_wrap():
    k0, k1 = V.K0_WRAP & 0xFFFFFFFF, V.K0_WRAP >> 32
    assert (k0 + 9 * 0x9E3779B9) % (1 << 32) == 0 and k1 != 0
    k0, k1 = V.K1_WRAP & 0xFFFFFFFF, V.K1_WRAP >> 32
    assert (k1 + 9 * 0xBB67AE85) % (1 << 32) == 0 and k0 != 0
    assert len(set(V.SEEDS)) == len(V.SEEDS) and all(0 <= s < 1 << 64 for s in V.SEEDS)


@pytest.mark.parametrize("seed", [-1, 1 << 64, (1 << 64) + 5, 1.0, 2.5, "3", None])
def test_a_seed_outside_the_key_is_refused(seed):
    """ctypes keeps the low 64 bits of an integer: 2^64 + 5 would render as seed 5, and -1 as 2^64 - 1."""
    with pytest.raises(ValueError, match="seed"):
        render._params(4, 5, seed, O.FLAGS_MAIN, 0)
    world, cam = R.scenes.main_hittables(), R.camera.main_camera(8)
    with pytest.raises(ValueError, match="seed"):
        render.render(world, cam, 1, 5, seed=seed)
    with pytest.raises(ValueError, match="seed"):
        render.render_frames(world, [cam], 1, 5, seed=seed)
    with pytest.raises(ValueError, match="seed"):
        render.render_ppm(world, cam, 1, 5, seed=seed)
    with pytest.raises(ValueError, match="seed"):
        render.render_png(world, cam, 1, 5, seed=seed)
    with pytest.raises(ValueError, match="seed"):
        render.Progressive(world, cam, 1, 5, seed=seed)


@pytest.mark.parametrize("seed", [0, 1, (1 << 64) - 1, np.uint64((1 << 64) - 1), np.int64(7), True])
def test_every_seed_of_the_key_is_kept(seed):
    prm = render._params(4, 5, seed, O.FLAGS_MAIN, 0, device=3)
    assert prm.seed == int(seed) and prm.device == 3 and (prm.spp, prm.max_depth, prm.flags) == (4, 5, O.FLAGS_MAIN)
    # the ctypes field itself truncates: the reason for the check
    assert _abi.Params(1, 1, (1 << 64) + 5, 0, 0, 0, 0, 0, 0, 0).seed == 5
