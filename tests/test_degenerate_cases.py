"""CPU side of tests/test_gpu_degenerate_rays.py: each of its cases reaches, in the oracle's own arithmetic
(tests/oracle_probe.py), the path it is for -- degenerate directions, NaN roots, the near-zero guard -- and the probe
itself counts what it should.  No GPU needed."""
import numpy as np
import pytest

import oracle_lib as O
import oracle_probe as OP
import test_gpu_degenerate_rays as T


def test_probe_sees_every_scan_and_nothing_degenerate_on_an_ordinary_render():
    scene = T.world(T.BASE + [T.GROUND], 64)
    p = OP.scans(scene, T.view(1.0), 4, 10, 3, O.FLAGS_MAIN)
    _, _, st = O.render(scene, T.view(1.0), 4, 10, seed=3, flags=O.FLAGS_MAIN)
    assert p["scans"] == p["segments"] == st.segments > st.samples
    assert p["degenerate"] == 0 and p["nan_roots"] == 0


@pytest.mark.parametrize("case", list(T.CAMERA_CASES))
def test_camera_cases(case):
    spheres, cam = T.CAMERA_CASES[case]
    for variant, (flags, depth) in T.VARIANTS.items():
        for pad in T.PADS:
            T.assert_reaches(T.world(spheres, pad), cam, 4, depth, 11, flags, cam.width * cam.height * 4,
                             case in T.NAN_ROOTS)


@pytest.mark.parametrize("case,variant", T.SCATTER_PARAMS, ids=[f"{c}-{v}" for c, v in T.SCATTER_PARAMS])
def test_scatter_cases(case, variant):
    spheres, cam, depth, _, nan_roots = T.SCATTER_CASES[case]
    for pad in T.PADS:
        p = T.assert_reaches(T.world(spheres, pad), cam, 4, depth, 21 + T.PADS.index(pad), T.VARIANTS[variant][0], 1,
                             nan_roots)
        assert p["degenerate"] < p["scans"], p  # and the primary rays are ordinary: both kinds in one render


def test_guard_case():
    _, _, s = T.guard_case()
    assert np.all(np.abs(s) < 1e-8) and np.any(s != 0.0), s
    spheres, cam, _ = T.guard_case()
    for pad in T.PADS:
        scene = T.world(spheres, pad)
        realm = OP.scans(scene, cam, 4, 10, T.GUARD_SEED, O.FLAGS_REALM)
        main = OP.scans(scene, cam, 4, 10, T.GUARD_SEED, O.FLAGS_MAIN)
        assert realm["degenerate"] >= 1 and main["degenerate"] == 0, (realm, main)
