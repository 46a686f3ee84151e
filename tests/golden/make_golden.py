"""Regenerates tests/golden/*.npz from a checkout of keychera/raytracing-clj (for its two
committed renders) and the CPU oracle:

    python tests/golden/make_golden.py path/to/raytracing-clj

1. reference_images.npz -- the reference's two committed renders, the only result
   pins it offers (SURVEY.md 4): scene.ppm (`-M:main`, 400x225) and scene-realm.ppm
   (`-M:realm`, 400x224), decoded from P3 text to uint8 arrays.  These are OUTPUT
   artefacts of the reference, not source.
2. oracle_fixtures.npz -- small renders by the CPU oracle (oracle/rt_oracle.c) on the
   shared Philox stream, one per variant / scene, so that the GPU parity tests also
   compare against COMMITTED vectors and an accidental change of the oracle shows.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def load_p3(path):
    toks = open(path).read().split()
    assert toks[0] == "P3" and toks[3] == "255"
    w, h = int(toks[1]), int(toks[2])
    return np.array(toks[4:], dtype=np.uint8).reshape(h, w, 3)


def fixture_cases():
    """name -> (bodies, camera, spp, depth, seed, flags, samples_per_unit)"""
    import oracle_lib as O
    import raytracing_clj_b200 as R

    cam, sc = R.camera, R.scenes
    cover = sc.cover_hittables(7)
    return {
        "main_64x36": (sc.main_hittables(), cam.main_camera(64), 16, 50, 1, O.FLAGS_MAIN, 0),
        "realm_64x35": (sc.realm_hittables(), cam.realm_camera(64), 16, 50, 1, O.FLAGS_REALM, 0),
        "i_64x35": (sc.i_hittables(), cam.i_camera(64), 16, 50, 1, O.FLAGS_I, 0),
        "realm_depth1_sky_64x35": (sc.realm_hittables(), cam.i_camera(64), 16, 1, 3, O.FLAGS_REALM, 0),
        "main_chunked_48x27": (sc.main_hittables(), cam.main_camera(48), 24, 50, 5, O.FLAGS_MAIN, 5),
        "cover_48x27": (cover, cam.main_camera(48, 27, **sc.COVER_CAMERA), 8, 50, 11, O.FLAGS_MAIN, 0),
    }


def main(ref):
    np.savez_compressed(os.path.join(HERE, "reference_images.npz"),
                        scene_main=load_p3(os.path.join(ref, "scene.ppm")),
                        scene_realm=load_p3(os.path.join(ref, "scene-realm.ppm")))
    import oracle_lib as O
    import raytracing_clj_b200 as R

    out = {}
    for name, (bodies, camera, spp, depth, seed, flags, unit) in fixture_cases().items():
        lin, rgb, st = O.render(R.scenes.to_soa(bodies), camera, spp, depth, seed=seed, flags=flags,
                                threads=4, samples_per_unit=unit)
        out[name + "/linear"] = lin
        out[name + "/rgb8"] = rgb
        out[name + "/segments"] = np.array([st.segments], dtype=np.uint64)
    np.savez_compressed(os.path.join(HERE, "oracle_fixtures.npz"), **out)
    print("wrote", sorted(os.listdir(HERE)))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
