"""The deterministic-RNG shim for the JVM reference (integration/clojure/src/rtclj/rng_shim.clj,
SURVEY.md section 8 row f-3) cannot run here (no JVM).  Its hand-out order is checked through a Python
model of the same state machine: a restatement of the reference's `main` loop that draws ONLY through
sequential `rand()` calls -- as the reference does -- must reproduce the oracle's counter-based render
bit for bit."""
import numpy as np

import oracle_lib as O
import raytracing_clj_b200 as R
import rng_shim_model as M

S, CAM = R.scenes, R.camera


def test_philox_model_equals_oracle_philox():
    rng = np.random.default_rng(0)
    for _ in range(200):
        c = [int(x) for x in rng.integers(0, 2**32, 4)]
        k = [int(x) for x in rng.integers(0, 2**32, 2)]
        assert list(M.philox4x32_10(*c, *k)) == [int(x) for x in O.philox(c, k)]


# Random123's published known-answer vectors for philox4x32-10 (kat_vectors): counter, key -> output
PHILOX_KAT = [
    ((0x00000000, 0x00000000, 0x00000000, 0x00000000), (0x00000000, 0x00000000),
     (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff), (0xffffffff, 0xffffffff),
     (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
]


def test_philox_known_answers():
    """Both implementations against the published vectors, not only against each other."""
    for ctr, key, out in PHILOX_KAT:
        assert O.philox(ctr, key) == out
        assert tuple(M.philox4x32_10(*ctr, *key)) == out


def test_camera_stage_is_sequential_words():
    st = M.ShimStream(seed=0x1234567890ABCDEF)
    st.begin_sample(77, 5)
    got = [st.rand() for _ in range(12)]
    want = [O.lib().rto_uniform(0x1234567890ABCDEF, 77, 5, 0, n // 4, n % 4) for n in range(12)]
    assert got == want


def test_unit_vector_fields_and_schlick_word():
    seed = 99
    st = M.ShimStream(seed)
    st.begin_sample(3, 1)
    st.set_stage(4)
    assert st.rand() == O.lib().rto_uniform(seed, 3, 1, 4, 0, 0)          # Schlick: word 0 of block 0
    got = st.unit_vector_scope(lambda: [st.rand() for _ in range(15)])()   # five candidates
    want = []
    for cand in range(5):
        w = [int(x) for x in O.philox([3, 1, 4, cand // 2], [seed, 0])]
        bits = w[2 * (cand % 2)] | (w[2 * (cand % 2) + 1] << 32)
        want += [((bits >> (21 * c)) & 0x1FFFFF) / 2097152.0 for c in range(3)]
    assert got == want


def _compare(world, cam, spp, depth, seed, realm=False):
    soa = S.to_soa(world)
    lin_o, _, st_o = O.render(soa, cam, spp, depth, seed=seed, flags=O.FLAGS_REALM if realm else O.FLAGS_MAIN, threads=2)
    lin_m, segs, _ = M.render_main(soa, cam, spp, depth, seed=seed, realm=realm)
    assert segs == st_o.segments
    assert np.array_equal(np.array(lin_m, dtype=np.float64), lin_o)


def test_sequential_reference_loop_reproduces_the_oracle_render():
    # the reference's own scene and camera (defocus disk, Schlick glass, fuzzy metal), tiny image
    _compare(S.main_hittables(), CAM.main_camera(16), 3, 50, seed=1)
    # a slice of the cover scene: many small spheres, all three materials
    _compare(S.cover_hittables(7)[:40], CAM.main_camera(12, 7, **S.COVER_CAMERA), 2, 50, seed=5)
    # depth cap reached inside glass
    _compare(S.main_hittables(), CAM.main_camera(10), 2, 3, seed=2)
    # seeds with the high word of the key set: both words of the key reach every draw
    _compare(S.main_hittables(), CAM.main_camera(10), 2, 50, seed=(1 << 64) - 1)
    _compare(S.main_hittables(), CAM.main_camera(10), 2, 50, seed=0xFFFFFFFF00000000)


def test_sequential_realm_loop_reproduces_the_oracle_render():
    # realm semantics: forward product, no Schlick draw, no near-zero guard, no defocus, x (1/spp)
    _compare(S.realm_hittables(), CAM.realm_camera(16), 3, 50, seed=1, realm=True)
    _compare(S.cover_hittables(3)[:30], CAM.realm_camera(12), 2, 6, seed=4, realm=True)
