"""Camera sequences on the GPU (rtclj_ctx_render_frames, rtclj_render_frames): frame f of a sequence is BIT-identical
to rtclj_ctx_render with cameras[f] and the same params -- for every kernel family, variant, summation order, shard,
grouping of frames into launches and device list -- and the call's counters are the sum of the single renders'."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as O
import raytracing_clj_b200 as R
from raytracing_clj_b200 import _abi, render

pytestmark = pytest.mark.gpu
S, CAM = R.scenes, R.camera
LIN_SENTINEL, RGB_SENTINEL = -7.25, 77


def device_count():
    n = C.c_int()
    _abi.check(_abi.lib().rtclj_device_count(C.byref(n)))
    return n.value


def orbit(make, n, look_from, look_at, **kw):
    """n cameras from make(look_from=...) on a turntable around look_at (frame 0 at look_from)."""
    return [make(look_from=CAM.turntable_look_from(k, n, look_from, look_at), look_at=look_at, **kw) for k in range(n)]


def _images(k, cam, lin=True, rgb=True):
    import torch
    shape = (k, cam.height, cam.width, 3)
    d_lin = torch.full(shape, LIN_SENTINEL, dtype=torch.float64, device="cuda:0") if lin else None
    d_rgb = torch.full(shape, RGB_SENTINEL, dtype=torch.uint8, device="cuda:0") if rgb else None
    return d_lin, d_rgb


def _host(t):
    return None if t is None else t.cpu().numpy()


def frames_ctx(ctx, cams, spp, depth, flags, *, unit=0, shard=None, seed=1, lin=True, rgb=True):
    import torch
    d_lin, d_rgb = _images(len(cams), cams[0], lin, rgb)
    stream = torch.cuda.current_stream().cuda_stream
    ctx.render_frames(cams, spp, depth, seed=seed, flags=flags, samples_per_unit=unit, shard=shard,
                      d_out_linear=d_lin.data_ptr() if lin else 0, d_out_rgb8=d_rgb.data_ptr() if rgb else 0,
                      stream=stream)
    st = ctx.stats(stream)
    return _host(d_lin), _host(d_rgb), st


def singles_ctx(ctx, cams, spp, depth, flags, *, unit=0, shard=None, seed=1, lin=True, rgb=True):
    """The frames one rtclj_ctx_render each; stats: segments / samples summed, samples_per_unit of the last."""
    import torch
    d_lin, d_rgb = _images(len(cams), cams[0], lin, rgb)
    stream = torch.cuda.current_stream().cuda_stream
    seg = samples = 0
    for f, cam in enumerate(cams):
        ctx.render(cam, spp, depth, seed=seed, flags=flags, samples_per_unit=unit, shard=shard,
                   d_out_linear=d_lin[f].data_ptr() if lin else 0, d_out_rgb8=d_rgb[f].data_ptr() if rgb else 0,
                   stream=stream)
        st = ctx.stats(stream)
        seg += st["segments"]
        samples += st["samples"]
    return _host(d_lin), _host(d_rgb), dict(segments=seg, samples=samples, samples_per_unit=st["samples_per_unit"])


def assert_frames(got, want, what):
    for f in range(max(len(x) if x is not None else 0 for x in want[:2])):
        if want[0] is not None:
            bad = np.argwhere(got[0][f].view(np.uint64) != want[0][f].view(np.uint64))
            assert bad.size == 0, f"{what}: frame {f}: {len(bad)} linear values differ, first {bad[0]}"
        if want[1] is not None:
            assert np.array_equal(got[1][f], want[1][f]), f"{what}: frame {f}: 8-bit image differs"


def check(world, cams, spp, depth, flags, what, **kw):
    ctx = render.Context(0)
    ctx.set_scene(world)
    got = frames_ctx(ctx, cams, spp, depth, flags, **kw)
    want = singles_ctx(ctx, cams, spp, depth, flags, **kw)
    ctx.close()
    assert_frames(got, want, what)
    assert got[2]["segments"] == want[2]["segments"] and got[2]["samples"] == want[2]["samples"], what
    assert got[2]["segments"] > 0 or depth <= 0, what
    assert got[2]["samples_per_unit"] == want[2]["samples_per_unit"], what
    return got


def main_cams(n=4, w=48, **kw):
    return orbit(CAM.main_camera, n, (-2.0, 2.0, 1.0), (0.0, 0.0, -1.0), width=w, **kw)


def cover_cams(n=3, w=48, h=27):
    kw = dict(S.COVER_CAMERA)
    return orbit(CAM.main_camera, n, kw.pop("look_from"), kw.pop("look_at"), width=w, height=h, **kw)


def realm_cams(n=3, w=40):
    return orbit(CAM.realm_camera, n, (-2.0, 2.0, 1.0), (0.0, 0.0, -1.0), width=w)


def i_cams(n=3, w=40):
    return [CAM.i_camera(w)] + [CAM.main_camera(w, CAM.i_camera(w).height, look_from=CAM.turntable_look_from(k, n),
                                                defocus_angle=0.0) for k in range(1, n)]


# (name, world, cameras, flags, depth, spp)
FAMILY_CASES = [
    ("library-choice", S.main_hittables(), main_cams(), O.FLAGS_MAIN, 50, 8),
    ("lane", S.main_hittables(), main_cams(), O.FLAGS_MAIN | _abi.F_LANE_KERNEL, 50, 8),       # packed (< 64 spheres)
    ("lane-cover", S.cover_hittables(7), cover_cams(), O.FLAGS_MAIN | _abi.F_LANE_KERNEL, 50, 6),  # unpacked
    ("lane2", S.cover_hittables(7), cover_cams(), O.FLAGS_MAIN | _abi.F_LANE2_KERNEL, 50, 6),
    ("lane2-small", S.main_hittables(), main_cams(), O.FLAGS_MAIN | _abi.F_LANE2_KERNEL, 50, 8),
    ("smem-table", S.main_hittables(), main_cams(), O.FLAGS_MAIN | _abi.F_SMEM_TABLE, 50, 8),
    ("smem-large", S.field_hittables(7, 14), orbit(CAM.main_camera, 3, S.FIELD_CAMERA["look_from"],
                                                  S.FIELD_CAMERA["look_at"], width=40, vfov=30.0), O.FLAGS_MAIN, 50, 4),
    ("no-cull", S.main_hittables(), main_cams(), O.FLAGS_MAIN | _abi.F_NO_CULL, 50, 8),
    ("primary-i", S.i_hittables(), i_cams(), O.FLAGS_I, 50, 16),
    ("primary-depth1", S.main_hittables(), main_cams(), O.FLAGS_MAIN, 1, 16),
    ("lane-depth1", S.main_hittables(), main_cams(), O.FLAGS_MAIN | _abi.F_LANE_KERNEL, 1, 16),
    ("depth0", S.main_hittables(), main_cams(), O.FLAGS_MAIN, 0, 4),
    ("realm", S.realm_hittables(), realm_cams(), O.FLAGS_REALM, 50, 8),
    ("realm-lane2", S.realm_hittables(), realm_cams(), O.FLAGS_REALM | _abi.F_LANE2_KERNEL, 50, 8),
    ("i-lane", S.i_hittables(), i_cams(), O.FLAGS_I | _abi.F_LANE_KERNEL, 50, 16),
    ("i-smem", S.i_hittables(), i_cams(), O.FLAGS_I | _abi.F_SMEM_TABLE, 50, 16),
]


@pytest.mark.parametrize("name,world,cams,flags,depth,spp", FAMILY_CASES, ids=[c[0] for c in FAMILY_CASES])
def test_every_kernel_family(name, world, cams, flags, depth, spp):
    if name == "smem-large":
        assert len(world) > 512
    got = check(world, cams, spp, depth, flags, name)
    if depth <= 0:
        assert not got[0].any() and not got[1].any()


def test_defocus_differs_between_frames():
    """One sequence mixes frames with and without the defocus disk, on the path kernels and the primary kernel."""
    cams = [CAM.main_camera(48, look_from=CAM.turntable_look_from(k, 4), defocus_angle=[10.0, 0.0, 3.0, -1.0][k])
            for k in range(4)]
    for flags, depth in ((O.FLAGS_MAIN, 50), (O.FLAGS_MAIN | _abi.F_LANE2_KERNEL, 50), (O.FLAGS_MAIN, 1)):
        check(S.main_hittables(), cams, 8, depth, flags, f"mixed defocus {flags:#x} depth {depth}")
    no_disk = [c for c in cams if c.defocus_angle <= 0.0]
    check(S.main_hittables(), no_disk, 8, 1, O.FLAGS_MAIN, "primary without the disk")


@pytest.mark.parametrize("unit,spp,depth,flags", [
    (0, 40, 50, O.FLAGS_MAIN),          # the library's chunks
    (3, 10, 50, O.FLAGS_MAIN),          # explicit samples_per_unit
    (64, 64, 50, O.FLAGS_MAIN),         # strict, through sample_buf
    (70, 70, 50, O.FLAGS_REALM),        # strict, through sample_buf, realm's forward product
    (0, 24, 1, O.FLAGS_MAIN),           # strict on the primary kernel (the library's default there)
    (24, 24, 50, O.FLAGS_I),            # strict -i
], ids=["chunked", "explicit-unit", "strict-sample-buf", "strict-realm", "strict-primary", "strict-i"])
def test_order_modes(unit, spp, depth, flags):
    cams = realm_cams(3, 40) if flags == O.FLAGS_REALM else main_cams(3, 40)
    world = S.realm_hittables() if flags == O.FLAGS_REALM else S.main_hittables()
    check(world, cams, spp, depth, flags, f"unit {unit}", unit=unit)


@pytest.mark.parametrize("flags,depth,unit,spp", [(O.FLAGS_MAIN, 50, 0, 8), (O.FLAGS_MAIN | _abi.F_LANE2_KERNEL, 50, 0, 8),
                                                  (O.FLAGS_MAIN, 50, 64, 64), (O.FLAGS_MAIN, 1, 0, 8)],
                         ids=["lane", "lane2", "strict", "primary"])
def test_shards_write_only_their_rows(flags, depth, unit, spp):
    cams = main_cams(3, 40)
    H = cams[0].height
    for index in range(3):
        got = check(S.main_hittables(), cams, spp, depth, flags, f"shard {index}", unit=unit, shard=(index, 3, 2))
        mine = set(render.shard_rows(H, index, 3, 2))
        for f in range(3):
            for j in range(H):
                if j in mine:
                    assert not (got[0][f, j] == LIN_SENTINEL).all(), (f, j)
                else:
                    assert (got[0][f, j] == LIN_SENTINEL).all() and (got[1][f, j] == RGB_SENTINEL).all(), (f, j)


def test_grouping_chunked_1080p():
    """1920x1080 x 152 spp in chunks: 19 chunks make 945 MB of unit sums per frame, so three frames take two launches."""
    cams = [CAM.main_camera(1920, look_from=CAM.turntable_look_from(k, 3)) for k in range(3)]
    assert render.pass_unit(1920, 1080, 152, 50) == 8
    check(S.main_hittables(), cams, 152, 50, O.FLAGS_MAIN, "1080p chunked")


def test_grouping_strict_1080p():
    """1920x1080 strict at 64 spp: 4.2 GB of sample colours per frame, more than a launch holds: groups of one,
    each under rtclj_ctx_render's own rules."""
    cams = [CAM.main_camera(1920, look_from=CAM.turntable_look_from(k, 2)) for k in range(2)]
    check(S.main_hittables(), cams, 64, 50, O.FLAGS_MAIN, "1080p strict", unit=64)


def test_more_frames_than_a_launch_takes():
    """130 frames: more cameras than the kernel parameters of one launch hold (128)."""
    cams = main_cams(130, 16)
    check(S.main_hittables(), cams, 4, 50, O.FLAGS_MAIN, "130 frames")
    check(S.main_hittables(), cams, 4, 1, O.FLAGS_MAIN, "130 frames, primary")


def test_degenerate_sequences():
    world, cam = S.main_hittables(), CAM.main_camera(48)
    check(world, [cam], 8, 50, O.FLAGS_MAIN, "one frame")
    got = check(world, [cam, cam, cam], 8, 50, O.FLAGS_MAIN, "one camera repeated")
    assert all(np.array_equal(got[0][0].view(np.uint64), got[0][f].view(np.uint64)) for f in (1, 2))
    ctx = render.Context(0)
    ctx.set_scene(world)
    cams = main_cams(3)
    full = frames_ctx(ctx, cams, 8, 50, O.FLAGS_MAIN)
    for lin, rgb in ((False, False), (True, False), (False, True)):
        part = frames_ctx(ctx, cams, 8, 50, O.FLAGS_MAIN, lin=lin, rgb=rgb)
        assert part[2]["segments"] == full[2]["segments"] and part[2]["samples"] == full[2]["samples"]
        assert_frames(part, (full[0] if lin else None, full[1] if rgb else None), f"outputs {lin} {rgb}")
    ctx.close()


def test_against_the_oracle():
    cams = main_cams(3, 64)
    soa = S.to_soa(S.main_hittables())
    lin, rgb, st = render.render_frames(S.main_hittables(), cams, 8, 50, seed=3, flags=O.FLAGS_MAIN, samples_per_unit=8)
    segments = 0
    for f, cam in enumerate(cams):
        lin_o, rgb_o, st_o = O.render(soa, cam, 8, 50, seed=3, flags=O.FLAGS_MAIN, threads=4)
        assert np.array_equal(lin[f].view(np.uint64), lin_o.view(np.uint64)) and np.array_equal(rgb[f], rgb_o), f
        segments += st_o.segments
    assert st["segments"] == segments


@pytest.mark.parametrize("pinned", [False, True], ids=["pageable", "pinned"])
@pytest.mark.parametrize("devs", ["one", "all"])
def test_host_path(devs, pinned):
    devices = [0] if devs == "one" else list(range(device_count()))
    if devs == "all" and len(devices) < 2:
        pytest.skip("one GPU")
    world, cams = S.cover_hittables(7), cover_cams(5, 64, 36)
    ctx = render.Context(0)
    ctx.set_scene(world)
    want = frames_ctx(ctx, cams, 6, 50, O.FLAGS_MAIN, unit=2)
    ctx.close()
    lib, n = _abi.lib(), len(cams)
    shape = (n, cams[0].height, cams[0].width, 3)
    nbytes = int(np.prod(shape))
    if pinned:
        p_lin, p_rgb = C.c_void_p(), C.c_void_p()
        _abi.check(lib.rtclj_host_alloc(nbytes * 8, C.byref(p_lin)))
        _abi.check(lib.rtclj_host_alloc(nbytes, C.byref(p_rgb)))
        lin = np.ctypeslib.as_array((C.c_double * nbytes).from_address(p_lin.value)).reshape(shape)
        rgb = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(p_rgb.value)).reshape(shape)
    else:
        lin, rgb = np.zeros(shape), np.zeros(shape, dtype=np.uint8)
    try:
        sc = render._scene_struct(S.to_soa(world))
        arr = (_abi.Camera * n)(*[render._camera_struct(c) for c in cams])
        prm = _abi.Params(6, 50, 1, O.FLAGS_MAIN, 2, 0, 0, 0, 0, 0)
        darr = (C.c_int32 * len(devices))(*devices)
        st = _abi.Stats()
        _abi.check(lib.rtclj_render_frames(C.byref(sc), arr, n, C.byref(prm), darr, len(devices), lin.ctypes.data,
                                           rgb.ctypes.data, C.byref(st)))
        assert_frames((lin, rgb), want, f"host path on {devices}, pinned {pinned}")
        assert st.segments == want[2]["segments"] and st.n_devices == len(devices)
    finally:
        if pinned:
            lib.rtclj_host_free(p_lin)
            lib.rtclj_host_free(p_rgb)
