"""The render loop, host side: body maps + camera -> the C ABI -> CUDA -> images.

Stands in for the loops inside the reference's `-main`s (src/raytracing.clj:141-171,
src/realm/raytracing.clj:325-346, src/experimental/raytracing_i.clj:146-163) and for
their PPM writers (raytracing.clj:172-175, realm/raytracing.clj:350-358).
Everything here calls librtclj_b200.so; nothing is computed in Python."""
from __future__ import annotations

import ctypes as C
import math
import operator
from typing import Iterable, List, Optional, Sequence

import numpy as np

from . import _abi, scenes
from .camera import Camera


def shard_rows(height: int, index: int, count: int, rows: int) -> List[int]:
    """The image rows shard `index` of `count` owns: rows are cut into tiles of `rows` rows and
    tile t belongs to shard t % count (rtclj_params.shard_*; DESIGN.md section 6)."""
    if count <= 1:
        return list(range(height))
    out: List[int] = []
    ntiles = (height + rows - 1) // rows
    for t in range(index, ntiles, count):
        out.extend(range(t * rows, min(height, (t + 1) * rows)))
    return out


def shard_plan(height: int, row_bytes: int, index: int, count: int, rows: int, max_piece_bytes: int = 0):
    """The copies the LIBRARY issues to download one shard (rtclj_shard_plan): a list of
    (byte offset, pitch, width, height) -- `height` runs of `width` bytes, `pitch` apart."""
    lib = _abi.lib()
    n = C.c_size_t()
    _abi.check(lib.rtclj_shard_plan(height, row_bytes, index, count, rows, max_piece_bytes, None, 0, C.byref(n)))
    buf = (C.c_uint64 * (4 * max(1, n.value)))()
    _abi.check(lib.rtclj_shard_plan(height, row_bytes, index, count, rows, max_piece_bytes, buf, n.value, C.byref(n)))
    return [tuple(int(buf[4 * i + k]) for k in range(4)) for i in range(n.value)]


def _scene_struct(soa):
    center, radius, kind, albedo, fuzz, ior = soa
    s = _abi.Scene(len(radius), 0, center.ctypes.data, radius.ctypes.data, kind.ctypes.data,
                   albedo.ctypes.data, fuzz.ctypes.data, ior.ctypes.data)
    s._keep = soa
    return s


def _camera_struct(cam) -> _abi.Camera:
    if isinstance(cam, _abi.Camera):
        return cam
    c = _abi.Camera()
    for name in ("pixel00", "pixel_du", "pixel_dv", "center", "defocus_u", "defocus_v"):
        getattr(c, name)[:] = [float(x) for x in getattr(cam, name)]
    c.defocus_angle = float(cam.defocus_angle)
    c.width, c.height = int(cam.width), int(cam.height)
    return c


def _params(samples_per_px, max_depth, seed, flags, samples_per_unit, device=0) -> _abi.Params:
    """The rtclj_params of a call.  The seed is the 64-bit Philox key (low word k0, high word k1): a seed outside
    [0, 2^64) is refused rather than wrapped, since ctypes would silently keep its low 64 bits only."""
    try:
        s = operator.index(seed)
    except TypeError:
        raise ValueError(f"seed must be an integer in [0, 2^64), got {seed!r}") from None
    if not 0 <= s < 1 << 64:
        raise ValueError(f"seed must be an integer in [0, 2^64), got {s}")
    return _abi.Params(int(samples_per_px), int(max_depth), s, int(flags), int(samples_per_unit), 0, 0, 0, int(device), 0)


def _as_soa(world):
    if isinstance(world, tuple) and len(world) == 6 and isinstance(world[0], np.ndarray):
        return world
    return scenes.to_soa(list(world))


def render(world, cam: Camera, samples_per_px: int = 100, max_depth: int = 50, *, seed: int = 1,
           flags: int = _abi.FLAGS_MAIN, samples_per_unit: int = 0, devices: Optional[Sequence[int]] = None,
           shard: Optional[tuple] = None, want_linear: bool = True, want_rgb8: bool = True,
           out_linear: Optional[np.ndarray] = None, out_rgb8: Optional[np.ndarray] = None):
    """Render `world` (a hittable list: body maps, or the SoA tuple) through the C ABI with
    HOST buffers.  Returns (linear float64 [H,W,3] | None, rgb8 uint8 [H,W,3] | None, stats dict).
    devices: GPUs to interleave rows over (default [0]); shard=(index, count, rows): render only
    that shard's rows (one-process-per-GPU hosts)."""
    lib = _abi.lib()
    soa = _as_soa(world)
    sc, cm = _scene_struct(soa), _camera_struct(cam)
    H, W = cm.height, cm.width
    if want_linear and out_linear is None:
        out_linear = np.zeros((H, W, 3), dtype=np.float64)
    if want_rgb8 and out_rgb8 is None:
        out_rgb8 = np.zeros((H, W, 3), dtype=np.uint8)
    prm = _params(samples_per_px, max_depth, seed, flags, samples_per_unit)
    st = _abi.Stats()
    lin_p = out_linear.ctypes.data if out_linear is not None else None
    rgb_p = out_rgb8.ctypes.data if out_rgb8 is not None else None
    if shard is not None:
        prm.shard_index, prm.shard_count, prm.shard_rows = (int(x) for x in shard)
        prm.device = int(devices[0]) if devices else 0
        _abi.check(lib.rtclj_render(C.byref(sc), C.byref(cm), C.byref(prm), lin_p, rgb_p, C.byref(st)))
    else:
        devs = list(devices) if devices else [0]
        arr = (C.c_int32 * len(devs))(*devs)
        _abi.check(lib.rtclj_render_multi(C.byref(sc), C.byref(cm), C.byref(prm), arr, len(devs),
                                          lin_p, rgb_p, C.byref(st)))
    return out_linear, out_rgb8, st.as_dict()


def _camera_array(cameras):
    cams = [_camera_struct(c) for c in cameras]
    arr = (_abi.Camera * max(1, len(cams)))(*cams)
    return arr, len(cams)


def render_frames(world, cameras: Sequence, samples_per_px: int = 100, max_depth: int = 50, *, seed: int = 1,
                  flags: int = _abi.FLAGS_MAIN, samples_per_unit: int = 0, devices: Optional[Sequence[int]] = None,
                  want_linear: bool = True, want_rgb8: bool = True):
    """A camera sequence of one scene (rtclj_render_frames): every frame in shared launches, rows interleaved over
    `devices` (default [0]).  Returns (linear float64 [K,H,W,3] | None, rgb8 uint8 [K,H,W,3] | None, stats dict);
    frame f is bit-identical to `render(world, cameras[f], ...)` with the same arguments, and the stats cover the
    whole sequence."""
    lib = _abi.lib()
    soa = _as_soa(world)
    sc = _scene_struct(soa)
    arr, n = _camera_array(cameras)
    H, W = (arr[0].height, arr[0].width) if n else (0, 0)
    out_linear = np.zeros((n, H, W, 3), dtype=np.float64) if want_linear else None
    out_rgb8 = np.zeros((n, H, W, 3), dtype=np.uint8) if want_rgb8 else None
    prm = _params(samples_per_px, max_depth, seed, flags, samples_per_unit)
    devs = list(devices) if devices else [0]
    darr = (C.c_int32 * len(devs))(*devs)
    st = _abi.Stats()
    _abi.check(lib.rtclj_render_frames(C.byref(sc), arr, n, C.byref(prm), darr, len(devs),
                                       out_linear.ctypes.data if out_linear is not None else None,
                                       out_rgb8.ctypes.data if out_rgb8 is not None else None, C.byref(st)))
    return out_linear, out_rgb8, st.as_dict()


def render_ppm(world, cam: Camera, samples_per_px: int = 100, max_depth: int = 50, *, seed: int = 1,
               flags: int = _abi.FLAGS_MAIN, samples_per_unit: int = 0, devices: Optional[Sequence[int]] = None):
    """The render loop and the write-color! loop in one call (raytracing.clj:141-175): returns
    (text of the P3 file as bytes, stats).  The image never visits the host: the shards are assembled on
    devices[0] and the device P3 writer runs there (rtclj_render_multi_ppm)."""
    lib = _abi.lib()
    soa = _as_soa(world)
    sc, cm = _scene_struct(soa), _camera_struct(cam)
    prm = _params(samples_per_px, max_depth, seed, flags, samples_per_unit)
    devs = list(devices) if devices else [0]
    arr = (C.c_int32 * len(devs))(*devs)
    n = C.c_size_t()
    _abi.check(lib.rtclj_render_multi_ppm(C.byref(sc), C.byref(cm), C.byref(prm), arr, len(devs), None, 0, C.byref(n), None))
    store = bytearray(n.value)
    buf = (C.c_char * n.value).from_buffer(store)
    st = _abi.Stats()
    _abi.check(lib.rtclj_render_multi_ppm(C.byref(sc), C.byref(cm), C.byref(prm), arr, len(devs), buf, n.value,
                                          C.byref(n), C.byref(st)))
    del buf
    return bytes(memoryview(store)[: n.value]), st.as_dict()


def render_png(world, cam: Camera, samples_per_px: int = 100, max_depth: int = 50, *, seed: int = 1,
               flags: int = _abi.FLAGS_MAIN, samples_per_unit: int = 0, devices: Optional[Sequence[int]] = None):
    """The render loop and ppm->png in one call: returns (bytes of a compressed PNG, stats).  The image never visits
    the host: the shards are assembled on devices[0] and the device PNG writer runs there (rtclj_render_multi_png);
    the bytes are those of encode_png(rgb8, device=k) on the rendered image."""
    lib = _abi.lib()
    soa = _as_soa(world)
    sc, cm = _scene_struct(soa), _camera_struct(cam)
    prm = _params(samples_per_px, max_depth, seed, flags, samples_per_unit)
    devs = list(devices) if devices else [0]
    arr = (C.c_int32 * len(devs))(*devs)
    n = C.c_size_t()
    _abi.check(lib.rtclj_render_multi_png(C.byref(sc), C.byref(cm), C.byref(prm), arr, len(devs), None, 0, C.byref(n), None))
    store = bytearray(n.value)
    buf = (C.c_char * n.value).from_buffer(store)
    st = _abi.Stats()
    _abi.check(lib.rtclj_render_multi_png(C.byref(sc), C.byref(cm), C.byref(prm), arr, len(devs), buf, n.value,
                                          C.byref(n), C.byref(st)))
    del buf
    return bytes(memoryview(store)[: n.value]), st.as_dict()


def render_frames_apng(world, cameras: Sequence, samples_per_px: int = 100, max_depth: int = 50, *, seed: int = 1,
                       flags: int = _abi.FLAGS_MAIN, samples_per_unit: int = 0, devices: Optional[Sequence[int]] = None,
                       shard_rows: int = 0, delay=(1, 30), plays: int = 0) -> bytes:
    """A camera sequence as one animated PNG (rtclj_render_frames_apng): the frames rendered as `render_frames` renders
    them, rows interleaved over `devices` (default [0]) in tiles of `shard_rows` rows, assembled on devices[0] and
    encoded there; only the file leaves the GPU.  delay = (numerator, denominator) seconds per frame, plays = loops
    (0: forever).  The bytes are those of encode_apng(rgb8 of render_frames(...), delay=delay, plays=plays)."""
    lib = _abi.lib()
    soa = _as_soa(world)
    sc = _scene_struct(soa)
    arr, n = _camera_array(cameras)
    prm = _params(samples_per_px, max_depth, seed, flags, samples_per_unit)
    prm.shard_rows = int(shard_rows)
    devs = list(devices) if devices else [0]
    darr = (C.c_int32 * len(devs))(*devs)
    num, den = (int(x) for x in delay)
    size = C.c_size_t()
    _abi.check(lib.rtclj_render_frames_apng(C.byref(sc), arr, n, C.byref(prm), num, den, int(plays), darr, len(devs),
                                            None, 0, C.byref(size), None))
    store = bytearray(size.value)
    buf = (C.c_char * size.value).from_buffer(store)
    _abi.check(lib.rtclj_render_frames_apng(C.byref(sc), arr, n, C.byref(prm), num, den, int(plays), darr, len(devs),
                                            buf, size.value, C.byref(size), None))
    del buf
    return bytes(memoryview(store)[: size.value])


#: the denoiser's defaults (DESIGN.md section 4.13: the sweep that chose them)
DENOISE_LEVELS, DENOISE_SIGMA_COLOR, DENOISE_SIGMA_GUIDE, DENOISE_GUIDE_SAMPLES = 3, 0.5, 0.4, 4


def _sigma(sigma_color, sigma_guide):
    return (C.c_double * 2)(float(sigma_color), float(sigma_guide))


def denoise(linear: np.ndarray, guide: np.ndarray, *, device: int = 0, levels: int = DENOISE_LEVELS,
            sigma_color: float = DENOISE_SIGMA_COLOR, sigma_guide: float = DENOISE_SIGMA_GUIDE, flags: int = 0):
    """The edge-avoiding a-trous filter of include/rtclj_b200.h on GPU `device` (rtclj_denoise_gpu): `linear` (the
    colour, float64 [H,W,3]) filtered under the edges of `guide` (float64 [H,W,3], the normal-shaded primary render of
    the same camera and seed: render(..., flags=FLAGS_I, max_depth=1)).  flags: only F_QUANT_LINEAR is read, for the
    8-bit image.  Returns (linear float64 [H,W,3], rgb8 uint8 [H,W,3])."""
    lin = np.ascontiguousarray(linear, dtype=np.float64)
    gd = np.ascontiguousarray(guide, dtype=np.float64)
    if lin.ndim != 3 or lin.shape[2] != 3 or gd.shape != lin.shape:
        raise ValueError(f"linear and guide must be [H,W,3] images of one size, got {lin.shape} and {gd.shape}")
    H, W, _ = lin.shape
    out_linear = np.empty_like(lin)
    out_rgb8 = np.empty(lin.shape, dtype=np.uint8)
    _abi.check(_abi.lib().rtclj_denoise_gpu(int(device), lin.ctypes.data, gd.ctypes.data, W, H, int(levels),
                                            _sigma(sigma_color, sigma_guide), int(flags), out_linear.ctypes.data,
                                            out_rgb8.ctypes.data))
    return out_linear, out_rgb8


def render_denoised(world, cam: Camera, samples_per_px: int = 100, max_depth: int = 50, *, seed: int = 1,
                    flags: int = _abi.FLAGS_MAIN, samples_per_unit: int = 0, devices: Optional[Sequence[int]] = None,
                    shard_rows: int = 0, guide_samples: int = DENOISE_GUIDE_SAMPLES, levels: int = DENOISE_LEVELS,
                    sigma_color: float = DENOISE_SIGMA_COLOR, sigma_guide: float = DENOISE_SIGMA_GUIDE,
                    want_linear: bool = True, want_rgb8: bool = True):
    """Render, guide and filter in one call (rtclj_render_denoised): the colour render as `render`, rows interleaved
    over `devices` (default [0]) in tiles of `shard_rows` rows; the guide rendered with the same camera and seed,
    guide_samples samples, max_depth 1 and normal shading; both assembled on devices[0] and denoised there.  Returns
    (linear float64 [H,W,3] | None, rgb8 uint8 [H,W,3] | None, stats dict): the stats are the colour render's, except
    total_ms, which covers the whole call."""
    lib = _abi.lib()
    soa = _as_soa(world)
    sc, cm = _scene_struct(soa), _camera_struct(cam)
    H, W = cm.height, cm.width
    out_linear = np.zeros((H, W, 3), dtype=np.float64) if want_linear else None
    out_rgb8 = np.zeros((H, W, 3), dtype=np.uint8) if want_rgb8 else None
    prm = _params(samples_per_px, max_depth, seed, flags, samples_per_unit)
    prm.shard_rows = int(shard_rows)
    devs = list(devices) if devices else [0]
    arr = (C.c_int32 * len(devs))(*devs)
    st = _abi.Stats()
    _abi.check(lib.rtclj_render_denoised(C.byref(sc), C.byref(cm), C.byref(prm), int(guide_samples), int(levels),
                                         _sigma(sigma_color, sigma_guide), arr, len(devs),
                                         out_linear.ctypes.data if out_linear is not None else None,
                                         out_rgb8.ctypes.data if out_rgb8 is not None else None, C.byref(st)))
    return out_linear, out_rgb8, st.as_dict()


def pass_unit(width: int, height: int, samples_per_px: int, max_depth: int, flags: int = _abi.FLAGS_MAIN,
              samples_per_unit: int = 0) -> int:
    """The pass unit an accumulation of these params reports (rtclj_ctx_accum_begin): 1 in strict order, else the
    unit size of the one-shot render (the library's choice for samples_per_unit <= 0)."""
    primary_only = max_depth == 1 or bool(flags & _abi.F_NORMAL_SHADING)
    if samples_per_unit >= samples_per_px or (samples_per_unit <= 0 and primary_only):
        return 1
    if samples_per_unit > 0:
        return samples_per_unit
    nchunks = math.ceil((64.0 * 148.0 * 512.0 * 8.0) / (float(width) * float(height)))  # auto_samples_per_unit
    nchunks = max(1, min(nchunks, max(1, samples_per_px // 8)))
    return (samples_per_px + nchunks - 1) // nchunks


def _adaptive_args(cam, samples_per_px, max_depth, flags, samples_per_unit, tolerance, min_samples):
    """(double[2] tolerance, min_samples) of an adaptive accumulation; min_samples <= 0: two pass units."""
    abs_tol, rel_tol = (float(x) for x in tolerance)
    if min_samples <= 0:
        min_samples = 2 * pass_unit(cam.width, cam.height, samples_per_px, max_depth, flags, samples_per_unit)
    return (C.c_double * 2)(abs_tol, rel_tol), int(min_samples)


def _frames_adaptive_args(arr, n, samples_per_px, max_depth, flags, samples_per_unit, tolerance, min_samples):
    """(double[2] tolerance or None, min_samples) of an accumulation over frames: tolerance None is a plain one."""
    if tolerance is None:
        return None, 0
    cam = arr[0] if n else _abi.Camera()
    return _adaptive_args(cam, int(samples_per_px), int(max_depth), int(flags), int(samples_per_unit), tolerance,
                          int(min_samples))


class Context:
    """Device-resident rendering: scene uploaded once, output left in device memory
    (pointers come from the caller, e.g. torch tensors), launches enqueued on the caller's
    CUDA stream.  This is what bench.py times as the in-HBM `value`."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        _abi.check(_abi.lib().rtclj_ctx_create(int(device), C.byref(self._h)))
        self.device = device

    def set_scene(self, world) -> None:
        soa = _as_soa(world)
        sc = _scene_struct(soa)
        _abi.check(_abi.lib().rtclj_ctx_set_scene(self._h, C.byref(sc)))

    def render(self, cam, samples_per_px: int, max_depth: int, *, seed: int = 1, flags: int = _abi.FLAGS_MAIN,
               samples_per_unit: int = 0, shard: Optional[tuple] = None, d_out_linear: int = 0,
               d_out_rgb8: int = 0, stream: int = 0) -> None:
        cm = _camera_struct(cam)
        prm = _params(samples_per_px, max_depth, seed, flags, samples_per_unit, self.device)
        if shard is not None:
            prm.shard_index, prm.shard_count, prm.shard_rows = (int(x) for x in shard)
        _abi.check(_abi.lib().rtclj_ctx_render(self._h, C.byref(cm), C.byref(prm),
                                               C.c_void_p(d_out_linear or None), C.c_void_p(d_out_rgb8 or None),
                                               C.c_void_p(stream or None)))

    def render_frames(self, cameras: Sequence, samples_per_px: int, max_depth: int, *, seed: int = 1,
                      flags: int = _abi.FLAGS_MAIN, samples_per_unit: int = 0, shard: Optional[tuple] = None,
                      d_out_linear: int = 0, d_out_rgb8: int = 0, stream: int = 0) -> None:
        """Enqueues a camera sequence (rtclj_ctx_render_frames): the device images hold len(cameras) full-size
        frames, frame f bit-identical to render(cameras[f], ...)."""
        arr, n = _camera_array(cameras)
        prm = _params(samples_per_px, max_depth, seed, flags, samples_per_unit, self.device)
        if shard is not None:
            prm.shard_index, prm.shard_count, prm.shard_rows = (int(x) for x in shard)
        _abi.check(_abi.lib().rtclj_ctx_render_frames(self._h, arr, n, C.byref(prm),
                                                      C.c_void_p(d_out_linear or None), C.c_void_p(d_out_rgb8 or None),
                                                      C.c_void_p(stream or None)))

    def stats(self, stream: int = 0) -> dict:
        st = _abi.Stats()
        _abi.check(_abi.lib().rtclj_ctx_stats(self._h, C.c_void_p(stream or None), C.byref(st)))
        return st.as_dict()

    def accum_begin(self, cam, samples_per_px: int, max_depth: int, *, seed: int = 1, flags: int = _abi.FLAGS_MAIN,
                    samples_per_unit: int = 0, shard: Optional[tuple] = None, stream: int = 0,
                    tolerance: Optional[Sequence[float]] = None, min_samples: int = 0) -> int:
        """Begins an accumulation over passes (rtclj_ctx_accum_begin) towards `samples_per_px` samples and
        returns its pass unit: every pass but the last must be a multiple of it.  tolerance = (abs, rel): an
        adaptive accumulation (rtclj_ctx_accum_begin_adaptive) whose passes trace only the pixels whose noise
        estimate is still above abs + rel * |mean|, after at least min_samples samples (<= 0: two pass units)."""
        cm = _camera_struct(cam)
        prm = _params(samples_per_px, max_depth, seed, flags, samples_per_unit, self.device)
        if shard is not None:
            prm.shard_index, prm.shard_count, prm.shard_rows = (int(x) for x in shard)
        unit = C.c_int32()
        if tolerance is None:
            _abi.check(_abi.lib().rtclj_ctx_accum_begin(self._h, C.byref(cm), C.byref(prm), C.byref(unit),
                                                        C.c_void_p(stream or None)))
        else:
            tol, least = _adaptive_args(cm, int(samples_per_px), int(max_depth), int(flags), int(samples_per_unit),
                                        tolerance, int(min_samples))
            _abi.check(_abi.lib().rtclj_ctx_accum_begin_adaptive(self._h, C.byref(cm), C.byref(prm), tol, least,
                                                                 C.byref(unit), C.c_void_p(stream or None)))
        return unit.value

    def accum_begin_frames(self, cameras: Sequence, samples_per_px: int, max_depth: int, *, seed: int = 1,
                           flags: int = _abi.FLAGS_MAIN, samples_per_unit: int = 0, shard: Optional[tuple] = None,
                           stream: int = 0, tolerance: Optional[Sequence[float]] = None, min_samples: int = 0) -> int:
        """Begins an accumulation over the frames of a camera sequence (rtclj_ctx_accum_begin_frames; plain, or
        adaptive with `tolerance` as in accum_begin) and returns the pass unit, the single frame's.  accum_step,
        accum_noise and stats then serve all frames: the device buffers hold len(cameras) full-size frames one after
        the other, frame f bit-identical to an accumulation of cameras[f] alone stepped alike."""
        arr, n = _camera_array(cameras)
        prm = _params(samples_per_px, max_depth, seed, flags, samples_per_unit, self.device)
        if shard is not None:
            prm.shard_index, prm.shard_count, prm.shard_rows = (int(x) for x in shard)
        tol, least = _frames_adaptive_args(arr, n, samples_per_px, max_depth, flags, samples_per_unit, tolerance,
                                           min_samples)
        unit = C.c_int32()
        _abi.check(_abi.lib().rtclj_ctx_accum_begin_frames(self._h, arr, n, C.byref(prm), tol, least, C.byref(unit),
                                                           C.c_void_p(stream or None)))
        return unit.value

    def accum_noise(self, d_samples: int = 0, d_stderr: int = 0, stream: int = 0) -> int:
        """After a step of an adaptive accumulation: writes this context's rows of the sample-count map (int32
        [H,W]) and of the noise estimate (float64 [H,W,3]) to the device pointers (either may be 0), and returns
        the number of pixels still active (synchronises `stream`)."""
        active = C.c_uint64()
        _abi.check(_abi.lib().rtclj_ctx_accum_noise(self._h, C.c_void_p(d_samples or None), C.c_void_p(d_stderr or None),
                                                    C.byref(active), C.c_void_p(stream or None)))
        return active.value

    def accum_step(self, samples: int, d_out_linear: int = 0, d_out_rgb8: int = 0, stream: int = 0) -> int:
        """Enqueues one pass of `samples` samples per pixel (rtclj_ctx_accum_step); the images at the device
        pointers are those of a one-shot render of all samples so far.  Returns the samples done."""
        done = C.c_int32()
        _abi.check(_abi.lib().rtclj_ctx_accum_step(self._h, int(samples), C.c_void_p(d_out_linear or None),
                                                   C.c_void_p(d_out_rgb8 or None), C.byref(done),
                                                   C.c_void_p(stream or None)))
        return done.value

    def encode_ppm(self, d_rgb8: int, width: int, height: int, d_out: int = 0, capacity: int = 0,
                   stream: int = 0) -> int:
        """The P3 writer (raytracing.clj:172-175) as device kernels: d_rgb8 -> text at d_out, both
        device pointers.  d_out = 0 is the sizing call.  Returns the text length in bytes."""
        n = C.c_size_t()
        _abi.check(_abi.lib().rtclj_ctx_encode_ppm_p3(self._h, C.c_void_p(d_rgb8), int(width), int(height),
                                                      C.c_void_p(d_out or None), int(capacity), C.byref(n),
                                                      C.c_void_p(stream or None)))
        return n.value

    def encode_png(self, d_rgb8: int, width: int, height: int, d_out: int = 0, capacity: int = 0,
                   stream: int = 0) -> int:
        """The compressed PNG writer (rtclj_ctx_encode_png) on device pointers: d_rgb8 -> PNG at d_out.  d_out = 0
        is the sizing call (a sufficient capacity, no GPU work).  Returns the PNG length in bytes; synchronises
        `stream`."""
        n = C.c_size_t()
        _abi.check(_abi.lib().rtclj_ctx_encode_png(self._h, C.c_void_p(d_rgb8), int(width), int(height),
                                                   C.c_void_p(d_out or None), int(capacity), C.byref(n),
                                                   C.c_void_p(stream or None)))
        return n.value

    def encode_apng(self, d_frames: int, width: int, height: int, n_frames: int, d_out: int = 0, capacity: int = 0, *,
                    delay=(1, 30), plays: int = 0, stream: int = 0) -> int:
        """The animated PNG writer (rtclj_ctx_encode_apng) on device pointers: n_frames consecutive uint8 [H,W,3]
        frames at d_frames -> APNG at d_out.  d_out = 0 is the sizing call (a sufficient capacity, no GPU work).
        Returns the file's length in bytes; synchronises `stream`."""
        n = C.c_size_t()
        num, den = (int(x) for x in delay)
        _abi.check(_abi.lib().rtclj_ctx_encode_apng(self._h, C.c_void_p(d_frames or None), int(width), int(height),
                                                    int(n_frames), num, den, int(plays), C.c_void_p(d_out or None),
                                                    int(capacity), C.byref(n), C.c_void_p(stream or None)))
        return n.value

    def denoise(self, d_linear: int, d_guide: int, width: int, height: int, *, levels: int = DENOISE_LEVELS,
                sigma_color: float = DENOISE_SIGMA_COLOR, sigma_guide: float = DENOISE_SIGMA_GUIDE, flags: int = 0,
                d_out_linear: int = 0, d_out_rgb8: int = 0, stream: int = 0) -> None:
        """Enqueues the denoiser (rtclj_ctx_denoise) on device pointers: d_linear / d_guide (float64 [H,W,3]) ->
        d_out_linear (float64, may equal d_linear) and d_out_rgb8 (uint8); either output may be 0."""
        _abi.check(_abi.lib().rtclj_ctx_denoise(self._h, C.c_void_p(d_linear or None), C.c_void_p(d_guide or None),
                                                int(width), int(height), int(levels), _sigma(sigma_color, sigma_guide),
                                                int(flags), C.c_void_p(d_out_linear or None),
                                                C.c_void_p(d_out_rgb8 or None), C.c_void_p(stream or None)))

    def encode_ms(self) -> tuple:
        """(line lengths + scan, text write) device milliseconds of the last encode_ppm call."""
        a, b = C.c_double(), C.c_double()
        _abi.check(_abi.lib().rtclj_ctx_encode_ms(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def close(self) -> None:
        if self._h:
            _abi.lib().rtclj_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Progressive:
    """A render that refines pass by pass (rtclj_progressive_*): the compute-pixel loop (raytracing.clj:141-171)
    run in passes into host buffers, rows interleaved over `devices` (default [0]).  After passes totalling d
    samples the images are bit-identical to `render(..., samples_per_px=d)` in the same summation order, so the
    last pass gives the one-shot image of `samples_per_px` samples.

        with Progressive(world, cam, 500, 50) as p:
            n = -(-25 // p.pass_unit) * p.pass_unit   # about 25 samples a pass, a multiple of the pass unit
            while p.samples_done < p.samples_per_px:
                lin, rgb8, st = p.step(min(n, p.samples_per_px - p.samples_done))   # show rgb8
    """

    def __init__(self, world, cam, samples_per_px: int = 100, max_depth: int = 50, *, seed: int = 1,
                 flags: int = _abi.FLAGS_MAIN, samples_per_unit: int = 0, devices: Optional[Sequence[int]] = None,
                 tolerance: Optional[Sequence[float]] = None, min_samples: int = 0):
        self._h = C.c_void_p()
        soa = _as_soa(world)
        sc, cm = _scene_struct(soa), _camera_struct(cam)
        self.height, self.width = cm.height, cm.width
        self.samples_per_px = int(samples_per_px)
        self.adaptive = tolerance is not None
        prm = _params(samples_per_px, max_depth, seed, flags, samples_per_unit)
        devs = list(devices) if devices else [0]
        arr = (C.c_int32 * len(devs))(*devs)
        unit = C.c_int32()
        if tolerance is None:
            _abi.check(_abi.lib().rtclj_progressive_create(C.byref(sc), C.byref(cm), C.byref(prm), arr, len(devs),
                                                           C.byref(unit), C.byref(self._h)))
        else:  # adaptive sampling (rtclj_progressive_create_adaptive): see Context.accum_begin
            tol, least = _adaptive_args(cm, int(samples_per_px), int(max_depth), int(flags), int(samples_per_unit),
                                        tolerance, int(min_samples))
            _abi.check(_abi.lib().rtclj_progressive_create_adaptive(C.byref(sc), C.byref(cm), C.byref(prm), tol, least,
                                                                    arr, len(devs), C.byref(unit), C.byref(self._h)))
        self.pass_unit = unit.value
        self.samples_done = 0

    def step(self, samples: int, *, want_linear: bool = True, want_rgb8: bool = True,
             out_linear: Optional[np.ndarray] = None, out_rgb8: Optional[np.ndarray] = None):
        """One pass of `samples` samples per pixel (the last pass may be any size; the others a multiple of
        pass_unit).  Returns (linear float64 [H,W,3] | None, rgb8 uint8 [H,W,3] | None, stats dict) of the
        image so far; out_linear / out_rgb8 are reused when given."""
        if not self._h:
            raise _abi.RtcljError(_abi.E_INVALID, "progressive render is closed")
        if want_linear and out_linear is None:
            out_linear = np.zeros((self.height, self.width, 3), dtype=np.float64)
        if want_rgb8 and out_rgb8 is None:
            out_rgb8 = np.zeros((self.height, self.width, 3), dtype=np.uint8)
        done, st = C.c_int32(), _abi.Stats()
        _abi.check(_abi.lib().rtclj_progressive_step(
            self._h, int(samples), out_linear.ctypes.data if out_linear is not None else None,
            out_rgb8.ctypes.data if out_rgb8 is not None else None, C.byref(done), C.byref(st)))
        self.samples_done = done.value
        return out_linear, out_rgb8, st.as_dict()

    def noise(self):
        """Adaptive renders: (samples int32 [H,W], the count each pixel has; stderr float64 [H,W,3], its noise
        estimate; active, the pixels the next pass would trace) after the last step."""
        if not self._h:
            raise _abi.RtcljError(_abi.E_INVALID, "progressive render is closed")
        samples = np.zeros((self.height, self.width), dtype=np.int32)
        stderr = np.zeros((self.height, self.width, 3), dtype=np.float64)
        active = C.c_uint64()
        _abi.check(_abi.lib().rtclj_progressive_noise(self._h, samples.ctypes.data, stderr.ctypes.data, C.byref(active)))
        return samples, stderr, active.value

    def close(self) -> None:
        if self._h:
            _abi.check(_abi.lib().rtclj_progressive_destroy(self._h))
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ProgressiveFrames(Progressive):
    """A camera sequence of one scene that refines pass by pass (rtclj_progressive_create_frames): every frame's pixels
    (adaptive: its live pixels) in shared launches, rows interleaved over `devices` (default [0]).  `Progressive`'s
    interface with arrays of K = len(cameras) frames: step returns linear float64 [K,H,W,3] and rgb8 uint8 [K,H,W,3],
    noise returns samples int32 [K,H,W], stderr float64 [K,H,W,3] and the active pixels of all frames.  After every
    step frame f is bit-identical to a `Progressive` of cameras[f] with the same arguments stepped alike.

        with ProgressiveFrames(world, turntable_cameras(60), 500, 50, tolerance=(0.004, 0.04)) as p:
            while p.samples_done < p.samples_per_px:
                lin, rgb8, st = p.step(min(50, p.samples_per_px - p.samples_done))
                if p.adaptive and p.noise()[2] == 0:
                    break   # every pixel of every frame has stopped
    """

    def __init__(self, world, cameras: Sequence, samples_per_px: int = 100, max_depth: int = 50, *, seed: int = 1,
                 flags: int = _abi.FLAGS_MAIN, samples_per_unit: int = 0, devices: Optional[Sequence[int]] = None,
                 tolerance: Optional[Sequence[float]] = None, min_samples: int = 0):
        self._h = C.c_void_p()
        soa = _as_soa(world)
        sc = _scene_struct(soa)
        arr, n = _camera_array(cameras)
        self.frames = n
        self.height, self.width = (arr[0].height, arr[0].width) if n else (0, 0)
        self.samples_per_px = int(samples_per_px)
        self.adaptive = tolerance is not None
        prm = _params(samples_per_px, max_depth, seed, flags, samples_per_unit)
        tol, least = _frames_adaptive_args(arr, n, samples_per_px, max_depth, flags, samples_per_unit, tolerance,
                                           min_samples)
        devs = list(devices) if devices else [0]
        darr = (C.c_int32 * len(devs))(*devs)
        unit = C.c_int32()
        _abi.check(_abi.lib().rtclj_progressive_create_frames(C.byref(sc), arr, n, C.byref(prm), tol, least, darr,
                                                              len(devs), C.byref(unit), C.byref(self._h)))
        self.pass_unit = unit.value
        self.samples_done = 0

    def step(self, samples: int, *, want_linear: bool = True, want_rgb8: bool = True,
             out_linear: Optional[np.ndarray] = None, out_rgb8: Optional[np.ndarray] = None):
        K, H, W = self.frames, self.height, self.width
        if want_linear and out_linear is None:
            out_linear = np.zeros((K, H, W, 3), dtype=np.float64)
        if want_rgb8 and out_rgb8 is None:
            out_rgb8 = np.zeros((K, H, W, 3), dtype=np.uint8)
        return super().step(samples, want_linear=want_linear, want_rgb8=want_rgb8, out_linear=out_linear,
                            out_rgb8=out_rgb8)

    def noise(self):
        if not self._h:
            raise _abi.RtcljError(_abi.E_INVALID, "progressive render is closed")
        K, H, W = self.frames, self.height, self.width
        samples = np.zeros((K, H, W), dtype=np.int32)
        stderr = np.zeros((K, H, W, 3), dtype=np.float64)
        active = C.c_uint64()
        _abi.check(_abi.lib().rtclj_progressive_noise(self._h, samples.ctypes.data, stderr.ctypes.data, C.byref(active)))
        return samples, stderr, active.value


def quantise_rgb8(linear: np.ndarray, flags: int = 0) -> np.ndarray:
    """write-color!'s arithmetic (raytracing.clj:19-26), on the host."""
    lin = np.ascontiguousarray(linear, dtype=np.float64)
    out = np.zeros(lin.shape, dtype=np.uint8)
    _abi.check(_abi.lib().rtclj_quantise_rgb8(lin.ctypes.data, lin.size, int(flags), out.ctypes.data))
    return out


def _two_call(fn, img: np.ndarray, *lead) -> bytes:
    """Sizing call, then the real call into a caller-owned buffer."""
    H, W, _ = img.shape
    n = C.c_size_t()
    _abi.check(fn(*lead, img.ctypes.data, W, H, None, 0, C.byref(n)))
    store = bytearray(n.value)
    buf = (C.c_char * n.value).from_buffer(store)
    _abi.check(fn(*lead, img.ctypes.data, W, H, buf, n.value, C.byref(n)))
    del buf
    return bytes(memoryview(store)[: n.value])


def encode_ppm(rgb8: np.ndarray, device: int | None = None) -> bytes:
    """"P3\\nW H\\n255\\n" then one "r g b\\n" line per pixel (raytracing.clj:172-175).
    device = None: the host encoder; device = k: the encoder kernels on GPU k (same bytes)."""
    img = np.ascontiguousarray(rgb8, dtype=np.uint8)
    lib = _abi.lib()
    if device is None:
        return _two_call(lib.rtclj_encode_ppm_p3, img)
    return _two_call(lib.rtclj_encode_ppm_p3_gpu, img, int(device))


def encode_png(rgb8: np.ndarray, device: int | None = None) -> bytes:
    """The PNG `ppm->png` writes next to the PPM (raytracing.clj:176).
    device = None: the host writer (stored deflate blocks); device = k: the compressed PNG writer on GPU k
    (rtclj_encode_png_gpu: filtered rows, run-length deflate, DESIGN.md section 4.11)."""
    img = np.ascontiguousarray(rgb8, dtype=np.uint8)
    if device is None:
        return _two_call(_abi.lib().rtclj_encode_png, img)
    return _two_call(_abi.lib().rtclj_encode_png_gpu, img, int(device))


def encode_apng(frames: np.ndarray, device: int = 0, delay=(1, 30), plays: int = 0) -> bytes:
    """An animated PNG of `frames` (uint8 [K,H,W,3]) written by the device PNG writer on GPU `device`
    (rtclj_encode_apng_gpu, DESIGN.md section 4.14): each frame's data are those of encode_png(frame, device).
    delay = (numerator, denominator) seconds per frame, plays = loops (0: forever)."""
    img = np.ascontiguousarray(frames, dtype=np.uint8)
    if img.ndim != 4 or img.shape[3] != 3:
        raise ValueError(f"frames must be a [K,H,W,3] array, got shape {img.shape}")
    K, H, W, _ = img.shape
    num, den = (int(x) for x in delay)
    lib = _abi.lib()
    n = C.c_size_t()
    _abi.check(lib.rtclj_encode_apng_gpu(int(device), img.ctypes.data, W, H, K, num, den, int(plays), None, 0, C.byref(n)))
    store = bytearray(n.value)
    buf = (C.c_char * n.value).from_buffer(store)
    _abi.check(lib.rtclj_encode_apng_gpu(int(device), img.ctypes.data, W, H, K, num, den, int(plays), buf, n.value,
                                         C.byref(n)))
    del buf
    return bytes(memoryview(store)[: n.value])


def decode_ppm(text: bytes) -> np.ndarray:
    """The reader half of `ppm->png` (ppm2png.clj:35-87): P3 text -> uint8 [H,W,3]."""
    lib = _abi.lib()
    w, h = C.c_int32(), C.c_int32()
    _abi.check(lib.rtclj_decode_ppm_p3(text, len(text), C.byref(w), C.byref(h), None, 0))
    out = np.zeros((h.value, w.value, 3), dtype=np.uint8)
    _abi.check(lib.rtclj_decode_ppm_p3(text, len(text), C.byref(w), C.byref(h), out.ctypes.data, out.size))
    return out


def ppm_to_png(source: str, dest: str) -> None:
    """`(ppm->png source dest)`, raytracing.clj:176."""
    with open(source, "rb") as f:
        rgb8 = decode_ppm(f.read())
    write_png(dest, rgb8)
    print(f"Processed {source} into {dest}")


def write_png(path: str, rgb8: np.ndarray, device: int | None = None) -> None:
    with open(path, "wb") as f:
        f.write(encode_png(rgb8, device))


def write_ppm(path: str, rgb8: np.ndarray, device: int | None = None) -> None:
    with open(path, "wb") as f:
        f.write(encode_ppm(rgb8, device))
