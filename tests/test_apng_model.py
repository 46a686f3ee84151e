"""The device APNG writer's definition (include/rtclj_b200.h, DESIGN.md section 4.14), checked on its numpy model without
a GPU: the model's files play as the input frames, carry the device PNG of every frame, number their chunks as the
format says; the library sizes and refuses without a device, exports and declares the new calls, ships their kernels
without local memory, and the Clojure shim binds them."""
import ctypes as C
import io
import os
import re
import shutil
import struct
import subprocess
import zlib

import numpy as np
import pytest
from PIL import Image

import apng_model as A
import png_model as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "raytracing-clj_b200", "librtclj_b200.so")
CASES = A.cpu_cases()
NEW = ("rtclj_ctx_encode_apng", "rtclj_encode_apng_gpu", "rtclj_render_frames_apng")


def chunks(data: bytes):
    """[(type, data)] with every CRC checked."""
    assert data[:8] == P.SIG
    i, out = 8, []
    while i < len(data):
        n = struct.unpack(">I", data[i:i + 4])[0]
        kind, body = data[i + 4:i + 8], data[i + 8:i + 8 + n]
        assert struct.unpack(">I", data[i + 8 + n:i + 12 + n])[0] == zlib.crc32(kind + body) & 0xFFFFFFFF
        out.append((kind, body))
        i += 12 + n
    assert i == len(data)
    return out


def frames_of(data: bytes):
    """Pillow's decoding: (frames [K,H,W,3], durations in ms, loop)."""
    im = Image.open(io.BytesIO(data))
    out, durations = [], []
    for k in range(im.n_frames):
        im.seek(k)
        out.append(np.array(im.convert("RGB")))
        durations.append(im.info.get("duration"))
    return np.stack(out), durations, im.info.get("loop")


@pytest.mark.parametrize("name", sorted(CASES))
def test_pillow_plays_the_input_frames(name):
    frames, delay, plays = CASES[name]
    got, durations, loop = frames_of(A.encode(frames, delay, plays))
    assert np.array_equal(got, frames)
    ms = 1000.0 * delay[0] / (delay[1] or 100)
    assert durations == [pytest.approx(ms)] * len(frames)
    assert loop == plays


@pytest.mark.parametrize("name", sorted(CASES))
def test_without_the_animation_chunks_the_file_is_frame_0s_png(name):
    frames, delay, plays = CASES[name]
    data = A.encode(frames, delay, plays)
    kept = [(k, d) for k, d in chunks(data) if k not in (b"acTL", b"fcTL", b"fdAT")]
    png = P.SIG + b"".join(P._chunk(k, d) for k, d in kept)
    assert png == P.encode(frames[0])


@pytest.mark.parametrize("name", sorted(CASES))
def test_every_frame_carries_its_own_png_stream(name):
    frames, delay, plays = CASES[name]
    ch = chunks(A.encode(frames, delay, plays))
    per_frame, cur = [], None
    for kind, body in ch:
        if kind == b"fcTL":
            cur = []
            per_frame.append(cur)
        elif kind == b"IDAT":
            cur.append(body)
        elif kind == b"fdAT":
            cur.append(body[4:])
    assert len(per_frame) == len(frames)
    for f, data in enumerate(per_frame):
        own = [d for k, d in chunks(P.encode(frames[f])) if k == b"IDAT"]
        assert data == own, f
        assert b"".join(data) and zlib.decompress(b"".join(data)) == P.filter_rows(frames[f])[0].tobytes()


@pytest.mark.parametrize("name", sorted(CASES))
def test_chunk_order_and_sequence_numbers(name):
    frames, delay, plays = CASES[name]
    K, H, W, _ = frames.shape
    ns = A.nseg(W, H)
    ch = chunks(A.encode(frames, delay, plays))
    kinds = [k for k, _ in ch]
    want = [b"IHDR", b"acTL"] + [b"fcTL"] + [b"IDAT"] * (ns + 2)
    for _ in range(1, K):
        want += [b"fcTL"] + [b"fdAT"] * (ns + 2)
    assert kinds == want + [b"IEND"]
    assert ch[1][1] == struct.pack(">II", K, plays)
    seqs = [struct.unpack(">I", d[:4])[0] for k, d in ch if k in (b"fcTL", b"fdAT")]
    assert seqs == list(range(len(seqs)))
    fctls = [d for k, d in ch if k == b"fcTL"]
    for f, d in enumerate(fctls):
        assert struct.unpack(">I", d[:4])[0] == (0 if f == 0 else 1 + (f - 1) * (ns + 3))
        assert d[4:] == struct.pack(">IIIIHHBB", W, H, 0, 0, delay[0], delay[1], 0, 0)


def test_cases_cover_the_edges():
    segs = lambda fr: len(range(0, len(P.filter_rows(fr)[0]), P.SEG))  # noqa: E731
    assert len(CASES["K1_main"][0]) == 1
    assert CASES["1x1_K4"][0].shape[1:3] == (1, 1)
    assert len(P.filter_rows(CASES["F_1x65536_K3"][0][0])[0]) == P.SEG
    assert len(P.filter_rows(CASES["F_3x65536_plus_1_K2"][0][0])[0]) == 3 * P.SEG + 1
    assert segs(CASES["F_3x65536_plus_1_K2"][0][0]) == 4
    kinds = []
    for fr in CASES["noise_and_constant"][0]:
        info = {}
        P.encode(fr, info)
        kinds.append(set(info["kinds"]))
    assert kinds == [{"stored"}, {"dynamic"}, {"stored"}, {"dynamic"}]
    assert CASES["delay_0_0"][1] == (0, 0) and CASES["delay_65535"][1] == (65535, 65535)


@pytest.mark.parametrize("W,H,K", [(1, 1, 1), (1, 1, 5), (85, 256, 3), (400, 225, 60), (30000, 3, 2), (1920, 1080, 4)])
def test_sizing_formula_is_the_all_stored_size(W, H, K):
    assert A.stored_bound(W, H, K) == A.stored_size(W, H, K)


def test_all_stored_frames_reach_the_bound():
    noise = np.random.default_rng(4).integers(0, 256, (3, 250, 300, 3), dtype=np.uint8)
    assert len(A.encode(noise)) == A.stored_bound(300, 250, 3)


needs_lib = pytest.mark.skipif(not os.path.exists(LIB), reason="library not built")


@needs_lib
def test_new_symbols_are_exported_and_declared():
    lib = C.CDLL(LIB)
    hdr = open(os.path.join(ROOT, "include", "rtclj_b200.h")).read()
    from raytracing_clj_b200 import _abi
    for name in NEW:
        assert getattr(lib, name)
        assert re.search(r"\b%s\(" % name, hdr)
        assert name in _abi.SYMBOLS


def _gpu_call(W, H, K, delay=(1, 30), plays=0, out=None, length=True):
    from raytracing_clj_b200 import _abi
    n = C.c_size_t()
    rc = _abi.lib().rtclj_encode_apng_gpu(0, None, W, H, K, delay[0], delay[1], plays, out, 0,
                                          C.byref(n) if length else None)
    return rc, n.value


@needs_lib
def test_sizing_calls_and_refusals_need_no_gpu():
    from raytracing_clj_b200 import _abi
    for W, H, K in ((400, 225, 60), (1, 1, 1), (1920, 1080, 8)):
        assert _gpu_call(W, H, K) == (0, A.stored_bound(W, H, K))
    assert _gpu_call(400, 225, 2, delay=(0, 0), plays=65535)[0] == 0
    assert _gpu_call(400, 225, 2, delay=(65535, 65535), plays=2 ** 31 - 1)[0] == 0
    E = _abi.E_INVALID
    for bad in (dict(K=0), dict(K=-1), dict(W=0), dict(H=-5), dict(delay=(-1, 30)), dict(delay=(1, 65536)),
                dict(delay=(65536, 1)), dict(delay=(1, -1)), dict(plays=-1), dict(length=False)):
        args = dict(W=400, H=225, K=3, delay=(1, 30), plays=0, length=True)
        args.update(bad)
        assert _gpu_call(**args)[0] == E, bad
    # the sequence-number limit: the last number (K - 1)(nseg + 3) must stay <= 2^31 - 1; 400 x 225 has 5 segments
    last_ok = (2 ** 31 - 1) // 8 + 1
    assert _gpu_call(400, 225, last_ok)[0] == 0
    assert _gpu_call(400, 225, last_ok + 1)[0] == E
    # the device-buffer call: a null context, and null frames once the output is given
    n = C.c_size_t()
    lib = _abi.lib()
    assert lib.rtclj_ctx_encode_apng(None, None, 4, 4, 2, 1, 30, 0, None, 0, C.byref(n), None) == E
    assert lib.rtclj_encode_apng_gpu(0, None, 4, 4, 2, 1, 30, 0, C.c_void_p(8), 100, C.byref(n)) == E


@needs_lib
def test_render_frames_apng_refuses_what_render_frames_refuses():
    import raytracing_clj_b200 as R
    from raytracing_clj_b200 import _abi
    lib = _abi.lib()
    sc = R.render._scene_struct(R.scenes.to_soa(R.scenes.main_hittables()))
    cams = [R.camera.main_camera(32, look_from=R.camera.turntable_look_from(k, 4)) for k in range(4)]

    def call(cams, flags=_abi.FLAGS_MAIN, delay=(1, 30), plays=0, n=None):
        arr = (_abi.Camera * len(cams))(*[R.render._camera_struct(c) for c in cams])
        prm = _abi.Params(4, 5, 1, flags, 0, 0, 0, 0, 0, 0)
        devs = (C.c_int32 * 1)(0)
        size = C.c_size_t()
        rc = lib.rtclj_render_frames_apng(C.byref(sc), arr, len(cams) if n is None else n, C.byref(prm), delay[0],
                                          delay[1], plays, devs, 1, None, 0, C.byref(size), None)
        return rc, lib.rtclj_last_error().decode(), size.value

    rc, _, size = call(cams)
    assert rc == 0 and size == A.stored_bound(32, 18, 4)
    rc, msg, _ = call(cams[:2] + [R.camera.main_camera(48)] + cams[3:])
    assert rc == _abi.E_INVALID and "frame 2" in msg
    bad = _abi.Camera.from_buffer_copy(R.render._camera_struct(cams[1]))
    bad.center[0] = float("inf")
    rc, msg, _ = call(cams[:1] + [bad])
    assert rc == _abi.E_INVALID and "frame 1" in msg
    for f in (_abi.F_WAVE_KERNEL, _abi.F_SPLIT_KERNEL):
        rc, msg, _ = call(cams, flags=_abi.FLAGS_MAIN | f)
        assert rc == _abi.E_INVALID and "sequence" in msg
    assert call(cams, n=0)[0] == _abi.E_INVALID
    assert call(cams, delay=(1, 70000))[0] == _abi.E_INVALID
    assert call(cams, plays=-2)[0] == _abi.E_INVALID


def test_cli_refuses_apng_without_frames():
    import raytracing_clj_b200 as R
    with pytest.raises(SystemExit) as e:
        R.main._cli(["main", "4", "5", "--apng"])
    assert "--frames" in str(e.value)


@needs_lib
@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not installed")
def test_apng_kernels_use_no_local_memory():
    out = subprocess.run(["cuobjdump", "-sass", LIB], check=True, capture_output=True, text=True).stdout
    bodies = {}
    for part in re.split(r"\n\s*Function : ", out)[1:]:
        bodies[part.split("\n", 1)[0].strip()] = part
    for k in ("png_filter_frames_kernel", "png_deflate_frames_kernel", "png_place_frames_kernel"):
        found = [b for n, b in bodies.items() if k in n]
        assert len(found) == 1, k
        assert not re.search(r"\b(LDL|STL)\b", found[0]), k


def test_clojure_shim_binds_the_new_calls():
    text = open(os.path.join(ROOT, "integration", "clojure", "src", "rtclj", "native.clj")).read()
    for name in ("rtclj_render_frames_apng", "rtclj_encode_apng_gpu"):
        assert '(downcall "%s"' % name in text
    assert "(defn render-frames-apng!" in text and "(defn encode-apng-gpu" in text
