"""The device PNG writer's definition (include/rtclj_b200.h, DESIGN.md section 4.11), checked on its numpy model
without a GPU: the model's files decode to their input, follow the filter heuristic and compress as the format was
chosen to; the library exports the new calls, ships their kernels without local memory, and the Clojure shim binds
them."""
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

import png_model as M

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "raytracing-clj_b200", "librtclj_b200.so")
CASES = M.cpu_cases()
NEW = ("rtclj_ctx_encode_png", "rtclj_encode_png_gpu", "rtclj_render_multi_png")


def chunks(png: bytes):
    assert png[:8] == M.SIG
    i, out = 8, []
    while i < len(png):
        n = struct.unpack(">I", png[i:i + 4])[0]
        kind, data = png[i + 4:i + 8], png[i + 8:i + 8 + n]
        assert struct.unpack(">I", png[i + 8 + n:i + 12 + n])[0] == zlib.crc32(kind + data) & 0xFFFFFFFF
        out.append((kind, data))
        i += 12 + n
    return out


def heuristic_types(img):
    """The filter each row should get, computed row by row from the PNG specification's predictor definitions
    (int32 arithmetic, the Paeth predictor by its three comparisons), independently of the model's blocked code."""
    H, W, _ = img.shape
    rows = img.reshape(H, 3 * W).astype(np.int32)
    types = []
    for y in range(H):
        x = rows[y]
        b = rows[y - 1] if y else np.zeros(3 * W, np.int32)
        a = np.concatenate([np.zeros(3, np.int32), x[:-3]])[:3 * W]
        c = np.concatenate([np.zeros(3, np.int32), b[:-3]])[:3 * W]
        p = a + b - c
        pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
        paeth = np.select([(pa <= pb) & (pa <= pc), pb <= pc], [a, b], c)
        costs = []
        for pred in (0, a, b, (a + b) // 2, paeth):
            v = (x - pred) % 256
            costs.append(int(np.where(v >= 128, 256 - v, v).sum()))
        types.append(costs.index(min(costs)))
    return types


@pytest.mark.parametrize("name", sorted(CASES))
def test_model_decodes_to_the_input(name):
    img = CASES[name]
    info = {}
    png = M.encode(img, info)
    ch = chunks(png)
    kinds = [k for k, _ in ch]
    nseg = len(info["kinds"])
    assert kinds == [b"IHDR", b"IDAT"] + [b"IDAT"] * nseg + [b"IDAT", b"IEND"]
    assert ch[0][1] == struct.pack(">IIBBBBB", img.shape[1], img.shape[0], 8, 2, 0, 0, 0)
    assert ch[1][1] == b"\x78\x01" and len(ch[-2][1]) == 4
    stream = b"".join(d for _, d in ch[1:-1])
    raw = zlib.decompress(stream)
    assert raw == info["filtered"].tobytes()
    assert len(raw) == img.shape[0] * (1 + 3 * img.shape[1])
    assert np.array_equal(np.array(Image.open(io.BytesIO(png)).convert("RGB")), img)
    # every segment decodes on its own (no match reaches back past its first byte)
    for k, (_, data) in enumerate(ch[2:-2]):
        d = zlib.decompressobj(-15)
        seg = d.decompress(data)
        assert seg == raw[k * M.SEG:(k + 1) * M.SEG]


@pytest.mark.parametrize("name", sorted(CASES))
def test_filter_bytes_are_the_heuristics_choice(name):
    img = CASES[name]
    F, types = M.filter_rows(img)
    assert types.tolist() == heuristic_types(img)
    assert F.reshape(img.shape[0], -1)[:, 0].tolist() == types.tolist()


def test_every_filter_type_wins_and_ties_go_to_the_lower_type():
    img = CASES["filters"]
    _, types = M.filter_rows(img)
    assert set(types.tolist()) == {0, 1, 2, 3, 4}
    assert [int(types[y]) for y in range(1, 15)] == [y % 5 for y in range(1, 15)]
    assert types[15] == 0  # all five cost 0
    assert types[17] == 2  # up and Paeth cost 0
    assert types[19] == 2  # a copy of the row above


def test_segment_edges():
    for name, k, plus in (("F_1x65536", 1, 0), ("F_2x65536", 2, 0), ("F_3x65536_plus_1", 3, 1)):
        info = {}
        M.encode(CASES[name], info)
        assert len(info["filtered"]) == k * M.SEG + plus
        assert len(info["kinds"]) == k + (1 if plus else 0)
    assert len(M.filter_rows(CASES["wide_30000"])[0]) > 4 * M.SEG  # a row longer than a segment
    info = {}
    M.encode(CASES["noise"], info)
    assert set(info["kinds"]) == {"stored"}
    info = {}
    M.encode(CASES["constant"], info)  # 258-runs that reach segment ends
    assert len(info["kinds"]) > 1 and set(info["kinds"]) == {"dynamic"}


def test_runs_are_cut_as_zlib_rle_cuts_them():
    seg = np.array([5] * 1 + [6] * 2 + [7] * 3 + [8] * 4 + [9] * 5 + [1] * 260 + [2] * 262 + [3] * 519, np.uint8)
    sym, xval, _, is_match = M.tokens(seg)
    lens = [int(M.LEN_BASE[s - 257] + x) if m else None for s, x, m in zip(sym.tolist(), xval.tolist(), is_match)]
    # runs of 1, 2, 3: literals; 4, 5: literal + match of 3, 4; 260 = 1 + 258 + 1; 262 = 1 + 258 + 3;
    # 519 = 1 + 2 * 258 + 2
    assert lens == ([None] + [None] * 2 + [None] * 3 + [None, 3] + [None, 4] + [None, 258, None] +
                    [None, 258, 3] + [None, 258, 258, None, None])


def test_length_limits_are_needed_and_kept():
    hist, _ = M.segment_histograms(M.filter_rows(CASES["limit15"])[0][:M.SEG])
    assert M.huffman_depth(hist) > 15 and M.package_merge(hist, 15).max() == 15
    _, clhist = M.segment_histograms(M.filter_rows(CASES["limit7"])[0][:M.SEG])
    assert M.huffman_depth(clhist) > 7 and M.package_merge(clhist, 7).max() == 7


def test_one_used_code_length_symbol_gets_a_partner():
    """The rule for a code-length code of one used symbol: the lowest other symbol also gets length 1, which makes
    the code complete.  The rule is defensive.  One code-length symbol cannot describe a valid block: all zeros has
    no end-of-block, and 257 or more equal non-zero lengths are over- or under-subscribed.  So no segment uses fewer
    than two symbols, which is checked here on the first segments of every case."""
    for u in (0, 8, 18):
        h = np.zeros(19, np.int64)
        h[u] = 5
        cll = M.cl_code_lengths(h)
        assert cll[u] == 1 and cll[1 if u == 0 else 0] == 1 and cll.sum() == 2
    for img in CASES.values():
        F = M.filter_rows(img)[0]
        for a0 in range(0, min(len(F), 4 * M.SEG), M.SEG):
            _, clhist = M.segment_histograms(F[a0:a0 + M.SEG])
            assert np.count_nonzero(clhist) >= 2


def test_package_merge_is_optimal_when_the_limit_does_not_bind():
    rng = np.random.default_rng(2)
    for _ in range(20):
        f = rng.integers(0, 50, 40)
        f[:2] += 1
        lens = M.package_merge(f, 15)
        assert sum(2.0 ** -l for l in lens[lens > 0]) == 1.0  # complete
        # same total cost as an unlimited Huffman code
        import heapq
        h = [int(x) for x in f if x]
        heapq.heapify(h)
        cost = 0
        while len(h) > 1:
            a, b = heapq.heappop(h), heapq.heappop(h)
            cost += a + b
            heapq.heappush(h, a + b)
        assert int((f * lens).sum()) == cost


def zlib_rle(F: bytes) -> int:
    c = zlib.compressobj(6, zlib.DEFLATED, 15, 9, zlib.Z_RLE)
    return len(c.compress(F) + c.flush())


@pytest.mark.parametrize("name", ["scene_main", "scene_realm"])
def test_size_close_to_zlib_rle_on_renders(name):
    info = {}
    png = M.encode(CASES[name], info)
    zdata = sum(len(d) for _, d in chunks(png)[1:-1])
    assert zdata <= 1.02 * zlib_rle(info["filtered"].tobytes()) + 64


def test_smooth_image_compresses_tenfold():
    img = CASES["smooth"]
    assert len(M.encode(img)) < M.stored_bound(img.shape[1], img.shape[0]) / 10


def test_stored_bound_is_the_host_writers_size_plus_chunk_overhead():
    for W, H in ((1, 1), (85, 256), (400, 225), (30000, 3)):
        N = H * (1 + 3 * W)
        nseg = -(-N // M.SEG)
        assert M.stored_bound(W, H) == 8 + 25 + 14 + 16 + 12 + 12 * nseg + N + 5 * sum(
            -(-min(M.SEG, N - i * M.SEG) // 65535) for i in range(nseg))


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


@needs_lib
def test_sizing_calls_need_no_gpu():
    lib = C.CDLL(LIB)
    n = C.c_size_t()
    lib.rtclj_encode_png_gpu.argtypes = [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t,
                                         C.POINTER(C.c_size_t)]
    assert lib.rtclj_encode_png_gpu(0, None, 400, 225, None, 0, C.byref(n)) == 0
    assert n.value == M.stored_bound(400, 225)
    assert lib.rtclj_encode_png_gpu(0, None, 0, 225, None, 0, C.byref(n)) == 1
    assert lib.rtclj_encode_png_gpu(0, None, 400, -1, None, 0, C.byref(n)) == 1
    assert lib.rtclj_encode_png_gpu(0, None, 400, 225, None, 0, None) == 1


@needs_lib
@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not installed")
def test_png_kernels_use_no_local_memory():
    out = subprocess.run(["cuobjdump", "-sass", LIB], check=True, capture_output=True, text=True).stdout
    bodies = {}
    for part in re.split(r"\n\s*Function : ", out)[1:]:
        name = part.split("\n", 1)[0].strip()
        bodies[name] = part
    for k in ("png_filter_kernel", "png_deflate_kernel", "png_place_kernel"):
        found = [b for n, b in bodies.items() if k in n]
        assert len(found) == 1, k
        assert not re.search(r"\b(LDL|STL)\b", found[0]), k


def test_clojure_shim_binds_the_new_calls():
    text = open(os.path.join(ROOT, "integration", "clojure", "src", "rtclj", "native.clj")).read()
    for name in ("rtclj_render_multi_png", "rtclj_encode_png_gpu"):
        assert '"%s"' % name in text
