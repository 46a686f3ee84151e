"""numpy model of the device PNG encoder (include/rtclj_b200.h, rtclj_encode_png_gpu; DESIGN.md section 4.11).

It produces the exact bytes the device writes, operation by operation:
  chunks     signature, IHDR, IDAT(78 01), one IDAT per 64 KiB segment, IDAT(Adler-32), IEND
  filtering  per row the PNG filter (bpp 3, a = b = c = 0 outside the image) of least sum |byte as int8|;
             a tie goes to the lower type
  segments   the filtered stream F cut at multiples of 65 536 bytes, each encoded on its own
  tokens     a maximal run of L equal bytes at s: literal at s, (L-1)//258 matches (258, distance 1), then
             the remainder q as one match when q >= 3, else q literals
  block      one dynamic block per segment: package-merge lengths (15 bits lit/len, 7 bits code-length code;
             items by (frequency, symbol), leaves before packages at equal weight), distance code {0: 1, 1: 1},
             HLIT >= 257, the code-length sequence run-length coded greedily, HCLEN trimmed to >= 4
  fallback   stored blocks of <= 65 535 bytes when the dynamic block, flush included, is not shorter
  end        a dynamic segment but the last is followed by a sync flush (000, pad, 00 00 FF FF); the last
             block has BFINAL = 1 and is padded to the byte
Vectorised with numpy so that a 4K image is modelled in seconds."""
from __future__ import annotations

import struct
import zlib

import numpy as np

SEG = 65536
SIG = b"\x89PNG\r\n\x1a\n"
LEN_BASE = np.array([3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131,
                     163, 195, 227, 258], dtype=np.int64)
LEN_EXTRA = np.array([0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0], dtype=np.int64)
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]

# match length (3..258) -> symbol index 0..28 (symbol 257 + index)
_LSYM = np.zeros(259, dtype=np.int64)
for _i in range(29):
    _LSYM[LEN_BASE[_i]:] = _i
_LSYM[258] = 28


def _paeth(a, b, c):
    p = a + b - c
    pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
    return np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c))


def filter_rows(rgb8: np.ndarray):
    """(F as uint8 [H * (1 + 3W)], filter type per row)."""
    img = np.ascontiguousarray(rgb8, dtype=np.uint8)
    H, W, _ = img.shape
    rows = img.reshape(H, 3 * W)
    out = np.empty((H, 1 + 3 * W), dtype=np.uint8)
    types = np.empty(H, dtype=np.uint8)
    step = max(1, (1 << 22) // (3 * W))
    for r0 in range(0, H, step):
        r1 = min(H, r0 + step)
        x = rows[r0:r1].astype(np.int16)
        b = rows[r0 - 1:r1 - 1].astype(np.int16) if r0 > 0 else np.vstack(
            [np.zeros((1, 3 * W), np.int16), rows[0:r1 - 1].astype(np.int16)])
        a = np.zeros_like(x)
        a[:, 3:] = x[:, :-3]
        c = np.zeros_like(b)
        c[:, 3:] = b[:, :-3]
        cand = np.stack([x, x - a, x - b, x - ((a + b) >> 1), x - _paeth(a, b, c)]).astype(np.uint8)
        cost = np.abs(cand.view(np.int8).astype(np.int32)).sum(axis=2)  # [5, rows]
        t = np.argmin(cost, axis=0)  # the first minimum: the lower type on a tie
        types[r0:r1] = t
        out[r0:r1, 0] = t
        out[r0:r1, 1:] = cand[t, np.arange(r1 - r0)]
    return out.reshape(-1), types


def package_merge(freq: np.ndarray, limit: int) -> np.ndarray:
    """Length-limited Huffman code lengths (boundary-free package-merge), >= 2 used symbols."""
    used = np.flatnonzero(freq)
    n = len(used)
    lens = np.zeros(len(freq), dtype=np.int64)
    order = used[np.lexsort((used, freq[used]))]  # by (frequency, symbol)
    leafw = freq[order].astype(np.int64)
    cur = leafw.copy()
    leafbits = []  # per level (deepest first): which merged positions hold leaves
    bits = np.zeros(n, dtype=bool)
    bits[:] = True
    leafbits.append(bits)
    for _ in range(limit - 1):
        npk = len(cur) // 2
        pkg = cur[0:2 * npk:2] + cur[1:2 * npk:2]
        lpos = np.arange(n) + np.searchsorted(pkg, leafw, side="left")    # packages strictly lighter come first
        ppos = np.arange(npk) + np.searchsorted(leafw, pkg, side="right")  # leaves of equal weight come first
        nxt = np.empty(n + npk, dtype=np.int64)
        nxt[lpos] = leafw
        nxt[ppos] = pkg
        bits = np.zeros(n + npk, dtype=bool)
        bits[lpos] = True
        leafbits.append(bits)
        cur = nxt
    m = 2 * n - 2
    counts = []
    for bits in reversed(leafbits):  # level 1 (the last built) down to the deepest
        c = int(bits[:m].sum())
        counts.append(c)
        m = 2 * (m - c)
    ln = np.zeros(n, dtype=np.int64)
    for c in counts:
        ln[:c] += 1
    lens[order] = ln
    return lens


def canonical_rev(lens: np.ndarray) -> np.ndarray:
    """Canonical codes (RFC 1951 3.2.2), bit-reversed for LSB-first packing."""
    maxl = int(lens.max())
    bl = np.bincount(lens, minlength=maxl + 1)
    bl[0] = 0
    nxt = [0] * (maxl + 2)
    code = 0
    for b in range(1, maxl + 1):
        code = (code + int(bl[b - 1])) << 1
        nxt[b] = code
    rev = np.zeros(len(lens), dtype=np.int64)
    for s, l in enumerate(lens.tolist()):
        if l:
            c = nxt[l]
            nxt[l] += 1
            rev[s] = int(format(c, f"0{l}b")[::-1], 2)
    return rev


def rle_lengths(seq):
    """The code-length sequence as (symbol, extra value, extra bits)."""
    out = []
    i, N = 0, len(seq)
    while i < N:
        v = seq[i]
        run = 1
        while i + run < N and seq[i + run] == v:
            run += 1
        i += run
        if v == 0:
            while run >= 11:
                k = min(run, 138)
                out.append((18, k - 11, 7))
                run -= k
            if run >= 3:
                out.append((17, run - 3, 3))
                run = 0
            out.extend([(0, 0, 0)] * run)
        else:
            out.append((v, 0, 0))
            run -= 1
            while run >= 3:
                k = min(run, 6)
                out.append((16, k - 3, 2))
                run -= k
            out.extend([(v, 0, 0)] * run)
    return out


def _pack(vals: np.ndarray, nbits: np.ndarray) -> bytes:
    """LSB-first bit packing of the fields (vals[i] in nbits[i] bits), padded to the byte."""
    keep = nbits > 0
    vals, nbits = vals[keep].astype(np.int64), nbits[keep].astype(np.int64)
    total = int(nbits.sum())
    starts = np.cumsum(nbits) - nbits
    idx = np.arange(total, dtype=np.int64) - np.repeat(starts, nbits)
    bits = ((np.repeat(vals, nbits) >> idx) & 1).astype(np.uint8)
    return np.packbits(bits, bitorder="little").tobytes()


def tokens(seg: np.ndarray):
    """(symbol, extra value, extra bits, is-match) per token of one segment, in stream order."""
    n = len(seg)
    starts = np.flatnonzero(np.concatenate([[True], seg[1:] != seg[:-1]]))
    L = np.diff(np.append(starts, n))
    full, q = (L - 1) // 258, (L - 1) % 258
    per = 1 + full + np.where(q >= 3, 1, q)
    first = np.cumsum(per) - per
    r = np.repeat(np.arange(len(starts)), per)
    k = np.arange(int(per.sum())) - first[r]
    byte = seg[starts].astype(np.int64)[r]
    fr, qr = full[r], q[r]
    is_match = (k >= 1) & ((k <= fr) | ((k == fr + 1) & (qr >= 3)))
    mlen = np.where(k <= fr, 258, qr)
    li = _LSYM[np.where(is_match, mlen, 3)]
    sym = np.where(is_match, 257 + li, byte)
    xbits = np.where(is_match, LEN_EXTRA[li], 0)
    xval = np.where(is_match, mlen - LEN_BASE[li], 0)
    return sym, xval, xbits, is_match


def stored_bytes(n: int) -> int:
    return n + 5 * ((n + 65534) // 65535)


def cl_code_lengths(clhist: np.ndarray) -> np.ndarray:
    """The code-length code: package-merge limited to 7 bits; with one used symbol the lowest other symbol gets
    length 1 as well (zlib's inflate rejects an incomplete code-length code)."""
    if np.count_nonzero(clhist) == 1:
        cll = np.zeros(19, dtype=np.int64)
        u = int(np.flatnonzero(clhist)[0])
        cll[u] = 1
        cll[1 if u == 0 else 0] = 1
        return cll
    return package_merge(clhist, 7)


def encode_segment(seg: np.ndarray, last: bool):
    """(bytes of the segment's deflate data, 'dynamic' | 'stored')."""
    n = len(seg)
    sym, xval, xbits, is_match = tokens(seg)
    hist = np.bincount(sym, minlength=286)
    hist[256] += 1
    ll = package_merge(hist, 15)
    hlit = max(257, int(np.flatnonzero(ll).max()) + 1)
    seq = ll[:hlit].tolist() + [1, 1]
    cl = rle_lengths(seq)
    clsym = np.array([c[0] for c in cl], dtype=np.int64)
    clhist = np.bincount(clsym, minlength=19)
    cll = cl_code_lengths(clhist)
    hclen = 19
    while hclen > 4 and cll[CL_ORDER[hclen - 1]] == 0:
        hclen -= 1
    llrev, clrev = canonical_rev(ll), canonical_rev(cll)
    head_v = [1 if last else 0, 2, hlit - 257, 1, hclen - 4] + [int(cll[CL_ORDER[i]]) for i in range(hclen)]
    head_n = [1, 2, 5, 5, 4] + [3] * hclen
    for s, xv, xn in cl:
        head_v += [int(clrev[s]), xv]
        head_n += [int(cll[s]), xn]
    T = len(sym)
    vals = np.empty(3 * T, dtype=np.int64)
    nb = np.empty(3 * T, dtype=np.int64)
    vals[0::3], nb[0::3] = llrev[sym], ll[sym]
    vals[1::3], nb[1::3] = xval, xbits
    vals[2::3], nb[2::3] = 0, is_match.astype(np.int64)  # distance code 0 (distance 1): one 0 bit
    bits = int(np.sum(head_n)) + int(nb.sum()) + int(ll[256])
    dyn = (bits + 7) // 8 if last else (bits + 3 + 7) // 8 + 4
    if dyn >= stored_bytes(n):
        out = bytearray()
        for b0 in range(0, n, 65535):
            m = min(65535, n - b0)
            out += bytes([1 if last and b0 + m == n else 0]) + struct.pack("<HH", m, m ^ 0xFFFF)
            out += seg[b0:b0 + m].tobytes()
        return bytes(out), "stored"
    v = np.concatenate([np.array(head_v, np.int64), vals, [int(llrev[256])]])
    w = np.concatenate([np.array(head_n, np.int64), nb, [int(ll[256])]])
    if last:
        data = _pack(v, w)
    else:  # sync flush: an empty stored block (000, pad to the byte, 00 00 FF FF)
        data = _pack(np.append(v, 0), np.append(w, 3)) + b"\x00\x00\xff\xff"
    assert len(data) == dyn, (len(data), dyn)
    return data, "dynamic"


def _chunk(kind: bytes, data: bytes) -> bytes:
    return struct.pack(">I", len(data)) + kind + data + struct.pack(">I", zlib.crc32(kind + data) & 0xFFFFFFFF)


def encode(rgb8: np.ndarray, info: dict | None = None) -> bytes:
    img = np.ascontiguousarray(rgb8, dtype=np.uint8)
    H, W, _ = img.shape
    F, types = filter_rows(img)
    out = [SIG, _chunk(b"IHDR", struct.pack(">IIBBBBB", W, H, 8, 2, 0, 0, 0)), _chunk(b"IDAT", b"\x78\x01")]
    kinds = []
    N = len(F)
    for a in range(0, N, SEG):
        data, kind = encode_segment(F[a:a + SEG], a + SEG >= N)
        kinds.append(kind)
        out.append(_chunk(b"IDAT", data))
    out.append(_chunk(b"IDAT", struct.pack(">I", zlib.adler32(F.tobytes()) & 0xFFFFFFFF)))
    out.append(_chunk(b"IEND", b""))
    if info is not None:
        info.update(filtered=F, types=types, kinds=kinds)
    return b"".join(out)


def stored_bound(width: int, height: int) -> int:
    """The sizing call's answer: every segment stored."""
    N = height * (1 + 3 * width)
    nseg = (N + SEG - 1) // SEG
    body = sum(12 + stored_bytes(min(SEG, N - i * SEG)) for i in range(nseg))
    return 8 + 25 + 14 + body + 16 + 12


# ---- the inputs the CPU and GPU tests share

def huffman_depth(freq) -> int:
    """Depth of an unlimited Huffman code of freq (to show that a case needs the length limit)."""
    import heapq
    heap = [(int(f), i) for i, f in enumerate(freq) if f]
    groups = {i: [i] for _, i in heap}
    depth = {i: 0 for _, i in heap}
    heapq.heapify(heap)
    nxt = len(freq)
    while len(heap) > 1:
        (fa, a), (fb, b) = heapq.heappop(heap), heapq.heappop(heap)
        g = groups.pop(a) + groups.pop(b)
        for s in g:
            depth[s] += 1
        groups[nxt] = g
        heapq.heappush(heap, (fa + fb, nxt))
        nxt += 1
    return max(depth.values())


def segment_histograms(seg: np.ndarray):
    """(lit/len histogram, code-length histogram) of one segment."""
    sym = tokens(seg)[0]
    hist = np.bincount(sym, minlength=286)
    hist[256] += 1
    ll = package_merge(hist, 15)
    hlit = max(257, int(np.flatnonzero(ll).max()) + 1)
    cl = rle_lengths(ll[:hlit].tolist() + [1, 1])
    return hist, np.bincount([c[0] for c in cl], minlength=19)


def image_limit15() -> np.ndarray:
    """One row whose literals have Fibonacci counts: an unlimited Huffman code would be 16 bits deep."""
    fib = [1, 1]
    while len(fib) < 23:
        fib.append(fib[-1] + fib[-2])
    vals = [0] + [x for k in range(1, 40) for x in (k, 256 - k)]
    seq = np.concatenate([np.full(fib[22 - i], vals[i], np.uint8) for i in range(23)])
    np.random.default_rng(1).shuffle(seq)
    return seq[: len(seq) // 3 * 3].reshape(1, -1, 3)


def image_limit7() -> np.ndarray:
    """One row of geometric-distributed bytes whose code-length code would be 8 bits deep unlimited."""
    rng = np.random.default_rng(1)
    r, k = rng.uniform(0.80, 0.97), rng.integers(40, 256)
    p = np.zeros(256)
    p[rng.permutation(256)[:k]] = r ** np.arange(k)
    p /= p.sum()
    return rng.choice(256, size=3 * 20000, p=p).astype(np.uint8).reshape(1, -1, 3)


def image_filters() -> np.ndarray:
    """Rows built so that each filter type wins somewhere, plus rows where filters tie: a small residual through
    filter t on noise (t = row % 5), then a zero row (all five tie: 0 wins), a constant row over a constant row
    (up and Paeth tie at cost 0: 2 wins), and a copy of the row above (up wins)."""
    rng = np.random.default_rng(5)
    W, H = 64, 24
    img = np.zeros((H, W, 3), dtype=np.uint8)
    img[0] = rng.integers(0, 256, (W, 3))
    for y in range(1, 15):
        t = y % 5
        prev = img[y - 1].reshape(-1).astype(np.int64)
        row = np.zeros(3 * W, dtype=np.int64)
        res = rng.integers(-2, 3, 3 * W)
        for x in range(3 * W):
            a = row[x - 3] if x >= 3 else 0
            b = prev[x]
            c = prev[x - 3] if x >= 3 else 0
            pred = [0, a, b, (a + b) >> 1, int(_paeth(np.int64(a), np.int64(b), np.int64(c)))][t]
            row[x] = (pred + res[x]) & 255 if t else rng.integers(0, 3) * (1 if x % 2 else -1) & 255
        img[y] = row.reshape(W, 3)
    img[15] = 0
    img[16] = 77
    img[17] = 77
    img[18] = img[14]
    img[19] = img[18]
    img[20:] = rng.integers(0, 256, (H - 20, W, 3))
    return img


def smooth_image(W: int = 960, H: int = 540) -> np.ndarray:
    """The kind of image -i renders: a sky gradient and normal-shaded spheres."""
    y, x = np.mgrid[0:H, 0:W].astype(np.float64)
    t = 0.5 * (1.0 - y / H)
    sky = np.stack([(1 - t) + 0.5 * t, (1 - t) + 0.7 * t, np.ones_like(t)], axis=2)
    img = sky
    for cx, cy, r in ((0.5, 0.55, 0.22), (0.2, 0.7, 0.12), (0.8, 0.65, 0.15)):
        dx, dy = (x / W - cx) * W / H, (y / H - cy)
        d2 = dx * dx + dy * dy
        inside = d2 < r * r
        nz = np.sqrt(np.clip(r * r - d2, 0, None)) / r
        n = np.stack([dx / r, -dy / r, nz], axis=2)
        img = np.where(inside[:, :, None], 0.5 * (n + 1.0), img)
    return (255.999 * np.clip(img, 0, 1)).astype(np.uint8)


def cpu_cases():
    """name -> image: every input the model is checked on, and the device against the model."""
    import os
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_images.npz"))
    rng = np.random.default_rng(11)
    return {
        "scene_main": gold["scene_main"],
        "scene_realm": gold["scene_realm"],
        "noise": rng.integers(0, 256, (250, 300, 3), dtype=np.uint8),
        "constant": np.full((300, 400, 3), 77, dtype=np.uint8),
        "1x1": np.array([[[1, 2, 3]]], dtype=np.uint8),
        "1xN": rng.integers(0, 4, (1, 5000, 3), dtype=np.uint8),
        "Nx1": rng.integers(0, 4, (5000, 1, 3), dtype=np.uint8),
        "wide_30000": (np.arange(3 * 30000 * 3) // 7 % 256).astype(np.uint8).reshape(3, 30000, 3),
        "F_1x65536": (rng.integers(0, 2, (256, 85, 3)) * 40).astype(np.uint8),
        "F_2x65536": (rng.integers(0, 2, (512, 85, 3)) * 40).astype(np.uint8),
        "F_3x65536_plus_1": (np.arange(65536 * 3) % 251).astype(np.uint8).reshape(1, 65536, 3),
        "filters": image_filters(),
        "limit15": image_limit15(),
        "limit7": image_limit7(),
        "smooth": smooth_image(),
    }
