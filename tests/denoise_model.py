"""numpy model of the denoiser's definition (include/rtclj_b200.h, DESIGN.md section 4.13): the exact float32
operations of rtclj_ctx_denoise, vectorised over pixels and sequential over the 25 taps, so that the device output
can be compared bit for bit.  Every constant is a np.float32 (NEP 50 keeps the arithmetic in float32) and the clamp
is np.fmax, whose NaN rule is fmaxf's."""
from __future__ import annotations

import numpy as np

F32 = np.float32
H5 = np.array([1.0 / 16, 1.0 / 4, 3.0 / 8, 1.0 / 4, 1.0 / 16], dtype=np.float32)
ONE, ZERO = F32(1.0), F32(0.0)
FLT_MIN = np.finfo(np.float32).tiny


def check(width: int, height: int, levels: int, sigma_color: float, sigma_guide: float):
    """None when the library accepts the arguments, else the reason it refuses them (RTCLJ_E_INVALID)."""
    if width <= 0 or height <= 0:
        return "size"
    if not 1 <= levels <= 8:
        return "levels"
    for s in (sigma_color, sigma_guide):
        if not (np.isfinite(s) and s > 0):
            return "sigma"
    with np.errstate(all="ignore"):
        c, g = F32(sigma_color), F32(sigma_guide)
        last = c * F32(2.0 ** -(levels - 1))
        if not np.isfinite(c * c) or not last * last >= FLT_MIN:
            return "sigma_color"
        if not np.isfinite(g * g) or not g * g >= FLT_MIN:
            return "sigma_guide"
    return None


def sigma2(sigma: float, level: int) -> np.float32:
    s = F32(sigma) * F32(2.0 ** -level)
    return s * s


def k(x):
    t = np.fmax(ONE - x, ZERO)
    return t * t


def _finite(img):
    return np.isfinite(img).all(axis=-1)


def _shift(img, sy, sx):
    """img[y + sy, x + sx] at (y, x); NaN where that lies outside the image (so the tap is skipped)."""
    H, W = img.shape[:2]
    out = np.full(img.shape, np.nan, dtype=img.dtype)
    y0, y1 = max(0, -sy), min(H, H - sy)
    x0, x1 = max(0, -sx), min(W, W - sx)
    if y0 < y1 and x0 < x1:
        out[y0:y1, x0:x1] = img[y0 + sy:y1 + sy, x0 + sx:x1 + sx]
    return out


def sqdist(a, b):
    d = a - b
    return (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]


def level(c, g, step: int, sc2, sg2):
    """c_(i+1) from c_i (float32 [H,W,3]) with guide g."""
    ok = _finite(c) & _finite(g)
    acc = np.zeros(c.shape, dtype=np.float32)
    wsum = np.zeros(c.shape[:2], dtype=np.float32)
    for dy in range(-2, 3):
        for dx in range(-2, 3):
            cq, gq = _shift(c, step * dy, step * dx), _shift(g, step * dy, step * dx)
            tap = ok & _finite(cq) & _finite(gq)
            w = ((H5[dx + 2] * H5[dy + 2]) * k(sqdist(cq, c) / sc2)) * k(sqdist(gq, g) / sg2)
            acc = np.where(tap[..., None], acc + w[..., None] * cq, acc)
            wsum = np.where(tap, wsum + w, wsum)
    return np.where(ok[..., None], acc / wsum[..., None], c)


def quantise(lin, linear: bool):
    """write-color! as the device computes it: (unsigned char)(int)v, the int conversion saturating, NaN -> 0."""
    with np.errstate(all="ignore"):
        if linear:
            v = 255.999 * lin
        else:
            gm = np.where(lin > 0.0, np.sqrt(np.where(lin > 0.0, lin, 0.0)), 0.0)
            v = 256.0 * np.where(gm < 0.999, gm, 0.999)
        v = np.where(np.isnan(v), 0.0, np.clip(np.trunc(v), -2.0 ** 31, 2.0 ** 31 - 1))
    return (v.astype(np.int64) & 0xFF).astype(np.uint8)


def denoise(C, G, levels: int, sigma_color: float, sigma_guide: float, flags: int = 0):
    """(linear float64 [H,W,3], rgb8 uint8 [H,W,3]) of the definition; flags: only RTCLJ_F_QUANT_LINEAR (32)."""
    C = np.asarray(C, dtype=np.float64)
    G = np.asarray(G, dtype=np.float64)
    assert check(C.shape[1], C.shape[0], levels, sigma_color, sigma_guide) is None
    with np.errstate(all="ignore"):
        c, g = C.astype(np.float32), G.astype(np.float32)
        filtered = _finite(c) & _finite(g)
        sg2 = F32(sigma_guide) * F32(sigma_guide)
        for i in range(levels):
            c = level(c, g, 1 << i, sigma2(sigma_color, i), sg2)
    lin = np.where(filtered[..., None], c.astype(np.float64), C)
    return lin, quantise(lin, bool(flags & 32))


def denoise_scalar(C, G, levels: int, sigma_color: float, sigma_guide: float):
    """The same definition as a per-pixel loop over Python floats rounded through np.float32 at every operation:
    an independent check of the vectorised model on small images."""
    H, W, _ = C.shape
    f = np.float32
    with np.errstate(over="ignore"):
        c = [[[f(C[y, x, ch]) for ch in range(3)] for x in range(W)] for y in range(H)]
        g = [[[f(G[y, x, ch]) for ch in range(3)] for x in range(W)] for y in range(H)]
    fin = lambda v: all(np.isfinite(t) for t in v)  # noqa: E731
    h = [f(1.0 / 16), f(0.25), f(0.375), f(0.25), f(1.0 / 16)]

    def kk(x):
        t = f(1.0) - x
        t = t if t > f(0.0) else f(0.0)  # fmax: a NaN t gives 0
        return t * t

    def d2(a, b):
        r, gg, bb = a[0] - b[0], a[1] - b[1], a[2] - b[2]
        return (r * r + gg * gg) + bb * bb

    base = [[fin(c[y][x]) and fin(g[y][x]) for x in range(W)] for y in range(H)]
    with np.errstate(all="ignore"):
        sg2 = f(sigma_guide) * f(sigma_guide)
        for i in range(levels):
            s = 1 << i
            sc = f(sigma_color) * f(2.0 ** -i)
            sc2 = sc * sc
            nxt = [[list(c[y][x]) for x in range(W)] for y in range(H)]
            for y in range(H):
                for x in range(W):
                    if not (fin(c[y][x]) and fin(g[y][x])):
                        continue
                    acc, wsum = [f(0.0)] * 3, f(0.0)
                    for dy in range(-2, 3):
                        for dx in range(-2, 3):
                            qy, qx = y + s * dy, x + s * dx
                            if not (0 <= qy < H and 0 <= qx < W) or not (fin(c[qy][qx]) and fin(g[qy][qx])):
                                continue
                            w = ((h[dx + 2] * h[dy + 2]) * kk(d2(c[qy][qx], c[y][x]) / sc2)) * kk(d2(g[qy][qx], g[y][x]) / sg2)
                            acc = [acc[ch] + w * c[qy][qx][ch] for ch in range(3)]
                            wsum = wsum + w
                    nxt[y][x] = [acc[ch] / wsum for ch in range(3)]
            c = nxt
    out = np.array(C, dtype=np.float64, copy=True)
    for y in range(H):
        for x in range(W):
            if base[y][x]:
                out[y, x] = [float(v) for v in c[y][x]]
    return out
