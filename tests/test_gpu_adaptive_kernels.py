"""The adaptive-sampling kernels of rtclj_adaptive.cuh on their own, through tests/native/adaptive_kernels.cu,
against numpy: the compaction at sizes whose scan takes several rounds of 1024 tiles, unit_stderr bit for bit and
against an exact reference, and finalize_adaptive_kernel on synthetic sums for every fold it does.  These reach
orders and edges that whole renders cannot see: the order of the list within a tile only changes which lane
traces which pixel, not any value."""
import math
import zlib
from decimal import Decimal, getcontext
from fractions import Fraction

import numpy as np
import pytest

import adaptive_kernels as K
import oracle_lib as O
from raytracing_clj_b200 import render

pytestmark = pytest.mark.gpu
EPS = 2.0 ** -53
TILE = 2048  # kListTile


def cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda:0")


# ---------------------------------------------------------------- compaction

SIZES = [1, 7, 2047, 2048, 2049, 2048 * 1024 - 1, 2048 * 1024, 2048 * 1024 + 1, 3 * 2 ** 21 + 5, 3840 * 2160]
PATTERNS = ["all", "none", "first", "last", "tile-ends", "half", "sparse"]


def live_pattern(n, pattern):
    live = np.zeros(n, dtype=np.uint8)
    if pattern == "all":
        live[:] = 1
    elif pattern == "first":
        live[0] = 1
    elif pattern == "last":
        live[-1] = 1
    elif pattern == "tile-ends":
        # the first and the last position of every tile of the descending order (position s is pixel n - 1 - s)
        starts = np.arange(0, n, TILE)
        ends = np.minimum(starts + TILE, n) - 1
        live[n - 1 - starts] = 1
        live[n - 1 - ends] = 1
    elif pattern in ("half", "sparse"):
        rng = np.random.default_rng(n)
        live[:] = rng.random(n) < (0.5 if pattern == "half" else 0.001)
    return live


def test_tile_size_is_the_one_the_sizes_were_chosen_for():
    assert K.list_tile() == TILE


@pytest.mark.parametrize("n", SIZES)
def test_compaction_lists_the_live_pixels_in_descending_order(n):
    """The list equals np.flatnonzero(live)[::-1] and the count is exact.  Above 1024 tiles (2^21 pixels) the scan
    of the tile counts takes more than one round and carries the sum of the earlier rounds."""
    for pattern in PATTERNS:
        live = live_pattern(n, pattern)
        got, count = K.relist(cuda(live))
        want = np.flatnonzero(live)[::-1].astype(np.uint32)
        assert count == len(want), (n, pattern, count, len(want))
        assert np.array_equal(got, want), (n, pattern, np.flatnonzero(got != want)[:5])


# ---------------------------------------------------------------- unit_stderr


def np_unit_stderr(s1, s2, n, u):
    """The header's operations in the header's order."""
    m = ((n + u - 1) // u).astype(np.float64)
    with np.errstate(all="ignore"):
        q = s1 * s1
        q = q / m
        v = s2 - q
        v = v / (m * (m - 1.0))
        v = v / (float(u) * float(u))
        v = np.fmax(v, 0.0)
        return np.sqrt(v)


def np_overflow(s1, s2):
    with np.errstate(all="ignore"):
        return ~(np.isfinite(s1 * s1) & np.isfinite(s2))


def device_stderr(s1, s2, n, u):
    s1, s2, n = (np.asarray(x) for x in (s1, s2, n))
    return K.unit_stderr(cuda(s1.astype(np.float64)), cuda(s2.astype(np.float64)), cuda(n.astype(np.int32)), u)


def moments(rng, count, u):
    """Moments of m >= 2 units of random unit sums, as the fold forms them, and their counts."""
    n = rng.integers(2 * u, 64 * u, size=count)
    s1, s2 = np.zeros(count), np.zeros(count)
    m = (n + u - 1) // u
    scale = 10.0 ** rng.uniform(-6, 6, size=count)
    for k in range(int(m.max())):
        x = rng.normal(rng.normal(size=count), 1.0, size=count) * scale
        x = np.where(k < m, x, 0.0)
        s1, s2 = s1 + x, s2 + x * x
    return s1, s2, n


@pytest.mark.parametrize("u", [1, 4, 7, 64])
def test_unit_stderr_is_the_headers_arithmetic_bit_for_bit(u):
    rng = np.random.default_rng(u)
    s1, s2, n = moments(rng, 4096, u)
    got, ovf = device_stderr(s1, s2, n, u)
    want = np_unit_stderr(s1, s2, n, u)
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
    assert not ovf.any()


def exact_stderr(s1, s2, n, u):
    """sqrt(max((S2 - S1^2/m) / (m (m-1) u^2), 0)) of the double inputs, exactly (the root at 50 digits)."""
    m = (n + u - 1) // u
    v = (Fraction(s2) - Fraction(s1) ** 2 / m) / (m * (m - 1) * u * u)
    v = max(v, Fraction(0))
    getcontext().prec = 50
    return (Decimal(v.numerator) / Decimal(v.denominator)).sqrt()


@pytest.mark.parametrize("u", [1, 4, 7])
def test_unit_stderr_is_within_its_rounding_bound_of_the_exact_value(u):
    """Error bound (eps = 2^-53, gamma_k = k eps / (1 - k eps), M = m (m - 1) u^2, q = S1^2 / m), without
    underflow: q is formed with 2 roundings, q' = q (1 + t2), |t2| <= gamma_2; the difference d = (S2 - q')(1 + d3)
    is off the exact D = S2 - q by at most gamma_2 q + eps (S2 + q (1 + gamma_2)) <= gamma_3 (S2 + q); the three
    divisions and the two products forming M and u^2 are 4 more relative roundings of the quotient, so the
    computed variance v is off V = D / M by at most B = gamma_8 (S2 + q) / M.  The clamp at 0 does not increase the
    distance, and sqrt(a) - sqrt(b) <= min(sqrt|a - b|, |a - b| / sqrt(b)); the root adds one rounding:
    |se - SE| <= eps se + min(sqrt(B), B / SE)."""
    rng = np.random.default_rng(100 + u)
    s1, s2, n = moments(rng, 400, u)
    # and pixels whose estimate is far below the mean (cancellation in S2 - S1^2/m)
    c1, c2, cn = moments(np.random.default_rng(7), 100, u)
    s1 = np.concatenate([s1, c1 + 1e4 * ((cn + u - 1) // u)])
    s2 = np.concatenate([s2, c2 + 2e4 * c1 + 1e8 * ((cn + u - 1) // u)])
    n = np.concatenate([n, cn])
    got, _ = device_stderr(s1, s2, n, u)
    g8 = 8 * EPS / (1 - 8 * EPS)
    for a, b, k, se in zip(s1, s2, n, got):
        SE = exact_stderr(float(a), float(b), int(k), u)
        m = (int(k) + u - 1) // u
        B = Fraction(g8) * (Fraction(float(b)) + Fraction(float(a)) ** 2 / m) / (m * (m - 1) * u * u)
        B = Decimal(B.numerator) / Decimal(B.denominator)
        err = abs(Decimal(float(se)) - SE)
        bound = Decimal(EPS) * Decimal(float(se)) + (min(B / SE, B.sqrt()) if SE > 0 else B.sqrt())
        assert err <= bound, (a, b, k, u, se, SE, bound)


def test_unit_stderr_edges():
    tiny = 5e-324
    cases = [
        # (s1, s2, n, u, expected stderr or None for "numpy's bits", expected overflow)
        (0.0, 0.0, 0, 4, 0.0, False),              # n = 0: 0/0, clamped: 0
        (0.7, 0.7 * 0.7, 1, 1, 0.0, False),            # one unit: (S2 - S1^2) / 0 = 0/0 -> 0, what accum_noise exports
        (3.0, 9.0, 3, 4, 0.0, False),              # one (short) unit of 4
        (1.25, 0.9, 5, 4, None, False),            # the short last unit: m = ceil(5 / 4) = 2
        (10.0, 60.0, 10, 4, None, False),          # m = 3
        (float(2 ** 29), float(2 ** 29), 2 ** 30, 1, None, False),  # u = 1, n = 2^30: M = 2^30 (2^30 - 1)
        (-0.0, 0.0, 8, 4, 0.0, False),
        (tiny * 2 ** 20, tiny, 8, 1, None, False),  # subnormal moments
        (1e-160, 3e-321, 4, 1, None, False),
        (1e160, float("inf"), 8, 4, 0.0, True),    # S1^2 and S2 overflowed: inf - inf, clamped to 0
        (2e154, 1e308, 16, 4, 0.0, True),          # S1^2 overflowed alone: -inf, clamped to 0
        (1e150, 1e301, 16, 4, None, False),        # large but finite
        (1e154, float("inf"), 8, 4, float("inf"), True),  # S2 alone: an infinite estimate
    ]
    # S2 one ulp below S1^2 / m: a negative variance, clamped to 0
    s1, m = 3.0, 4
    q = (s1 * s1) / m
    cases.append((s1, float(np.nextafter(q, 0.0)), 16, 4, 0.0, False))
    s1a, s2a, na = (np.array([c[i] for c in cases]) for i in range(3))
    for u in sorted({c[3] for c in cases}):
        idx = [i for i, c in enumerate(cases) if c[3] == u]
        got, ovf = device_stderr(s1a[idx], s2a[idx], na[idx], u)
        want = np_unit_stderr(s1a[idx], s2a[idx], na[idx].astype(np.int64), u)
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), [cases[i] for i in idx]
        for j, i in enumerate(idx):
            exp, exp_ovf = cases[i][4], cases[i][5]
            if exp is not None:
                assert got[j] == exp and not math.copysign(1.0, got[j]) < 0, (cases[i], got[j])
            assert bool(ovf[j]) == exp_ovf, cases[i]
            assert bool(ovf[j]) == bool(np_overflow(np.float64(cases[i][0]), np.float64(cases[i][1])))


# ---------------------------------------------------------------- finalize_adaptive_kernel

F_MEAN_DIVIDE, F_QUANT_LINEAR = O.F_MEAN_DIVIDE, O.F_QUANT_LINEAR


def np_quantise(c, linear):
    with np.errstate(all="ignore"):
        if linear:
            v = 255.999 * c
        else:
            g = np.where(c > 0.0, np.sqrt(np.where(c > 0.0, c, 0.0)), 0.0)
            lo = np.where(g > 0.0, g, 0.0)
            v = 256.0 * np.where(lo < 0.999, lo, 0.999)
        return np.where(np.isnan(v), 0, np.trunc(np.nan_to_num(v)).astype(np.int64) & 0xFF).astype(np.uint8)


def np_finalize(st, mode, nchunks, spp, flags, strict, mean_n, decide, unit, target, least, tol, W, H, shard):
    """finalize_adaptive_kernel restated: returns the new state dict."""
    st = {k: v.copy() for k, v in st.items()}
    tr = st["live"] != 0
    s1, s2 = st["acc"].copy(), st["acc2"].copy()
    if mode == "strict":
        for k in range(spp):
            x = st["sample_buf"][k, :, :3]
            s1[tr] = s1[tr] + x[tr]
            s2[tr] = s2[tr] + x[tr] * x[tr]
    elif mode == "seeded":
        s1[tr] = st["partial"][tr]
    else:
        for c in range(nchunks):
            x = st["partial"][:, c]
            s1[tr] = s1[tr] + x[tr]
            s2[tr] = s2[tr] + x[tr] * x[tr]
    st["acc"][tr] = s1[tr]
    if mode != "seeded":
        st["acc2"][tr] = s2[tr]
    if not decide:
        return st
    st["samples"][tr] = mean_n
    n = st["samples"].astype(np.int64)
    mean = (0.0 + s1) if strict else s1.copy()
    if flags & F_MEAN_DIVIDE:
        mean = mean / n[:, None].astype(np.float64)
    else:
        mean = mean * (1.0 / n[:, None].astype(np.float64))
    rows = np.array(render.shard_rows(H, *shard)) if shard else np.arange(H)
    lin = st["lin"].reshape(H, W, 3)
    rgb = st["rgb"].reshape(H, W, 3)
    lin[rows] = mean.reshape(len(rows), W, 3)
    rgb[rows] = np_quantise(mean, bool(flags & F_QUANT_LINEAR)).reshape(len(rows), W, 3)
    se = np_unit_stderr(s1, s2, n[:, None], unit)
    with np.errstate(invalid="ignore"):
        t = tol[0] + tol[1] * np.abs(mean)
    noisy = (n < least) | (se > t).any(axis=1) | np_overflow(s1, s2).any(axis=1)
    st["live"][tr] = ((n < target) & noisy)[tr].astype(np.uint8)
    return st


def synthetic_state(rng, P, W, H, mode, nchunks, spp, mean_n):
    def signed(shape):
        x = rng.normal(0.5, 1.0, size=shape)
        x[rng.random(shape) < 0.05] = -0.0
        x[rng.random(shape) < 0.05] = 0.0
        return x
    live = (rng.random(P) < 0.7).astype(np.uint8)
    st = dict(live=live,
              acc=signed((P, 3)) * 8, acc2=np.abs(rng.normal(0, 30, size=(P, 3))),
              samples=np.where(live != 0, mean_n - (spp if mode != "chunked" else nchunks * 4),
                               rng.integers(1, mean_n, size=P)).astype(np.int32),
              lin=np.full((H * W * 3,), np.nan), rgb=np.full((H * W * 3,), 77, dtype=np.uint8))
    if mode == "strict":
        sb = np.zeros((spp, P, 4))
        sb[:, :, :3] = signed((spp, P, 3))
        st["sample_buf"] = sb
    elif mode == "seeded":
        st["partial"] = signed((P, 3)) * 8
    else:
        st["partial"] = signed((P, nchunks, 3))
    return st


def run_finalize(st, mode, nchunks, spp, flags, strict, mean_n, decide, unit, target, least, tol, W, shard, P):
    dev = {k: cuda(v) for k, v in st.items()}
    A = K.AParams()
    A.sample_buf = dev["sample_buf"].data_ptr() if "sample_buf" in dev else None
    A.sample_stride = P
    A.partial = dev["partial"].data_ptr() if "partial" in dev else None
    A.out_linear, A.out_rgb8 = dev["lin"].data_ptr(), dev["rgb"].data_ptr()
    A.W, A.spp, A.nchunks = W, spp, nchunks
    A.shard_index, A.shard_count, A.shard_rows = shard if shard else (0, 1, 10 ** 6)
    A.flags, A.local_pixels = flags, P
    A.acc, A.acc2 = dev["acc"].data_ptr(), dev["acc2"].data_ptr()
    A.samples, A.live = dev["samples"].data_ptr(), dev["live"].data_ptr()
    A.seeded, A.strict, A.mean_n, A.decide = int(mode == "seeded"), int(strict), mean_n, int(decide)
    A.unit, A.target, A.min_samples = unit, target, least
    A.abs_tol, A.rel_tol = tol
    K.finalize(A)
    return {k: v.cpu().numpy() for k, v in dev.items()}


MODES = [("chunked", c) for c in range(1, 6)] + [("strict", 1), ("seeded", 1)]
LAYOUTS = [("main", O.FLAGS_MAIN, None), ("realm-shard", O.FLAGS_REALM, (1, 3, 2)), ("i-shard", O.FLAGS_I, (2, 3, 2))]


@pytest.mark.parametrize("decide", [1, 0])
@pytest.mark.parametrize("layout", LAYOUTS, ids=[l[0] for l in LAYOUTS])
@pytest.mark.parametrize("mode,nchunks", MODES, ids=[f"{m}{c}" for m, c in MODES])
def test_finalize_adaptive_kernel_against_numpy(mode, nchunks, layout, decide):
    """Images, samples, live, S1 and S2 bit for bit against numpy; with decide = 0 (a sub-pass of a strict pass)
    nothing but S1 and S2 changes."""
    _, flags, shard = layout
    W, H = 13, 11
    P = (len(render.shard_rows(H, *shard)) if shard else H) * W
    rng = np.random.default_rng(zlib.crc32(f"{mode}{nchunks}{layout[0]}{decide}".encode()))
    strict = mode != "chunked"
    spp = 7 if mode == "strict" else 1
    unit = 1 if strict else 4
    mean_n, least = 20, 8
    st = synthetic_state(rng, P, W, H, mode, nchunks, spp, mean_n)
    # a tolerance at the median estimate, so that both outcomes occur, and a target above the pass for some runs
    probe = np_finalize(st, mode, nchunks, spp, flags, strict, mean_n, 1, unit, 10 ** 6, least, (1e300, 0.0), W, H, shard)
    se = np_unit_stderr(probe["acc"], probe["acc2"], probe["samples"][:, None].astype(np.int64), unit).max(axis=1)
    tol = (float(np.median(se)), 0.01)
    target = 24 if decide else mean_n
    args = (mode, nchunks, spp, flags, strict, mean_n, decide, unit, target, least, tol, W)
    got = run_finalize(st, *args, shard, P)
    want = np_finalize(st, *args, H, shard)
    for k in want:
        assert np.array_equal(np.asarray(got[k]).view(np.uint8), np.asarray(want[k]).view(np.uint8)), (k, mode, decide)
    if decide:
        tr = st["live"] != 0
        assert got["live"][tr].any() and not got["live"][tr].all()
    else:
        for k in ("lin", "rgb", "samples", "live"):
            assert np.array_equal(got[k].view(np.uint8), st[k].view(np.uint8)), k


def test_overflowing_moments_count_as_noisy():
    """A unit sum above sqrt(DBL_MAX) overflows S2 and S1^2: the variance is inf - inf = NaN, which the clamp would
    read as 0.  Such a pixel stays active under any tolerance; its neighbours with finite moments stop."""
    W, H = 16, 4
    P = W * H
    rng = np.random.default_rng(5)
    st = synthetic_state(rng, P, W, H, "chunked", 4, 1, 16)
    st["live"][:] = 1
    st["samples"][:] = 0
    st["acc"][:] = 0.0
    st["acc2"][:] = 0.0
    big = rng.random(P) < 0.25
    st["partial"][big, :, 1] = 1e160 * (1.0 + rng.random((big.sum(), 4)))
    args = ("chunked", 4, 1, O.FLAGS_MAIN, False, 16, 1, 4, 64, 8, (1e300, 1e300), W)
    got = run_finalize(st, *args, None, P)
    want = np_finalize(st, *args, H, None)
    for k in want:
        assert np.array_equal(np.asarray(got[k]).view(np.uint8), np.asarray(want[k]).view(np.uint8)), k
    assert np.array_equal(got["live"] != 0, big)
