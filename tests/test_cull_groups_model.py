"""CPU model of the two-level cull of render_lane2_kernel (DESIGN.md 4.2, "group bound"; no GPU needed): the host's
slot order and group records (rtclj_abi.cu, cull_groups) and the kernel's fp32 group test (rtclj_lane2_kernel.cuh,
level 1), restated in numpy.  The kernel's survivors equal the flat cull's only if a group record that rejects a line
has no member whose own fp32 cull value for that line is >= 0; this checks that on random, grazing and far-away rays
and on degenerate groups."""
import numpy as np

from test_kernel_arithmetic_models import EPS32, F32, fma32, round_up_f32

GROUP = 16                       # kGroupSpheres
GROUP_KQ = F32(1.0 - 1.0 / 512)  # kGroupKq


def cull_groups(c32, ws, r):
    """cull_groups of rtclj_abi.cu: c32 (n, 3) float32 shifted centres, ws (n,) their Ws, r (n,) radii ->
    slot -> list index (-1: padding), the group records' centres (ng, 3) float32 and Ws (ng,) float32."""
    n = len(r)
    ng = (n + GROUP - 1) // GROUP
    order = sorted(range(n), key=lambda i: -abs(r[i]))                   # stable: list order among equal radii
    n0 = n - GROUP * max(ng - 1, 0)

    def split(lo, hi):
        m = (hi - lo) // GROUP
        if m <= 1:
            return
        part = c32[order[lo:hi]]
        ext = [F32(part[:, a].max()) - F32(part[:, a].min()) for a in range(3)]
        a = 0 if ext[0] >= ext[1] and ext[0] >= ext[2] else 1 if ext[1] >= ext[2] else 2
        mid = lo + m // 2 * GROUP
        order[lo:hi] = sorted(order[lo:hi], key=lambda i: (c32[i, a], i))
        split(lo, mid)
        split(mid, hi)

    split(n0, n)
    groups = [sorted(order[:n0])] + [sorted(order[n0 + (g - 1) * GROUP: n0 + g * GROUP]) for g in range(1, ng)]
    slots = np.full(ng * GROUP, -1)
    for g, members in enumerate(groups):
        slots[g * GROUP: g * GROUP + len(members)] = members
    lam, t, slack = 2.0 ** -15, 2.0 ** -5, 2.0 ** -14
    gc = np.zeros((ng, 3), F32)
    gws = np.zeros(ng, F32)
    for g, members in enumerate(groups):
        m = np.array(members)
        c = c32[m].astype(np.float64)
        C = (0.5 * (c.min(0) + c.max(0))).astype(F32)
        c2 = (c * c).sum(1)
        Q = np.max(np.sqrt(r[m] * r[m] * (1.0 + lam) + lam * c2) + np.sqrt(((c - C.astype(np.float64)) ** 2).sum(1)))
        C2 = float((C.astype(np.float64) ** 2).sum())
        A = (1.0 + t) * Q * Q * (1.0 + slack) + slack * C2
        if np.any(ws[m] >= F32(3.0e38)) or not (A < 1e36 and C2 < 1e36):
            gc[g], gws[g] = 0.0, F32(3.0e38)
        else:
            gc[g], gws[g] = C, round_up_f32(np.array([A - C2]))[0]
    return slots, gc, gws


def table(C, r):
    """The host's fp32 cull records (rtclj_ctx_set_scene): shifted centres and Ws, 3e38 where |c| or |r| >= 1e15."""
    shift = np.sort(C, axis=0)[len(C) // 2]
    far = np.maximum(np.abs(C - shift).max(1), np.abs(r))
    c32 = np.where((far < 1e15)[:, None], C - shift, 0.0).astype(F32)
    c2 = (c32.astype(np.float64) ** 2).sum(1)
    eps = float(EPS32)
    ws = np.where(far < 1e15, round_up_f32(r * r * (1.0 + 8.0 * eps) - c2 * (1.0 - 96.0 * eps)), F32(3.0e38)).astype(F32)
    return shift, c32, ws


def view(O, D, shift, rng):
    """make_view: per ray 2o, d-hat, -o.d-hat and the |o|^2 term."""
    of = (O - shift).astype(F32)
    df = D.astype(F32)
    l2 = (df[:, 0] * df[:, 0] + df[:, 1] * df[:, 1]) + df[:, 2] * df[:, 2]
    inv = (1.0 / np.sqrt(l2.astype(np.float64))).astype(F32)
    for _ in range(2):                                                  # rsqrt.approx: up to 2 ulp off
        inv = np.nextafter(inv, np.where(rng.random(len(inv)) < 0.5, F32(0), F32(np.inf)))
    dh = df * inv[:, None]
    nbeta = -fma32(of[:, 2], dh[:, 2], fma32(of[:, 1], dh[:, 1], of[:, 0] * dh[:, 0]))
    kq = fma32(of[:, 2], of[:, 2], fma32(of[:, 1], of[:, 1], of[:, 0] * of[:, 0])) * -(F32(1.0) - F32(96.0) * EPS32)
    return F32(2.0) * of, dh, nbeta, kq


def cull_values(c, ws, o2, dh, nbeta, kq):
    """The kernel's fp32 cull value of every (ray, record): b^2 + s in the FFMA2 order of the cull block."""
    cx, cy, cz = (c[None, :, k] for k in range(3))
    bb = fma32(cz, dh[:, 2:3], fma32(cy, dh[:, 1:2], fma32(cx, dh[:, 0:1], nbeta[:, None] + F32(0) * cx)))
    ss = fma32(cz, o2[:, 2:3], fma32(cy, o2[:, 1:2], fma32(cx, o2[:, 0:1], ws[None, :] + kq[:, None])))
    return fma32(bb, bb, ss)


def check_scene(C, r, O, D, rng):
    """Asserts the invariant on every (ray, group); returns how many (ray, group) pairs the records reject."""
    shift, c32, ws = table(C, r)
    slots, gc, gws = cull_groups(c32, ws, r)
    assert sorted(slots[slots >= 0].tolist()) == list(range(len(r)))   # every list index in exactly one slot
    o2, dh, nbeta, kq = view(O, D, shift, rng)
    with np.errstate(over="ignore", invalid="ignore"):
        member = np.signbit(cull_values(c32, ws, o2, dh, nbeta, kq))      # True: the flat cull rejects
        group = np.signbit(cull_values(gc, gws, o2, dh, nbeta, kq * GROUP_KQ))
    for g in range(len(gws)):
        m = slots[g * GROUP:(g + 1) * GROUP]
        m = m[m >= 0]
        bad = group[:, g] & ~member[:, m].all(1)
        assert not bad.any(), (g, int(np.argmax(bad)))
    return int(group.sum())


def grazing_rays(C, r, m, rng, far=1.0):
    """Rays whose line passes at |r| (1 +- 1e-6) from a random sphere's centre, from origins up to `far` scene
    sizes away."""
    j = rng.integers(0, len(r), m)
    d = rng.normal(size=(m, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    p = rng.normal(size=(m, 3))
    p -= (p * d).sum(1, keepdims=True) * d
    p /= np.linalg.norm(p, axis=1, keepdims=True)
    touch = C[j] + p * (np.abs(r[j]) * (1.0 + rng.uniform(-1e-6, 1e-6, m)))[:, None]
    size = np.ptp(C, axis=0).max() + np.abs(r).max() + 1e-30
    O = touch - d * (size * far * rng.uniform(0.0, 1.0, m))[:, None]
    return O, d * 10.0 ** rng.uniform(-3, 3, (m, 1))


def cover_like(rng, n, scale):
    """A slab of small spheres with the ground and three large spheres, as the cover scene."""
    C = np.column_stack([rng.uniform(-11, 11, n), rng.uniform(0.15, 0.25, n), rng.uniform(-11, 11, n)]) * scale
    r = np.full(n, 0.2 * scale)
    C[0], r[0] = (0.0, -1000.0 * scale, 0.0), 1000.0 * scale
    for k, x in ((1, 0.0), (2, -4.0), (3, 4.0)):
        C[k], r[k] = (x * scale, scale, 0.0), scale
    return C, r


def test_rejected_groups_hold_no_member_the_flat_cull_keeps():
    rng = np.random.default_rng(20261022)
    rejected = 0
    for case in range(60):
        n = int(rng.choice([1, 15, 16, 17, 64, 100, 257, 484, 512]))
        scale = 10.0 ** rng.uniform(-3, 8)
        if case % 3 == 0 and n >= 4:
            C, r = cover_like(rng, n, scale)
        else:
            C = rng.normal(0, scale, (n, 3)) * np.where(rng.random((n, 1)) < 0.2, 0.01, 1.0)
            r = scale * 10.0 ** rng.uniform(-3, 0, n) * np.where(rng.random(n) < 0.05, -1.0, 1.0)
        C = C + rng.normal(0, scale, 3) * (1e3 if case % 4 == 0 else 1.0)    # a scene far from the origin
        m = 600
        O1, D1 = grazing_rays(C, r, m, rng, far=10.0 ** rng.uniform(-1, 3))
        O2 = C[rng.integers(0, n, m)] + rng.normal(0, scale, (m, 3)) * 10.0 ** rng.uniform(-2, 4, (m, 1))
        D2 = rng.normal(0, 1, (m, 3))
        rejected += check_scene(C, r, np.vstack([O1, O2]), np.vstack([D1, D2]), rng)
    assert rejected > 100_000


def test_degenerate_groups():
    """Coincident centres, zero and negative radii, one sphere, a group of huge spheres, spheres beyond the fp32
    range of the table (never rejected) -- and rays that start exactly at a centre."""
    rng = np.random.default_rng(7)
    scenes = [
        (np.zeros((40, 3)), np.zeros(40)),
        (np.tile([[1.0, 2.0, 3.0]], (33, 1)), np.linspace(-1.0, 1.0, 33)),
        (np.array([[0.5, 0.5, 0.5]]), np.array([0.25])),
        (rng.normal(0, 1e6, (48, 3)), np.full(48, 1e6)),
        (np.vstack([rng.normal(0, 1.0, (31, 3)), [[1e16, 0.0, 0.0]]]), np.append(np.full(31, 0.1), 1.0)),
        (np.vstack([rng.normal(0, 1.0, (20, 3)), [[0.0, 0.0, 0.0]]]), np.append(np.full(20, 0.1), 3e15)),
    ]
    for C, r in scenes:
        O1, D1 = grazing_rays(C, r, 400, rng, far=10.0)
        O2 = C[rng.integers(0, len(r), 100)]
        D2 = rng.normal(0, 1, (100, 3))
        check_scene(C, r, np.vstack([O1, O2]), np.vstack([D1, D2]), rng)


def test_the_cover_scene_field_is_grouped_by_place():
    """Group 0 takes the ground and the three large spheres with the padding; the field's groups are compact."""
    rng = np.random.default_rng(3)
    C, r = cover_like(rng, 484, 1.0)
    shift, c32, ws = table(C, r)
    slots, gc, gws = cull_groups(c32, ws, r)
    assert len(gws) == 31 and sorted(slots[:4].tolist()) == [0, 1, 2, 3] and (slots[4:16] == -1).all()
    radius = np.sqrt(gws[1:].astype(np.float64) + (gc[1:].astype(np.float64) ** 2).sum(1))
    assert radius.max() < 4.5, radius.max()  # 16 spheres of a 22 x 22 field: about a 4 x 4 patch
