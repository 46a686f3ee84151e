"""CPU models of two pieces of device arithmetic whose correctness the kernels rely on (no GPU needed): the
packed prefilter candidate (rtclj_kernels.cuh: cand_key / cand_insert) and the operand window of the
shared-reciprocal division (div_by / divs_by).  The models restate the device code operation for operation in
numpy float32 / integer arithmetic; the GPU side of both is covered by the parity tests and by
tools/microbench/div_recip_check.cu (profiles/r2_div_recip_check.txt)."""
import numpy as np

F32 = np.float32


def cand_key(lo, i):
    """rtclj_kernels.cuh cand_key(): clamp, lower by 2^-13 of itself (one fused multiply-add), index into the nine
    low mantissa bits."""
    lk = np.maximum(lo.astype(F32), F32(-1.0e38))
    # fmaf(-|lk|, 2^-13, lk): the product and the sum are exact in double, so one rounding to float32 = the fused result
    lk = (lk.astype(np.float64) - np.abs(lk.astype(np.float64)) * 2.0 ** -13).astype(F32)
    lk = lk - F32(1.0e-30)   # covers |lo| < 2^-113, where the relative step underflows
    bits = (lk.view(np.uint32) & np.uint32(0xFFFFFE00)) | i.astype(np.uint32)
    return bits.view(F32)


def test_packed_candidate_is_a_lower_bound_that_carries_its_index():
    rng = np.random.default_rng(7)
    n = 400_000
    mag = 10.0 ** rng.uniform(-30, 30, n)
    lo = (rng.choice([-1.0, 1.0], n) * mag).astype(F32)
    lo[:1000] = F32(0.0)
    lo[1000:2000] = F32(-np.inf)           # an fp32 overflow in the bound
    lo[2000:2100] = np.finfo(F32).tiny     # smallest normal
    idx = rng.integers(0, 512, n)
    key = cand_key(lo, idx)
    assert np.all(np.isfinite(key))
    assert np.array_equal(key.view(np.uint32) & np.uint32(0x1FF), idx.astype(np.uint32))
    # still a lower bound, whatever the index bits (-inf, "no information", becomes -1e38: below every root, which
    # the input range keeps under 1e30 in magnitude -- DESIGN.md 4.8)
    assert np.all(key <= np.maximum(lo, F32(-1.0e38)))
    finite = np.isfinite(lo) & (np.abs(lo) > 1e-20)
    assert np.all(np.abs(key[finite] - lo[finite]) <= np.abs(lo[finite]) * F32(2.0 ** -12))   # and a tight one
    assert np.all(key < F32(1.0e38))                          # never mistaken for an empty slot (3.0e38)


def test_candidate_insertion_keeps_the_three_smallest_sorted():
    rng = np.random.default_rng(11)
    for _ in range(300):
        m = int(rng.integers(1, 9))
        lo = rng.normal(0, 50, m).astype(F32)
        idx = rng.permutation(512)[:m]
        keys = cand_key(lo, idx)
        k = [F32(3.0e38)] * 3
        displaced = []
        for key in keys:                                      # cand_insert(): a float min / max pair per slot
            for s in range(3):
                t = min(k[s], key); key = max(k[s], key); k[s] = t
            if key < F32(1.0e38):
                displaced.append(key)
        want = sorted(keys.tolist())
        assert [float(x) for x in k[: min(m, 3)]] == want[: min(m, 3)]
        assert sorted(float(x) for x in displaced) == want[3:]
        for s in range(min(m, 3)):                            # the slot still names its sphere
            assert int(np.array([k[s]], dtype=F32).view(np.uint32)[0] & 0x1FF) in set(int(x) for x in idx)


def exp_off(v):
    """rtclj_kernels.cuh exp_off(): biased exponent of a double, offset so that ONE unsigned compare tests a window."""
    hi = (np.atleast_1d(np.asarray(v, dtype=np.float64)).view(np.uint64) >> np.uint64(32)).astype(np.uint64)
    off = ((hi & np.uint64(0x7FF00000)) + np.uint64(2 ** 32 - (543 << 20))) & np.uint64(0xFFFFFFFF)   # mod 2^32, as on the device
    return off.astype(np.uint32) if np.ndim(v) else np.uint32(off[0])


K_EXP_SPAN = np.uint32(961 << 20)


def test_division_window_on_the_operands_bounds_the_quotient():
    """Both operands inside [2^-480, 2^481) => the quotient inside (2^-961, 2^961), i.e. inside the range on which
    the fast path was verified against `/` -- so the kernels do not test the quotient."""
    rng = np.random.default_rng(3)
    n = 300_000
    e = rng.integers(-1074, 1024, (2, n))
    m = rng.uniform(1.0, 2.0, (2, n))
    with np.errstate(over="ignore", under="ignore"):
        a = np.ldexp(m[0], e[0]) * rng.choice([-1.0, 1.0], n)
        b = np.ldexp(m[1], e[1]) * rng.choice([-1.0, 1.0], n)
    a[:50] = 0.0; a[50:100] = -0.0; a[100:150] = np.inf; a[150:200] = np.nan
    with np.errstate(all="ignore"):
        ok = (exp_off(a) < K_EXP_SPAN) & (exp_off(b) < K_EXP_SPAN)
        q = a / b
    assert ok.sum() > 10_000
    assert np.all(np.isfinite(q[ok]))
    assert np.all((np.abs(q[ok]) > 2.0 ** -961) & (np.abs(q[ok]) < 2.0 ** 961))
    lo_edge, hi_edge = 2.0 ** -480, np.nextafter(2.0 ** 481, 0)
    assert exp_off(lo_edge) < K_EXP_SPAN and exp_off(hi_edge) < K_EXP_SPAN
    assert not exp_off(np.nextafter(lo_edge, 0)) < K_EXP_SPAN and not exp_off(2.0 ** 481) < K_EXP_SPAN
    for special in (0.0, -0.0, 5e-324, np.inf, -np.inf, np.nan):   # zero, denormal, inf, NaN: outside, they divide
        assert not exp_off(special) < K_EXP_SPAN


def test_zero_numerator_on_the_fast_path_has_the_quotients_sign():
    """div_by(): a zero numerator returns n * y with y ~ 1/d, sign(y) = sign(d): the exact signed zero of n / d."""
    for n in (0.0, -0.0):
        for d in (3.0, -3.0, 1e-300, -1e300):
            y = 1.0 / d                                        # any value with the sign of d
            assert np.signbit(n * y) == np.signbit(np.float64(n) / np.float64(d))


# ---------------------------------------------------------------------------------------------------------------
# The conservative fp32 cull and the fp32 root prefilter (DESIGN.md "cull error bound"), restated in numpy: host
# side of the table = rtclj_abi.cu rtclj_ctx_set_scene, device side = make_view / the cull block / the prefilter of
# rtclj_kernels.cuh and rtclj_path_step.cuh.  Checked against the reference's own double arithmetic
# (hittable.clj:9-23): a sphere the reference can hit is never culled and never dropped by the prefilter.
def fma32(a, b, c):
    """fmaf: the product of two float32 is exact in float64; the sum's double rounding is far below the margins"""
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(F32)


EPS32 = F32(2.0 ** -24)


def round_up_f32(v):
    f = v.astype(F32)
    return np.where(f.astype(np.float64) < v, np.nextafter(f, F32(np.inf)), f)


def cull_model(C, r, O, D, rng):
    """Returns per (ray, sphere): dd (conservative discriminant), far_hi, lo, and per ray tmin_lo, len32."""
    shift = np.median(C, axis=0) if len(C) % 2 else np.sort(C, axis=0)[len(C) // 2]     # nth_element(n / 2)
    c32 = (C - shift).astype(F32)                                                      # (n, 3)
    c2 = (c32.astype(np.float64) ** 2).sum(1)
    eps = float(EPS32)
    ws = round_up_f32(r * r * (1.0 + 8.0 * eps) - c2 * (1.0 - 96.0 * eps))            # (n,)
    of = (O - shift).astype(F32)                                                       # (m, 3)
    df = D.astype(F32)
    l2 = (df[:, 0] * df[:, 0] + df[:, 1] * df[:, 1]) + df[:, 2] * df[:, 2]             # fp32, unfused
    inv = (1.0 / np.sqrt(l2.astype(np.float64))).astype(F32)
    inv = np.nextafter(inv, np.where(rng.random(len(inv)) < 0.5, F32(0), F32(np.inf)))  # rsqrt.approx: up to 2 ulp off
    inv = np.nextafter(inv, np.where(rng.random(len(inv)) < 0.5, F32(0), F32(np.inf)))
    dh = df * inv[:, None]
    len32 = l2 * inv
    mo = np.abs(of).max(1)
    nbeta = -fma32(of[:, 2], dh[:, 2], fma32(of[:, 1], dh[:, 1], of[:, 0] * dh[:, 0]))
    kq = fma32(of[:, 2], of[:, 2], fma32(of[:, 1], of[:, 1], of[:, 0] * of[:, 0])) * -(F32(1.0) - F32(96.0) * EPS32)
    cx, cy, cz = (c32[None, :, k] for k in range(3))
    bb = fma32(cz, dh[:, 2:3], fma32(cy, dh[:, 1:2], fma32(cx, dh[:, 0:1], nbeta[:, None] + F32(0) * cx)))
    two = F32(2.0)
    ss = fma32(cz, two * of[:, 2:3], fma32(cy, two * of[:, 1:2], fma32(cx, two * of[:, 0:1], ws[None, :] + kq[:, None])))
    dd = fma32(bb, bb, ss)
    sq = np.sqrt(np.maximum(dd, F32(0)).astype(np.float64)).astype(F32)
    sq = np.nextafter(sq, np.where(rng.random(sq.shape) < 0.5, F32(0), F32(np.inf)))    # sqrt.approx
    sq = sq * (F32(1.0) + F32(16.0) * EPS32)
    eb = EPS32 * (F32(24.0) * (np.abs(cx) + np.abs(cy) + np.abs(cz)) + F32(40.0) * mo[:, None])
    far_hi = bb + sq + eb
    lo = bb - sq - eb
    tmin_lo = F32(1e-3) * len32 * (F32(1.0) - F32(16.0) * EPS32)
    return dd, far_hi, lo, tmin_lo, len32


def reference_roots(C, r, O, D):
    """hittable.clj:9-23 in double: near and far root per (ray, sphere), NaN where the discriminant is negative."""
    oc = C[None, :, :] - O[:, None, :]
    a = (D * D).sum(1)[:, None]
    h = (D[:, None, :] * oc).sum(2)
    c = (oc * oc).sum(2) - (r * r)[None, :]
    disc = h * h - a * c
    with np.errstate(invalid="ignore"):
        sq = np.sqrt(disc)
    return (h - sq) / a, (h + sq) / a, disc


def test_fp32_cull_and_prefilter_never_drop_a_sphere_the_reference_can_hit():
    rng = np.random.default_rng(20261019)
    checked_hits = 0
    for case in range(200):
        n, m = int(rng.integers(1, 40)), 400
        scale = 10.0 ** rng.uniform(-2, 4)
        C = rng.normal(0, scale, (n, 3)) + rng.normal(0, scale * 3, 3)
        r = np.abs(rng.normal(0, scale * 0.3, n)) + scale * 1e-3
        if case % 3 == 0:
            r[0] = scale * 1000.0; C[0] = [0.0, -r[0], 0.0]                         # a ground sphere
        if case % 5 == 0:
            r[-1] = -r[-1]                                                          # the inner bubble's negative radius
        kind = case % 4
        O = rng.normal(0, scale * (0.1, 1.0, 5.0, 30.0)[kind], (m, 3)) + C[rng.integers(0, n, m)] * (kind < 2)
        D = rng.normal(0, 1, (m, 3)) * 10.0 ** rng.uniform(-3, 3, (m, 1))           # the reference never normalises d
        j = rng.integers(0, n, m // 2)                                              # half of the rays start ON a sphere
        u = rng.normal(0, 1, (m // 2, 3)); u /= np.linalg.norm(u, axis=1, keepdims=True)
        O[: m // 2] = C[j] + u * np.abs(r[j])[:, None]
        dd, far_hi, lo, tmin_lo, len32 = cull_model(C, r, O, D, rng)
        near, far, disc = reference_roots(C, r, O, D)
        can_hit = (disc >= 0.0) & ((near > 1e-3) | (far > 1e-3))                    # the reference would accept a root
        checked_hits += int(can_hit.sum())
        # (1) the cull: D' < 0 proves a miss
        assert not np.any(can_hit & (dd < 0)), case
        # (2) the prefilter's first rejection: the far root certainly at or below t_min
        rej_far = far_hi < tmin_lo[:, None]
        assert not np.any(can_hit & (dd >= 0) & rej_far), case
        # (3) its bounds: lo <= root * |d| <= far_hi for the root the reference accepts
        root = np.where(near > 1e-3, near, far)
        arc = root * np.sqrt((D * D).sum(1))[:, None]
        ok = can_hit & (dd >= 0)
        slack = 1.0 + 16.0 * float(EPS32)
        assert np.all(lo[ok].astype(np.float64) <= arc[ok] * slack + 1e-300), case
        assert np.all(far_hi[ok].astype(np.float64) * slack >= arc[ok]), case
    assert checked_hits > 40_000


def test_symmetric_uniforms_in_one_conversion_equal_the_reference_form_for_every_input():
    """rtclj_kernels.cuh sym21 / sym24: (f - 2^20) 2^-20 and ((w >> 8) - 2^23) 2^-23 against the oracle's form
    -1 + 2 u with u = f 2^-21 / (w >> 8) 2^-24 (vec3a.clj:71-79 `rand-double -1 1` on the shim's uniforms) --
    EVERY 21-bit field and EVERY 24-bit value, bit patterns included (the midpoint must be +0.0)."""
    f = np.arange(1 << 21, dtype=np.int64)
    a = (f - (1 << 20)).astype(np.float64) * (1.0 / (1 << 20))
    b = -1.0 + 2.0 * (f.astype(np.float64) * (1.0 / (1 << 21)))
    assert np.array_equal(a.view(np.uint64), b.view(np.uint64))
    w = np.arange(1 << 24, dtype=np.int64)
    a = (w - (1 << 23)).astype(np.float64) * (1.0 / (1 << 23))
    b = -1.0 + 2.0 * (w.astype(np.float64) * (1.0 / (1 << 24)))
    assert np.array_equal(a.view(np.uint64), b.view(np.uint64))


def test_list_scan_with_strict_bounds_equals_the_lexicographic_minimum():
    """hit-anything (raytracing.clj:33-43) scans the list passing closest-so-far as t-max, with strict bounds in the
    sphere test (hittable.clj:15-21).  The kernels resolve cull survivors in ANY order as the lexicographic minimum
    of (root_i, i), root_i = the near root if it exceeds t-min, else the far root if that does (exact_test_lex).
    Equivalence on random root sets drawn from a few values, so that exact ties are frequent."""
    rng = np.random.default_rng(5)
    tmin = 1e-3
    vals = np.array([-2.0, 0.0, 5e-4, 1e-3, 2e-3, 0.5, 0.5, 1.0, 3.0])
    for _ in range(20_000):
        n = int(rng.integers(1, 7))
        near = rng.choice(vals, n)
        far = np.maximum(near, rng.choice(vals, n))          # near <= far
        miss = rng.random(n) < 0.3                           # negative discriminant
        # the reference: sequential, strict bounds, first body wins an exact tie
        closest, best = np.inf, -1
        for i in range(n):
            if miss[i]:
                continue
            root = near[i]
            if root <= tmin or closest <= root:
                root = far[i]
                if root <= tmin or closest <= root:
                    continue
            closest, best = root, i
        # the kernels: any order (here: reversed), lexicographic minimum
        c2, b2 = np.inf, -1
        for i in reversed(range(n)):
            if miss[i]:
                continue
            root = near[i]
            if root <= tmin:
                root = far[i]
                if root <= tmin:
                    continue
            if root < c2 or (root == c2 and i < b2):
                c2, b2 = root, i
        assert (closest, best) == (c2, b2), (near, far, miss)


def reference_pick(roots, tmin=1e-3):
    """hit-anything's sequential scan (hittable.clj:15-21, rt_oracle.c sphere_root), which scan_all_ni restates: near
    root, then far root, accepted when !(root <= t_min || closest <= root) -- true for a NaN root."""
    closest, best = np.inf, -1
    for i, r in enumerate(roots):
        if r is None:
            continue
        for root in r:
            if not (root <= tmin or closest <= root):
                closest, best = root, i
                break
    return closest, best


def lex_pick(roots, tmin=1e-3):
    """exact_test_lex in any order (here: reversed): the near root unless it is <= t_min, then the far root unless it
    is <= t_min; lexicographic minimum of (root_i, i), which a NaN root never is."""
    closest, best = np.inf, -1
    for i in reversed(range(len(roots))):
        if roots[i] is None:
            continue
        root = roots[i][0]
        if root <= tmin:
            root = roots[i][1]
            if root <= tmin:
                continue
        if root < closest or (root == closest and i < best):
            closest, best = root, i
    return closest, best


def primary_pick(roots, tmin=1e-3):
    """render_primary_kernel: exact_test_lex's choice of root, in list order, accepted when !(closest <= root)."""
    closest, best = np.inf, -1
    for i, r in enumerate(roots):
        if r is None:
            continue
        root = r[0]
        if root <= tmin:
            root = r[1]
            if root <= tmin:
                continue
        if not (closest <= root):
            closest, best = root, i
    return closest, best


def test_scan_rules_on_nan_roots():
    """Root pairs (h -+ sq) / a from operands drawn with NaN, +-inf, zero and exact ties at t_min = 1e-3 (a degenerate
    direction: |d|^2 = a is 0 or inf).  reference_pick is the rule of the oracle and of the exhaustive scans
    (exact_test_div restates it operation for operation), so the checks here are of the two rules that differ from it
    in form: the lexicographic form of the cull path never accepts a NaN root, so it differs from the reference
    exactly on sets with one; the primary kernel's rule (lexicographic choice of root, then `!(closest <= root)`)
    equals the reference on every set.  The kernels' scans themselves are compared with the oracle on the GPU
    (tests/test_gpu_degenerate_rays.py)."""
    rng = np.random.default_rng(17)
    hs = np.array([-np.inf, -1e300, -2.0, -0.0, 0.0, 5e-4, 1e-3, 2e-3, 1.0, 3.0, 1e300, np.inf, np.nan])
    sqs = np.array([0.0, 1e-3, 1.0, 2.0, 1e300, np.inf, np.nan])
    As = np.array([0.0, 1.0, 1.0, 2.0, 1e-300, 1e300, np.inf])
    differ = with_nan = 0
    for _ in range(20_000):
        n = int(rng.integers(1, 6))
        roots = []
        for _ in range(n):
            if rng.random() < 0.2:
                roots.append(None)                           # negative discriminant
                continue
            h, sq, a = rng.choice(hs), rng.choice(sqs), rng.choice(As)
            with np.errstate(all="ignore"):
                roots.append((np.float64(h - sq) / a, np.float64(h + sq) / a))
        want = reference_pick(roots)
        got = primary_pick(roots)
        assert got[1] == want[1] and (got[0] == want[0] or (got[0] != got[0] and want[0] != want[0])), roots
        nan = any(r is not None and (r[0] != r[0] or r[1] != r[1]) for r in roots)
        lex = lex_pick(roots)
        same = lex[1] == want[1] and (lex[0] == want[0] or (lex[0] != lex[0] and want[0] != want[0]))
        if not nan:
            assert same, roots                               # without a NaN root the cull path's rule is exact
        with_nan += nan
        differ += not same
    assert with_nan > 2000 and differ > 500, (with_nan, differ)


def test_cull_path_never_sees_a_nan_root():
    """Why the cull path may keep exact_test_lex: none of its roots is NaN.  The argument is the chain of bounds below,
    each taken at its worst case from the input limits; the random rays after it only spot-check the arithmetic.

    * The cull path runs only when fp32 |d|^2 lies in (1e-30, 1e30) (make_view).  fp32 rounds each component and
      the sum by at most 2^-24 relative, so the fp64 |d|^2 = a is below 1e30 (1 + 2^-20); and some fp32 component is
      at least sqrt(1e-30 / 3.1) > 5e-16, a normal fp32 value, so a > 2.5e-31 > 0: no 0 / 0, no x / inf.
    * Scene coordinates and radii are below 1e18 (rtclj_ctx_set_scene); a ray starts at the camera (|center| plus the
      defocus vectors below 1e18 per axis, validate()) or at a hit point on a sphere, below 2e18 per axis up to
      rounding.  So each component of oc = C - O is below 3e18 (with slack: 3.1e18), |oc| below sqrt(3) 3.1e18.
    * Then |h| <= |d| |oc|, c <= |oc|^2 + r^2, |disc| <= h^2 + a |c|: all finite, far below 1e70, so sqrt(disc),
      h -+ sq and (h -+ sq) / a are finite numbers (or disc < 0: no root)."""
    slack = 1.01
    a_max, a_min = 1e30 * (1.0 + 2.0 ** -20), (1e-30 / 3.1)
    assert np.float32(np.sqrt(a_min)) > np.finfo(np.float32).tiny                    # a normal fp32 component
    oc_max = np.sqrt(3.0) * 3.1e18 * slack
    h_max = np.sqrt(a_max) * oc_max * slack
    c_max = (oc_max ** 2 + 1e18 ** 2) * slack
    disc_max = (h_max ** 2 + a_max * c_max) * slack
    root_max = (h_max + np.sqrt(disc_max)) / (a_min / slack)
    assert disc_max < 1e70 and np.isfinite(root_max), (disc_max, root_max)
    # spot check at the extremes, random directions: every intermediate finite, no NaN root
    rng = np.random.default_rng(23)
    for _ in range(2000):
        u = rng.normal(size=3)
        D = u / np.linalg.norm(u) * rng.choice([1.1e-15, 9e14])
        O = rng.choice([-1.0, 1.0], 3) * rng.choice([0.0, 1.99e18], 3)
        C = rng.choice([-1.0, 1.0], 3) * rng.choice([0.0, 9.9e17], 3)
        r = rng.choice([-9.9e17, 1.0, 9.9e17])
        oc = C - O
        a, h, c = float(D @ D), float(D @ oc), float(oc @ oc) - r * r
        disc = h * h - a * c
        assert np.isfinite(h * h) and np.isfinite(a * c) and np.isfinite(disc) and abs(disc) < disc_max
        if disc >= 0.0:
            assert np.isfinite((h - np.sqrt(disc)) / a) and np.isfinite((h + np.sqrt(disc)) / a)
    # and the fp32 test that routes a ray to the exhaustive scan brackets exactly that range of |d|
    for d, degenerate in ((1e-16, True), (1.2e-15, False), (8e14, False), (1e16, True), (0.0, True), (np.inf, True)):
        f = np.float32(d)
        with np.errstate(over="ignore", invalid="ignore"):
            l2 = f * f
        assert (not (l2 > np.float32(1e-30) and l2 < np.float32(1e30))) == degenerate, d


def test_tickets_visit_every_unit_once_from_the_last_pixel_to_the_first():
    """rtclj_kernels.cuh unit_of_ticket(): ticket -> (local pixel, chunk) with a pixel's chunks on consecutive tickets
    and the pixels handed out from the shard's last to its first (the top rows -- sky -- last, DESIGN.md section 6);
    `unit` = pixel * nchunks + chunk addresses the unit sums."""
    rng = np.random.default_rng(2)
    for _ in range(200):
        npix, nchunks = int(rng.integers(1, 400)), int(rng.integers(1, 21))
        t = np.arange(npix * nchunks, dtype=np.uint32)
        q = t // np.uint32(nchunks)
        p_local = np.uint32(npix - 1) - q
        unit = p_local * np.uint32(nchunks) + (t - q * np.uint32(nchunks))
        assert np.array_equal(np.sort(unit), t)                          # a bijection onto the unit sums
        assert np.array_equal(unit // nchunks, p_local)                  # what the kernels recover from `unit`
        assert np.all(np.diff(p_local.astype(np.int64)) <= 0) and p_local[0] == npix - 1 and p_local[-1] == 0
        same = p_local[1:] == p_local[:-1]
        assert np.all((unit[1:] - unit[:-1])[same] == 1)                 # chunks of a pixel in order
