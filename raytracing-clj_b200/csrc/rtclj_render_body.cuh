// rtclj_render_body.cuh -- the body of render_kernel, render_listed_kernel and render_frames_kernel (rtclj_kernels.cuh),
// included inside each __global__ function, which defines kConstTab, kSampleBuf, kPacked and kListed and its parameter P
// (render_frames_kernel: FP, whose P it is, and RTCLJ_FRAMES_BODY, so the other kernels compile from unchanged text).
// Textual rather than a shared __forceinline__ device function: inlined, the body compiled to different code for
// the 512-thread instantiation (the launch bounds no longer bound threadIdx.x where it is read, and loops were
// rotated differently), whereas render_kernel must stay the kernel that was measured (DESIGN.md section 4.10).
// No include guard: included once per kernel.
  constexpr int kT = threads_of(kConstTab, kPacked);
  // the listed tickets, read once (32 bits: the host keeps a launch below 2^32 units)
  const unsigned listed_units = kListed ? (unsigned)total_units_of<true>(P) : 0u;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const unsigned tab_bytes = kConstTab ? 0u : P.geom_bytes;  // the table is in shared memory only in that mode
  unsigned* lists = reinterpret_cast<unsigned*>(smem_raw + tab_bytes);
  const unsigned smem_base = (unsigned)__cvta_generic_to_shared(smem_raw);
  const unsigned list_bytes = (kConstTab ? 33u : (unsigned)kListCap) * kT * 4u;  // masks[33] or entries[kListCap] per lane
  const unsigned bar = smem_base + tab_bytes + list_bytes;
  const int tid = threadIdx.x, lane = tid & 31;
  const unsigned gtid = blockIdx.x * kT + tid;

  // ---- stage the fp32 sphere table into shared memory: one TMA bulk copy per 32 KB
  if (!kConstTab && P.geom_bytes) {
    if (tid == 0) mbar_init(bar, 1);
    __syncthreads();
    if (tid == 0) {
      mbar_expect_tx(bar, P.geom_bytes);
      for (unsigned off = 0; off < P.geom_bytes; off += 32768u) {
        unsigned sz = P.geom_bytes - off < 32768u ? P.geom_bytes - off : 32768u;
        bulk_g2s(smem_base + off, reinterpret_cast<const unsigned char*>(P.geom32) + off, sz, bar);
      }
    }
    mbar_wait(bar, 0);
  }

  const unsigned flags = P.flags;
  const bool reverse = flags & F_REVERSE_PRODUCT;
  const unsigned FULL = 0xffffffffu;

  bool active = true, need_unit = true, need_cam = false, has_ray = false;
  unsigned unit = 0;  // work-unit ticket (the host guarantees total_units < 2^32)
  unsigned pixel = 0;
  int pi = 0, pj = 0, k = 0, k_end = 0;
  // unit sum (3 doubles per lane) lives in shared memory: touched once per sample, and six
  // registers fewer are live across the cull
  double* sums = reinterpret_cast<double*>(smem_raw + tab_bytes + list_bytes + 16) + tid;
  d3 O = mk(0.0, 0.0, 0.0), D = mk(0.0, 0.0, 1.0);
  d3 T = mk(1.0, 1.0, 1.0);
  int depth_left = 0, nstack = 0;
  unsigned stage = 0;
  unsigned n_samples = 0, n_seg = 0, n_exact = 0, n_ovf = 0, n_pref = 0;

  for (;;) {
    uint4 wq = make_uint4(0u, 0u, 0u, 0u);  // block 0 of the lane's next draw stage (scatter or camera)
    bool have_wq = false;
    if (__any_sync(FULL, has_ray)) {  // false only on the very first pass
    // ---- fp32 view of the ray for the cull (coordinates translated by -shift)
    int cnt = 0;
    bool scan_all = (flags & F_NO_CULL) != 0;
    const float ofx = (float)(O.x - P.shift[0]), ofy = (float)(O.y - P.shift[1]), ofz = (float)(O.z - P.shift[2]);
    float dhx, dhy, dhz, len32;
    {
      const float dfx = (float)D.x, dfy = (float)D.y, dfz = (float)D.z;
      const float l2 = dfx * dfx + dfy * dfy + dfz * dfz;
      const float inv = rsqrtf(l2);
      if (!(l2 > 1e-30f && l2 < 1e30f)) scan_all = true;  // degenerate direction: exact scan
      dhx = dfx * inv; dhy = dfy * inv; dhz = dfz * inv;
      len32 = l2 * inv;  // |d| to ~8 eps
    }
    const float mo = fmaxf(fabsf(ofx), fmaxf(fabsf(ofy), fabsf(ofz)));
    // Conservative discriminant in EXPANDED form (8 packed ops per sphere pair, no C - O):
    //   D' = b^2 + s,  b = c.dhat - o.dhat,  s = Ws + 2 c.o - |o|^2(1 - 96 eps)
    // with c = C - shift, o = O - shift in fp32 and Ws = r^2(1+8eps) - |c|^2(1 - 96 eps) from the
    // host.  D' >= D_true because the total fp32 error is below 76 eps (|c|^2 + |o|^2) + 5 eps r^2
    // (DESIGN.md "cull error bound"); 96 leaves a margin.
    const float nbetaf = -fmaf(ofz, dhz, fmaf(ofy, dhy, ofx * dhx));
    const float kqf = fmaf(ofz, ofz, fmaf(ofy, ofy, ofx * ofx)) * -(1.0f - 96.0f * kEps32);
    // ---- (A)+(B): cull a stretch of blocks into the survivor list, resolve the list exactly,
    // and continue only if the list filled up before the last block (rare "flush").
    int best = -1;
    double closest = __longlong_as_double(0x7ff0000000000000LL);
    const double a = lensq(D);
    const float tmin_lo = 1e-3f * len32 * (1.0f - 16.0f * kEps32);  // t_min in arc-length units, lower bound
    int blk = 0;                         // next full 16-pair block to cull (half-block index = 2*blk)
    unsigned blkany = 0;                 // constant-table path: which blocks have a survivor (top bits)
    bool tail_done = P.tail8 == 0;
    const bool do_cull = (flags & F_NO_CULL) == 0;
#pragma unroll 1
    for (;;) {
      cnt = 0;
      if (do_cull) {
        // One block = 16 sphere pairs.  Each packed discriminant shifts its two sign bits into
        // `acc` (sphere s of the block -> bit 31-s).  The "did anything survive" branch looks at
        // the PREVIOUS block's mask, which has long been ready, so neither it nor the counted
        // back edge stalls the FFMA2 stream; a block with survivors costs two predicated stores.
        const f32x2 nbeta = splat2(nbetaf), kq = splat2(kqf);
        const f32x2 o2x = splat2(2.0f * ofx), o2y = splat2(2.0f * ofy), o2z = splat2(2.0f * ofz);
        const f32x2 dx2 = splat2(dhx), dy2 = splat2(dhy), dz2 = splat2(dhz);
        unsigned* my_list = lists + tid;
        auto record = [&](unsigned hi16, unsigned lo16, int h) {
          if (scan_all) return;  // a degenerate ray ignores the cull (exhaustive fp64 scan below)
          if (hi16) my_list[cnt++ * kT] = ((unsigned)h << 16) | hi16;
          if (lo16) my_list[cnt++ * kT] = ((unsigned)(h + 1) << 16) | lo16;
        };
        auto pairs = [&](int pair, unsigned& acc) {  // `pair` is warp-uniform
          f32x2 cx, cy, cz, rs;
          if (kConstTab) {
            const uint4 u = P.ctab[2 * pair], v = P.ctab[2 * pair + 1];
            cx = ((f32x2)u.y << 32) | u.x; cy = ((f32x2)u.w << 32) | u.z;
            cz = ((f32x2)v.y << 32) | v.x; rs = ((f32x2)v.w << 32) | v.z;
          } else {
            lds_pair(smem_base + 32u * (unsigned)pair, cx, cy);
            lds_pair(smem_base + 32u * (unsigned)pair + 16u, cz, rs);
          }
          const f32x2 bb = fma2(cz, dz2, fma2(cy, dy2, fma2(cx, dx2, nbeta)));
          const f32x2 ss = fma2(cz, o2z, fma2(cy, o2y, fma2(cx, o2x, add2(rs, kq))));
          const f32x2 dd = fma2(bb, bb, ss);
          acc = __funnelshift_l((unsigned)dd, acc, 1);
          acc = __funnelshift_l((unsigned)(dd >> 32), acc, 1);
        };
        // scenes larger than the shared-memory budget: the pairs that did not fit are read from
        // global memory (warp-uniform address, L1/L2) -- slower, but any list up to 65 532 spheres runs
        auto pairs_global = [&](int pair, unsigned& acc) {
          const ulonglong2 u = __ldg(reinterpret_cast<const ulonglong2*>(P.geom32) + 2 * (size_t)pair);
          const ulonglong2 v = __ldg(reinterpret_cast<const ulonglong2*>(P.geom32) + 2 * (size_t)pair + 1);
          const f32x2 bb = fma2(v.x, dz2, fma2(u.y, dy2, fma2(u.x, dx2, nbeta)));
          const f32x2 ss = fma2(v.x, o2z, fma2(u.y, o2y, fma2(u.x, o2x, add2(v.y, kq))));
          const f32x2 dd = fma2(bb, bb, ss);
          acc = __funnelshift_l((unsigned)dd, acc, 1);
          acc = __funnelshift_l((unsigned)(dd >> 32), acc, 1);
        };
        unsigned acc_prev = 0xffffffffu;
        if (kConstTab) {
          // Small scenes (<= 32 blocks): the table sits in constant memory and reaches FFMA2 as
          // UNIFORM register operands (LDCU -> UR.F32x2), which costs no per-lane register-file
          // write bandwidth.  ptxas keeps the loads uniform only while the loop body stores to
          // warp-uniform-indexed addresses, so every block's 32-bit survivor mask is stored
          // unconditionally (one STS) and `blkany` remembers which blocks have a survivor; there is
          // no list, no branch and no overflow on this path.
          const int nhb = P.nconst;  // blocks of kCBP pairs on this path, <= 32
#pragma unroll 1  // (unrolling by 2 was measured: 7 % slower -- the 64 uniform registers of a block are all live)
          for (int ub = 0; ub < nhb; ++ub) {
            unsigned acc = 0xffffffffu;
#pragma unroll
            for (int p = 0; p < kCBP; ++p) pairs(ub * kCBP + p, acc);
            // kCBP == 8: 16 sign bits in the low half (sphere s -> bit 15-s) under 16 ones from the initial value
            my_list[ub * kT] = acc;
            blkany = (blkany >> 1) | (acc != 0xffffffffu ? 0x80000000u : 0u);
          }
          blk = P.nblocks;
          tail_done = true;
        } else {
          // stop early when this lane's list lacks room for the pending block (2 entries) plus the
          // one computed next (2 entries); the lane then resolves what it has and comes back (rare)
          const int blk_smem_end = min(P.nblocks, P.smem_blocks);
#pragma unroll 1
          while (blk < blk_smem_end && cnt <= kListCap - 4) {  // blocks resident in shared memory
            unsigned acc = 0xffffffffu;
#pragma unroll
            for (int p = 0; p < kBlockPairs; ++p) pairs(blk * kBlockPairs + p, acc);
            if (acc_prev != 0xffffffffu) record(~acc_prev >> 16, ~acc_prev & 0xffffu, 2 * blk - 2);
            acc_prev = acc;
            ++blk;
          }
#pragma unroll 1
          while (blk >= blk_smem_end && blk < P.nblocks && cnt <= kListCap - 4) {  // the overflow, from global memory
            unsigned acc = 0xffffffffu;
#pragma unroll 4
            for (int p = 0; p < kBlockPairs; ++p) pairs_global(blk * kBlockPairs + p, acc);
            if (acc_prev != 0xffffffffu) record(~acc_prev >> 16, ~acc_prev & 0xffffu, 2 * blk - 2);
            acc_prev = acc;
            ++blk;
          }
        }
        if (!kConstTab && acc_prev != 0xffffffffu) record(~acc_prev >> 16, ~acc_prev & 0xffffu, 2 * blk - 2);
        if (!kConstTab && blk == P.nblocks && !tail_done && cnt <= kListCap - 1) {
          unsigned acc_tail = 0xffffffffu;  // last half block: 8 pairs, 16 sign bits in the low half
          if (P.nblocks < P.smem_blocks) {
#pragma unroll
            for (int p = 0; p < kBlockPairs / 2; ++p) pairs(P.nblocks * kBlockPairs + p, acc_tail);
          } else {
#pragma unroll 4
            for (int p = 0; p < kBlockPairs / 2; ++p) pairs_global(P.nblocks * kBlockPairs + p, acc_tail);
          }
          tail_done = true;
          if (acc_tail != 0xffffffffu) record(~acc_tail & 0xffffu, 0u, 2 * P.nblocks);
        }
      }

      if (has_ray) {
        // ---- (B) exact closest hit (hit-anything, raytracing.clj:33-43 = Ray.hitAnything
        // realm/raytracing.clj:192-203) over the cull survivors.
        if (scan_all) {  // degenerate direction or RTCLJ_F_NO_CULL: every sphere, list order, fp64 only
          { const HitPick hp = scan_all_ni(P.geom64, P.n, O, D, a, closest, best); closest = hp.closest; best = hp.best; }
          n_exact += (unsigned)P.n;
        } else {
          // Pass 1 (fp32, rigorous bounds, DESIGN.md): drop survivors certainly behind the origin
          // or beyond closest-so-far; keep the two with the smallest lower bound on their root.
          // Then ONE exact test, warp-convergent, on the likeliest winner; the runner-up only if
          // its bound still allows it to win.  Anything displaced is tested on the spot (rare).
          const double ya = recip_refined(a);  // every root of this segment divides by a = |d|^2
          const bool a_ok = recip_safe(a);
          int c1 = -1, c2 = -1, c3 = -1;
          float lo1 = 3.0e38f, lo2 = 3.0e38f, lo3 = 3.0e38f;  // (kPacked: the packed keys)
          int e = 0, base = 0;     // entry cursor and the sphere index of bit 15 of `cur`
          unsigned cur = 0;        // survivor bits of the current entry still to visit
          // constant-table path: walk the blocks flagged in `blkany` (block j sits at bit
          // 32 - nblocks_total + j) and the clear bits of their stored masks (sphere s -> bit 2 kCBP - 1 - s)
          unsigned any = blkany;
          const int nb_shift = 32 - P.nconst;
#pragma unroll 1
          for (;;) {
            int i;
            if (kConstTab) {
              if (cur == 0) {
                if (any == 0) break;
                const int j = (__ffs(any) - 1) - nb_shift;
                any &= any - 1;
                cur = ~lists[j * kT + tid];
                n_pref += (unsigned)__popc(cur);  // counted per block, not per survivor: one add instead of a live counter in the walk
                base = j * (2 * kCBP) - (32 - 2 * kCBP);  // __clz counts the (32 - 2 kCBP) leading zeros too
              }
              const int bit = __clz(cur);
              cur &= ~(0x80000000u >> bit);
              i = base + bit;
            } else {
              if (cur == 0) {
                if (e >= cnt) break;
                const unsigned ent = lists[e++ * kT + tid];
                cur = ent & 0xffffu;
                n_pref += (unsigned)__popc(cur);
                base = (int)(ent >> 16) * 16 + 15;
              }
              const int b = 31 - __clz(cur);
              cur &= ~(1u << b);
              i = base - b;
            }
            if (i >= P.n) continue;
            float cx, cy, cz, ws;
            if (kConstTab) {  // per-lane index: read the same table through L1 instead
              const float4 g = __ldg(P.geomA + i);
              cx = g.x; cy = g.y; cz = g.z; ws = g.w;
            } else if ((i >> 5) < P.smem_blocks) {
              const unsigned pa = smem_base + (unsigned)(i >> 1) * 32u + (unsigned)(i & 1) * 4u;
              cx = lds_f32(pa); cy = lds_f32(pa + 8u); cz = lds_f32(pa + 16u); ws = lds_f32(pa + 24u);
            } else {  // beyond the shared-memory part of the table
              const float4 g = __ldg(P.geomA + i);
              cx = g.x; cy = g.y; cz = g.z; ws = g.w;
            }
            const float bb = fmaf(cz, dhz, fmaf(cy, dhy, fmaf(cx, dhx, nbetaf)));
            const float ss = fmaf(cz, 2.0f * ofz, fmaf(cy, 2.0f * ofy, fmaf(cx, 2.0f * ofx, ws + kqf)));
            const float dd = fmaf(bb, bb, ss);                           // >= D_true (inflated)
            const float sq = sqrt_approx(fmaxf(dd, 0.0f)) * (1.0f + 16.0f * kEps32);
            // |b32 - b_true| <= 12 eps (|c| + |o|); the sums below add <= 6 eps (|c| + |o|) more
            const float eb = kEps32 * (24.0f * (fabsf(cx) + fabsf(cy) + fabsf(cz)) + 40.0f * mo);
            const float far_hi = bb + sq + eb;
            float lo = bb - sq - eb;                                     // <= every root of sphere i
            const float clo_hi = __double2float_ru(closest) * len32 * (1.0f + 16.0f * kEps32);
            if (far_hi < tmin_lo || lo > clo_hi) continue;
            // keep the three candidates with the smallest lower bounds, sorted; a fourth is tested on the spot
            if (kPacked) {
              const float out = cand_insert(cand_key(lo, i), lo1, lo2, lo3);
              i = out < 1.0e38f ? cand_index(out) : -1;
            } else {
              if (lo < lo1) { const int ti = c1; const float tl = lo1; c1 = i; lo1 = lo; i = ti; lo = tl; }
              if (i >= 0 && lo < lo2) { const int ti = c2; const float tl = lo2; c2 = i; lo2 = lo; i = ti; lo = tl; }
              if (RTCLJ_LANE_CANDS > 2 && i >= 0 && lo < lo3) { const int ti = c3; const float tl = lo3; c3 = i; lo3 = lo; i = ti; lo = tl; }
            }
            if (i >= 0) {  // (rare)
              const HitPick hp = exact_test_lex_ni(P.geom64, i, O, D, a, ya, a_ok, closest, best);
              closest = hp.closest; best = hp.best; n_exact++;
            }
          }
#pragma unroll 1
          for (int s2 = 0; s2 < RTCLJ_LANE_CANDS; ++s2) {  // one inlined test site; the others only while their bound allows a win
            const float lo_i = s2 == 0 ? lo1 : (s2 == 1 ? lo2 : lo3);
            const int ci = kPacked ? (lo_i < 1.0e38f ? cand_index(lo_i) : -1)
                                                             : (s2 == 0 ? c1 : (s2 == 1 ? c2 : c3));
            if (ci < 0) break;
            if (s2 && !(lo_i <= __double2float_ru(closest) * len32 * (1.0f + 16.0f * kEps32))) break;
            exact_test_lex(P.geom64, ci, O, D, a, ya, a_ok, closest, best);
            n_exact++;
          }
        }
      }
      if (kConstTab || !do_cull || (blk == P.nblocks && tail_done)) break;
      n_ovf++;  // some lane's list filled up: resolved what we had, cull the remaining blocks
    }

    if (has_ray) {
      n_seg++;

      // ---- (C) shade.  kind: material id, or K_MISS / K_NORMAL / K_END
      const bool hit = best >= 0;
      const MatRec* m = P.mat + (hit ? best : 0);
      int kind = hit ? ((flags & F_NORMAL_SHADING) ? K_NORMAL : m->kind) : K_MISS;
      d3 Pt = O, N = mk(0.0, 0.0, 0.0);
      bool front = false;
      if (hit) {
        const double2 g0 = __ldg(reinterpret_cast<const double2*>(P.geom64 + best));
        const double2 g1 = __ldg(reinterpret_cast<const double2*>(P.geom64 + best) + 1);
        Pt = add(O, muls(D, closest));                                  // ray/at, ray.clj:7-8
        const d3 outward = divs_by(sub(Pt, mk(g0.x, g0.y, g1.x)), g1.y);  // hittable.clj:25
        front = dot(D, outward) < 0.0;                                  // hit.clj:14-15
        N = front ? outward : neg(outward);
        // A hit with one segment left ends black (raytracing.clj:46-47); the scatter draws the
        // reference still makes there are unobservable with a counter-based stream.
        if (kind >= 0 && depth_left <= 1) kind = K_END;
      }
      bool done = false;
      d3 color = mk(0.0, 0.0, 0.0);
      const bool wants_unit = kind == K_LAMBERTIAN || kind == K_METAL;
      // ONE Philox call serves every lane: a lane that scatters draws block 0 of stage = hit number
      // (unit-vector candidates / Schlick); a lane whose sample ends on a miss and whose unit goes
      // on draws block 0 of the camera stage of its next sample, consumed further down.
      double cx = 0.0, cy = 0.0, cz = 0.0, l2 = 1.0, schlick_u = 0.0;
      const bool next_cam = kind == K_MISS && k + 1 < k_end;
      if (kind >= 0) stage++;
      if (kind >= 0 || next_cam) {
        wq = RTCLJ_PHILOX(P, pixel, (unsigned)k + (next_cam ? 1u : 0u), next_cam ? 0u : stage, 0u);
        have_wq = next_cam;
      }
      if (kind >= 0) {
        uint4 w = wq;
        schlick_u = u24(w.x);
        if (wants_unit) {  // vec3a/random-unit-vec3 (vec3a.clj:74-79): rejection sampling; block n holds
          unsigned block = 0;  // candidates 2n (words 0,1) and 2n+1 (words 2,3), 3 x 21 bits each
          int half = 0;
#pragma unroll 1
          for (;;) {
            const unsigned wa = half ? w.z : w.x, wb = half ? w.w : w.y;
            cx = sym21(wa & 0x1fffffu);
            cy = sym21((wa >> 21) | ((wb & 0x3ffu) << 11));
            cz = sym21((wb >> 10) & 0x1fffffu);
            l2 = cx * cx + cy * cy + cz * cz;
            if ((l2 > 1e-160 && l2 <= 1.0) || block == 0xffffffu) break;
            if (half == 0) { half = 1; continue; }
            half = 0;
            w = philox_ni(pixel, (unsigned)k, stage, ++block, P.k0, P.k1);
          }
        }
      }
      // one sqrt and one 3-way divide serve every kind: unit candidate / |d| normalisation
      d3 U = mk(0.0, 0.0, 0.0);
      if (kind >= 0 || kind == K_MISS) {
        const double sq = dsqrt(wants_unit ? l2 : a);
        U = divs_by(wants_unit ? mk(cx, cy, cz) : D, sq);
      }
      if (kind == K_MISS) {
        // sky, raytracing.clj:55-58 / realm/raytracing.clj:229-236
        const double g = 0.5 * (U.y + 1.0);
        d3 sky = mk((1.0 - g) * 1.0 + g * 0.5, (1.0 - g) * 1.0 + g * 0.7, (1.0 - g) * 1.0 + g * 1.0);
        if (reverse) {  // ((sky*att_n)*att_{n-1})...*att_1, raytracing.clj:52-53
          color = sky;
#pragma unroll 1
          for (int s = nstack - 1; s >= 0; --s) {
            const int b = P.stack[(size_t)s * P.stack_stride + gtid];
            color = mulv(color, ld3(P.mat[b].albedo));
          }
        } else {
          color = mulv(T, sky);  // realm/raytracing.clj:236
        }
        done = true;
      } else if (kind == K_NORMAL) {                   // raytracing_i.clj:62-66
        color = muls(add(N, mk(1.0, 1.0, 1.0)), 0.5);
        done = true;
      } else if (kind == K_END) {
        done = true;
      } else {
        if (kind == K_DIELECTRIC) {  // material.clj:34-46, realm/raytracing.clj:160-177
          // albedo[] of a dielectric record holds host-precomputed 1/ior and the two Schlick
          // ratios (1-ri)/(1+ri) for ri = 1/ior and ri = ior (same IEEE operations, done once)
          const double ri = front ? m->albedo[0] : m->param;
          const double cos_t = jmin1(dot(neg(U), N));
          const double sin_t = dsqrt(1.0 - cos_t * cos_t);
          bool do_reflect = ri * sin_t > 1.0;
          if (!do_reflect && (flags & F_SCHLICK)) {  // `or` short-circuits, material.clj:42
            const double q = front ? m->albedo[1] : m->albedo[2];  // material/reflectance, material.clj:30-32
            const double r0 = q * q;
            const double mm = 1.0 - cos_t;
            const double m2 = mm * mm;
            const double m5 = m2 * m2 * mm;
            do_reflect = (r0 + (1.0 - r0) * m5) > schlick_u;
          }
          if (do_reflect) {  // vec3a/reflect, vec3a.clj:94-95
            D = sub(U, muls(N, 2.0 * dot(U, N)));
          } else {           // vec3a/refract, vec3a.clj:97-101
            const d3 perp = muls(add(U, muls(N, cos_t)), ri);
            const d3 para = muls(N, -dsqrt(fabs(1.0 - lensq(perp))));
            D = add(perp, para);
          }
        } else {
          if (kind == K_LAMBERTIAN) {  // material.clj:13-19, realm/raytracing.clj:138-145
            d3 s = add(U, N);
            if ((flags & F_NEAR_ZERO_GUARD) && fabs(s.x) < 1e-8 && fabs(s.y) < 1e-8 && fabs(s.z) < 1e-8) s = N;
            D = s;
          } else {                     // material.clj:21-28, realm/raytracing.clj:147-158
            d3 refl = sub(D, muls(N, 2.0 * dot(D, N)));
            refl = add(muls(U, m->param), refl);
            if (!(dot(refl, N) > 0.0)) done = true;  // absorbed -> black
            D = refl;
          }
          if (!done) {
            if (reverse) P.stack[(size_t)nstack++ * P.stack_stride + gtid] = (unsigned short)best;
            else T = mulv(T, ld3(m->albedo));  // realm/raytracing.clj:225
          }
        }
        O = Pt;
        depth_left--;
      }
      if (done) {
        has_ray = false;
        if (kSampleBuf) {  // strict order: the sample's colour is stored, finalize_kernel adds in sample order
          store_sample(P, unit, k, color);
          if (++k == k_end) need_unit = true; else need_cam = true;
        } else {
          const double sum_r = sums[0] + color.x, sum_g = sums[kT] + color.y, sum_b = sums[2 * kT] + color.z;  // raytracing.clj:153
          sums[0] = sum_r; sums[kT] = sum_g; sums[2 * kT] = sum_b;
          if (++k == k_end) {
            double* out = P.partial + (size_t)unit * 3u;
            out[0] = sum_r; out[1] = sum_g; out[2] = sum_b;
            need_unit = true;
          } else {
            need_cam = true;
          }
        }
      }
    }
    }  // any lane had a ray

    // ---- refill: ballot-compacted tickets from the global work queue
    {
      const bool want = active && need_unit;
      const unsigned mask = __ballot_sync(FULL, want);
      if (mask) {
        const int leader = __ffs(mask) - 1;
        unsigned long long base = 0;
        if (lane == leader) base = atomicAdd(P.queue, (unsigned long long)__popc(mask));
        base = __shfl_sync(FULL, base, leader);
        if (want) {
          const unsigned long long ticket = base + (unsigned long long)__popc(mask & ((1u << lane) - 1u));
          need_unit = false;
          if (ticket >= (kListed ? (unsigned long long)listed_units : P.total_units)) {
            active = false;
          } else {
#if RTCLJ_FRAMES_BODY
            int chunk;
            const unsigned p_local = unit_of_frame_ticket(FP, (unsigned)ticket, unit, chunk);
#else
            const unsigned p_local = kListed ? unit_of_listed_ticket(P, (unsigned)ticket, unit)
                                             : unit_of_ticket(P, (unsigned)ticket, unit);
            const int chunk = (int)(unit - p_local * (unsigned)P.nchunks);
#endif
            const int lr = (int)(p_local / (unsigned)P.W);
            pi = (int)(p_local - (unsigned)lr * (unsigned)P.W);
            const int tile = lr / P.shard_rows;
            pj = (tile * P.shard_count + P.shard_index) * P.shard_rows + (lr - tile * P.shard_rows);
            pixel = (unsigned)pj * (unsigned)P.W + (unsigned)pi;
            k = P.sample_base + chunk * P.spu;
            k_end = min(k + P.spu, P.spp);
            sums[0] = 0.0; sums[kT] = 0.0; sums[2 * kT] = 0.0;
            need_cam = true;
          }
        }
      }
      // (aligning the phases of all warps with a CTA barrier here was measured: 22 % slower)
      if (!__any_sync(FULL, active)) break;
    }

    // ---- camera ray: raytracing.clj:144-151, realm/raytracing.clj:332-339
    if (active && need_cam) {
      need_cam = false;
      has_ray = true;
      uint4 w = wq;  // usually drawn by the merged call above; a new unit / an absorbed path draws here
      if (!have_wq) w = philox_ni(pixel, (unsigned)k, 0u, 0u, P.k0, P.k1);
#if RTCLJ_FRAMES_BODY
      frame_camera_ray<true>(P, FP.cam[unit / FP.frame_units], pixel, pi, pj, k, w, O, D);
#else
      const double sx = (double)pi + (u24(w.x) - 0.5);
      const double sy = (double)pj + (u24(w.y) - 0.5);
      d3 ps = add(add(ld3(P.p00), muls(ld3(P.du), sx)), muls(ld3(P.dv), sy));
      O = ld3(P.center);
      if (P.use_defocus) {  // vec3a/random-in-unit-disk, vec3a.clj:81-86
        double px = sym24(w.z), py = sym24(w.w);
        unsigned block = 0;
        int half = 1;
        while (!(px * px + py * py < 1.0) && block < 0xffffffu) {
          if (half == 1) { w = philox_ni(pixel, (unsigned)k, 0u, ++block, P.k0, P.k1); half = 0; } else half = 1;
          px = sym24(half ? w.z : w.x);
          py = sym24(half ? w.w : w.y);
        }
        O = add(add(O, muls(ld3(P.ddu), px)), muls(ld3(P.ddv), py));  // raytracing.clj:89-93
      }
      D = sub(ps, O);
#endif
      depth_left = P.max_depth;
      stage = 0;
      nstack = 0;
      T = mk(1.0, 1.0, 1.0);
      n_samples++;
    }

  }

  // ---- counters: REDUX on 16-bit halves (each lane's count fits 32 bits), one atomic per warp
  {
    const unsigned v[5] = {n_samples, n_seg, n_exact, n_ovf, n_pref};
#pragma unroll 1
    for (int q = 0; q < 5; ++q) {
      const unsigned lo = __reduce_add_sync(FULL, v[q] & 0xffffu), hi = __reduce_add_sync(FULL, v[q] >> 16);
      if (lane == 0) atomicAdd(P.stats + q, (unsigned long long)lo + ((unsigned long long)hi << 16));
    }
  }
