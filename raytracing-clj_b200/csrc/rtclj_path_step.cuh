// rtclj_path_step.cuh -- everything that happens to ONE path between two culls: exact resolve of the cull
// survivors, shading, accumulation, work-unit refill and the next camera ray.  Shared by the kernels that keep
// a path's state in registers while it is processed (rtclj_lane2_kernel.cuh, rtclj_split_kernel.cuh); the
// arithmetic and its order are those of render_kernel<true> (rtclj_kernels.cuh), i.e. the reference's:
// hit-anything raytracing.clj:33-43, hittable.clj:9-31, material.clj:13-46, ray-color raytracing.clj:45-58,
// compute-pixel raytracing.clj:141-155.
#pragma once
#include "rtclj_kernels.cuh"

namespace rtclj {

// out of line: the kernels that include this must stay inside the 32 KB instruction cache
__device__ __noinline__ d3 lane2_divs_by(d3 v, double d) { return divs_by(v, d); }
// the step's merged Philox call: inline with the host's round keys (46 instructions; the out-of-line copy with
// its own key schedule is 60 + the call)
#ifndef RTCLJ_LANE2_PHILOX_INLINE
#define RTCLJ_LANE2_PHILOX_INLINE 1
#endif

// fp32 view of a ray for the conservative cull (coordinates translated by -shift); DESIGN.md "cull error bound"
struct RayView { float ofx, ofy, ofz, dhx, dhy, dhz, len32, mo, nbetaf, kqf; bool degenerate; };
__device__ __forceinline__ RayView make_view(const KParams& P, d3 O, d3 D) {
  RayView v;
  v.ofx = (float)(O.x - P.shift[0]); v.ofy = (float)(O.y - P.shift[1]); v.ofz = (float)(O.z - P.shift[2]);
  const float dfx = (float)D.x, dfy = (float)D.y, dfz = (float)D.z;
  const float l2 = dfx * dfx + dfy * dfy + dfz * dfz;
  const float inv = rsqrtf(l2);
  v.degenerate = !(l2 > 1e-30f && l2 < 1e30f);  // exact scan instead
  v.dhx = dfx * inv; v.dhy = dfy * inv; v.dhz = dfz * inv;
  v.len32 = l2 * inv;  // |d| to ~8 eps
  v.mo = fmaxf(fabsf(v.ofx), fmaxf(fabsf(v.ofy), fabsf(v.ofz)));
  //   D' = b^2 + s,  b = c.dhat - o.dhat,  s = Ws + 2 c.o - |o|^2(1 - 96 eps)
  v.nbetaf = -fmaf(v.ofz, v.dhz, fmaf(v.ofy, v.dhy, v.ofx * v.dhx));
  v.kqf = fmaf(v.ofz, v.ofz, fmaf(v.ofy, v.ofy, v.ofx * v.ofx)) * -(1.0f - 96.0f * kEps32);
  return v;
}

enum { PS_FRESH = 0, PS_RAY = 1, PS_DEAD = 2 };  // a path: needs a work unit / carries a ray / has run out of work

struct PathRegs { d3 O, D; unsigned pixel, unit; int k, k_end, depth_left, nstack, status; };
struct PathCounters { unsigned samples, seg, exact, pref; };

// bany: which cull blocks have a survivor for this path (block j at bit 32 - nconst + j);
// survivors_of_block(j): the 16 survivor bits of block j (sphere s of the block -> bit 15 - s);
// sums: the path's three unit sums, kSumStride doubles apart; stack_col: its column of the attenuation stack.
// kListed: tickets go to the pixels of KParams::list, `total_units` of them (total_units_of, read once per kernel).
// kFrames: the units of a camera sequence, P = FP->P (unit_of_frame_ticket, frame_camera_ray).
template <bool kSampleBuf, int kSumStride, bool kListed = false, bool kFrames = false, class SurvivorsOfBlock>
__device__ __forceinline__ void path_step(const KParams& P, PathRegs& pr, PathCounters& pc, unsigned bany,
                                          SurvivorsOfBlock survivors_of_block, double* sums, size_t stack_col, int lane,
                                          unsigned long long total_units = 0, const FrameKParams* FP = nullptr) {
  d3& O = pr.O; d3& D = pr.D;
  unsigned& pixel = pr.pixel; unsigned& unit = pr.unit;
  int& k = pr.k; int& k_end = pr.k_end; int& depth_left = pr.depth_left; int& nstack = pr.nstack; int& status = pr.status;
  unsigned& n_samples = pc.samples; unsigned& n_seg = pc.seg; unsigned& n_exact = pc.exact; unsigned& n_pref = pc.pref;
  const unsigned flags = P.flags;
  const bool reverse = flags & F_REVERSE_PRODUCT;
  const unsigned FULL = 0xffffffffu;
  uint4 wq = make_uint4(0u, 0u, 0u, 0u);  // block 0 of the path's next draw stage (scatter or camera)
  bool have_wq = false, need_cam = false;
  bool need_unit = status == PS_FRESH;
  if (status == PS_RAY) {
    // ---- exact closest hit (hit-anything, raytracing.clj:33-43) over the cull survivors
    const RayView vw = make_view(P, O, D);
    int best = -1;
    double closest = __longlong_as_double(0x7ff0000000000000LL);
    const double a = lensq(D);
    if ((flags & F_NO_CULL) || vw.degenerate) {  // every sphere, list order, fp64 only
#pragma unroll 1
      for (int i = 0; i < P.n; ++i) { const HitPick hp = exact_test_ni(P.geom64, i, O, D, a, closest, best); closest = hp.closest; best = hp.best; }
      n_exact += (unsigned)P.n;
    } else {
      // fp32 prefilter with rigorous bounds, then the exact test on the candidates that can still win
      const float tmin_lo = 1e-3f * vw.len32 * (1.0f - 16.0f * kEps32);
      const double ya = recip_refined(a);
      const bool a_ok = recip_safe(a);
#if !RTCLJ_PACKED_CANDS
      int c1 = -1, c2 = -1, c3 = -1;
#endif
      float lo1 = kCandEmpty, lo2 = kCandEmpty, lo3 = kCandEmpty;  // candidates (packed keys, rtclj_kernels.cuh)
      unsigned cur = 0, any = bany;
      int bbase = 0;
      const int nb_shift = 32 - P.nconst;
#pragma unroll 1
      for (;;) {
        if (cur == 0) {
          if (any == 0) break;
          const int j = (__ffs(any) - 1) - nb_shift;
          any &= any - 1;
          cur = survivors_of_block(j);  // sphere s of the block -> bit 15 - s, set = survivor
          n_pref += (unsigned)__popc(cur);
          bbase = j * 16 - 16;  // __clz counts the 16 leading zeros too
        }
        const int bit = __clz(cur);
        cur &= ~(0x80000000u >> bit);
        int i = bbase + bit;
        if (i >= P.n) continue;
        const float4 g4 = __ldg(P.geomA + i);
        const float cx = g4.x, cy = g4.y, cz = g4.z, ws = g4.w;
        const float bb = fmaf(cz, vw.dhz, fmaf(cy, vw.dhy, fmaf(cx, vw.dhx, vw.nbetaf)));
        const float ss = fmaf(cz, 2.0f * vw.ofz, fmaf(cy, 2.0f * vw.ofy, fmaf(cx, 2.0f * vw.ofx, ws + vw.kqf)));
        const float dd = fmaf(bb, bb, ss);                           // >= D_true (inflated)
        const float sq = sqrt_approx(fmaxf(dd, 0.0f)) * (1.0f + 16.0f * kEps32);
        const float eb = kEps32 * (24.0f * (fabsf(cx) + fabsf(cy) + fabsf(cz)) + 40.0f * vw.mo);
        const float far_hi = bb + sq + eb;
        float lo = bb - sq - eb;                                     // <= every root of sphere i
        const float clo_hi = __double2float_ru(closest) * vw.len32 * (1.0f + 16.0f * kEps32);
        if (far_hi < tmin_lo || lo > clo_hi) continue;
        // keep the three candidates with the smallest lower bounds, sorted; a fourth is tested on the spot
#if RTCLJ_PACKED_CANDS
        {
          const float out = cand_insert(cand_key(lo, i), lo1, lo2, lo3);
          i = out < 1.0e38f ? cand_index(out) : -1;
        }
#else
        if (lo < lo1) { const int ti = c1; const float tl = lo1; c1 = i; lo1 = lo; i = ti; lo = tl; }
        if (i >= 0 && lo < lo2) { const int ti = c2; const float tl = lo2; c2 = i; lo2 = lo; i = ti; lo = tl; }
        if (i >= 0 && lo < lo3) { const int ti = c3; const float tl = lo3; c3 = i; lo3 = lo; i = ti; lo = tl; }
#endif
        if (i >= 0) {  // (very rare)
          const HitPick hp = exact_test_lex_ni(P.geom64, i, O, D, a, ya, a_ok, closest, best);
          closest = hp.closest; best = hp.best; n_exact++;
        }
      }
#pragma unroll 1
      for (int s2 = 0; s2 < 3; ++s2) {  // one inlined test site; the others only while their bound allows a win
        const float lo_i = s2 == 0 ? lo1 : (s2 == 1 ? lo2 : lo3);
#if RTCLJ_PACKED_CANDS
        const int ci = lo_i < 1.0e38f ? cand_index(lo_i) : -1;
#else
        const int ci = s2 == 0 ? c1 : (s2 == 1 ? c2 : c3);
#endif
        if (ci < 0) break;
        if (s2 && !(lo_i <= __double2float_ru(closest) * vw.len32 * (1.0f + 16.0f * kEps32))) break;
        exact_test_lex(P.geom64, ci, O, D, a, ya, a_ok, closest, best);  // (out of line it costs 2.8 % of a bench frame)
        n_exact++;
      }
    }
    n_seg++;

    // ---- (C) shade.  kind: material id, or K_MISS / K_NORMAL / K_END
    const unsigned stage = (unsigned)(P.max_depth - depth_left) + 1u;  // number of the scatter this hit would be
    const bool hit = best >= 0;
    const MatRec* m = P.mat + (hit ? best : 0);
    int kind = hit ? ((flags & F_NORMAL_SHADING) ? K_NORMAL : m->kind) : K_MISS;
    d3 Pt = O, N = mk(0.0, 0.0, 0.0);
    bool front = false;
    if (hit) {
      const double2 g0 = __ldg(reinterpret_cast<const double2*>(P.geom64 + best));
      const double2 g1 = __ldg(reinterpret_cast<const double2*>(P.geom64 + best) + 1);
      Pt = add(O, muls(D, closest));                                  // ray/at, ray.clj:7-8
      const d3 outward = lane2_divs_by(sub(Pt, mk(g0.x, g0.y, g1.x)), g1.y);  // hittable.clj:25
      front = dot(D, outward) < 0.0;                                  // hit.clj:14-15
      N = front ? outward : neg(outward);
      // a hit with one segment left ends black (raytracing.clj:46-47)
      if (kind >= 0 && depth_left <= 1) kind = K_END;
    }
    bool done = false;
    d3 color = mk(0.0, 0.0, 0.0);
    const bool wants_unit = kind == K_LAMBERTIAN || kind == K_METAL;
    // ONE Philox call serves every lane: a lane that scatters draws block 0 of the stage; a lane whose
    // sample ends on a miss and whose unit goes on draws block 0 of its next camera ray
    double cx = 0.0, cy = 0.0, cz = 0.0, l2 = 1.0, schlick_u = 0.0;
    const bool next_cam = kind == K_MISS && k + 1 < k_end;
    if (kind >= 0 || next_cam) {
#if RTCLJ_LANE2_PHILOX_INLINE
      wq = RTCLJ_PHILOX(P, pixel, (unsigned)k + (next_cam ? 1u : 0u), next_cam ? 0u : stage, 0u);
#else
      wq = philox_ni(pixel, (unsigned)k + (next_cam ? 1u : 0u), next_cam ? 0u : stage, 0u, P.k0, P.k1);
#endif
      have_wq = next_cam;
    }
    if (kind >= 0) {
      uint4 w = wq;
      schlick_u = u24(w.x);
      if (wants_unit) {  // vec3a/random-unit-vec3 (vec3a.clj:74-79): rejection sampling
        unsigned block = 0;
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
      U = lane2_divs_by(wants_unit ? mk(cx, cy, cz) : D, sq);
    }
    if (kind == K_MISS) {
      // sky, raytracing.clj:55-58 / realm/raytracing.clj:229-236, times the attenuations of the
      // path's scattering hits in the reference's order
      const double g = 0.5 * (U.y + 1.0);
      const d3 sky = mk((1.0 - g) * 1.0 + g * 0.5, (1.0 - g) * 1.0 + g * 0.7, (1.0 - g) * 1.0 + g * 1.0);
      if (reverse) {  // ((sky*att_n)*att_{n-1})...*att_1, raytracing.clj:52-53
        color = sky;
#pragma unroll 1
        for (int s = nstack - 1; s >= 0; --s) color = mulv(color, ld3(P.mat[P.stack[(size_t)s * P.stack_stride + stack_col]].albedo));
      } else {        // ((1*att_1)*att_2)...*att_n * sky, realm/raytracing.clj:206,225,236
        d3 T = mk(1.0, 1.0, 1.0);
#pragma unroll 1
        for (int s = 0; s < nstack; ++s) T = mulv(T, ld3(P.mat[P.stack[(size_t)s * P.stack_stride + stack_col]].albedo));
        color = mulv(T, sky);
      }
      done = true;
    } else if (kind == K_NORMAL) {                   // raytracing_i.clj:62-66
      color = muls(add(N, mk(1.0, 1.0, 1.0)), 0.5);
      done = true;
    } else if (kind == K_END) {
      done = true;
    } else {
      if (kind == K_DIELECTRIC) {  // material.clj:34-46, realm/raytracing.clj:160-177
        const double ri = front ? m->albedo[0] : m->param;  // host-precomputed 1/ior | ior
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
        if (!done) P.stack[(size_t)nstack++ * P.stack_stride + stack_col] = (unsigned short)best;
      }
      O = Pt;
      depth_left--;
    }
    if (done) {
      status = PS_FRESH;  // no ray until the camera gives it one
      if (kSampleBuf) {  // strict order: the sample's colour is stored, finalize_kernel adds in sample order
        store_sample(P, unit, k, color);
        if (++k == k_end) need_unit = true; else need_cam = true;
      } else {
        const double sum_r = sums[0] + color.x, sum_g = sums[kSumStride] + color.y, sum_b = sums[2 * kSumStride] + color.z;  // raytracing.clj:153
        sums[0] = sum_r; sums[kSumStride] = sum_g; sums[2 * kSumStride] = sum_b;
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

  // ---- refill: ballot-compacted tickets from the global work queue (replaces the reference's
  // row-chunk pool, raytracing.clj:157-171)
  {
    const unsigned mask = __ballot_sync(FULL, need_unit);
    if (mask) {
      const int leader = __ffs(mask) - 1;
      unsigned long long base = 0;
      if (lane == leader) base = atomicAdd(P.queue, (unsigned long long)__popc(mask));
      base = __shfl_sync(FULL, base, leader);
      if (need_unit) {
        const unsigned long long ticket = base + (unsigned long long)__popc(mask & ((1u << lane) - 1u));
        if (ticket >= (kListed ? total_units : P.total_units)) {
          status = PS_DEAD;
        } else {
          int chunk = 0;
          const unsigned p_local = kFrames ? unit_of_frame_ticket(*FP, (unsigned)ticket, unit, chunk)
                                   : kListed ? unit_of_listed_ticket(P, (unsigned)ticket, unit)
                                             : unit_of_ticket(P, (unsigned)ticket, unit);
          if (!kFrames) chunk = (int)(unit - p_local * (unsigned)P.nchunks);
          const int lr = (int)(p_local / (unsigned)P.W);
          const int pi = (int)(p_local - (unsigned)lr * (unsigned)P.W);
          const int tile = lr / P.shard_rows;
          const int pj = (tile * P.shard_count + P.shard_index) * P.shard_rows + (lr - tile * P.shard_rows);
          pixel = (unsigned)pj * (unsigned)P.W + (unsigned)pi;
          k = P.sample_base + chunk * P.spu;
          k_end = min(k + P.spu, P.spp);
          sums[0] = 0.0; sums[kSumStride] = 0.0; sums[2 * kSumStride] = 0.0;
          need_cam = true;
        }
      }
    }
  }

  // ---- camera ray: raytracing.clj:144-151, realm/raytracing.clj:332-339
  if (need_cam) {
    status = PS_RAY;
    uint4 w = wq;  // usually drawn by the merged call above; a new unit / an absorbed path draws here
    if (!have_wq) w = philox_ni(pixel, (unsigned)k, 0u, 0u, P.k0, P.k1);
    const unsigned pj = pixel / (unsigned)P.W, pi = pixel - pj * (unsigned)P.W;
    if (kFrames) {
      frame_camera_ray<true>(P, FP->cam[unit / FP->frame_units], pixel, (int)pi, (int)pj, k, w, O, D);
    } else {
      const double sx = (double)pi + (u24(w.x) - 0.5);
      const double sy = (double)pj + (u24(w.y) - 0.5);
      const d3 ps = add(add(ld3(P.p00), muls(ld3(P.du), sx)), muls(ld3(P.dv), sy));
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
    }
    depth_left = P.max_depth;
    nstack = 0;
    n_samples++;
  }
}

}  // namespace rtclj
