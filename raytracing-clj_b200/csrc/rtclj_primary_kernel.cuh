// Primary-ray renders of a handful of spheres: BASELINE config 4 -- experimental.raytracing-i's normal
// shading (raytracing_i.clj:59-73, 146-163) and the full path at max-depth 1 (raytracing.clj:45-58 with
// depth = 1: a hit is black, a miss is sky).  Every sample is ONE camera ray and ONE closest-hit search, so
// none of the path machinery of render_kernel (ray state across steps, attenuation stack, material
// branches, survivor lists, refill per step) is needed: one lane owns a work unit (a pixel, or a chunk of
// its samples), loops over the samples in order with the sum in registers, and all 32 lanes of a warp run
// the same instructions.  The arithmetic is the other kernels' helper for helper (same Philox words, same
// fp64 operations in the same order), so the image is bit-identical to theirs and to the oracle (tests).
//
// The exact geometry of the <= kPrimarySpheres spheres travels in the kernel parameters (KParams::ctab is
// unused here: there is no fp32 cull), so the hot loop reads no memory at all: the sphere constants reach the
// DFMA pipe as constant-bank operands.  Bound: the fp64 pipe (B200: 64 lanes per SM) -- ~160 fp64
// instructions per sample, DESIGN.md section 4.6.
#pragma once
#include "rtclj_kernels.cuh"

namespace rtclj {

constexpr int kPrimarySpheres = 6;    // the measured crossover of scan vs cull for primary rays (rtclj_abi.cu)
#ifndef RTCLJ_PRIM_THREADS
#define RTCLJ_PRIM_THREADS 256
#endif
#ifndef RTCLJ_PRIM_MINB
#define RTCLJ_PRIM_MINB 3
#endif
#ifndef RTCLJ_PRIM_UNROLL
#define RTCLJ_PRIM_UNROLL 1
#endif
constexpr int kPrimaryThreads = RTCLJ_PRIM_THREADS;

// kSeeded: an accumulation's strict pass (rtclj_ctx_accum_step).  One unit per pixel, whose three sums start
// from the pixel's running sums P.acc instead of 0.0, so that the pass continues the sequential sum of the
// passes before it; finalize_kernel stores the unit sum back.  Its own kernel (render_primary_seeded_kernel),
// so that render_primary_kernel's code stays as it is.
// kListed: the pixels of KParams::list only (an adaptive accumulation's pass, DESIGN.md section 4.10).  Seeded and
// listed, the kernel also continues the pixel's sums of squared sample colours (KParams::acc2) in three more
// registers, in sample order, and stores them back in place: the fold's S2 in strict order without a sample buffer.
// kFrames: the units of a camera sequence, P = FP->P (render_primary_frames_kernel).  Unit u belongs to frame
// u / frame_units, tickets in unit order as here; kDefocus: some frame of the launch has the defocus disk.
template <bool kDefocus, bool kSeeded, bool kListed = false, bool kFrames = false>
__device__ __forceinline__ void render_primary_body(const KParams& P, const FrameKParams* FP = nullptr) {
  constexpr unsigned FULL = 0xffffffffu;
  constexpr bool kMoments = kSeeded && kListed;
  const int lane = threadIdx.x & 31;
  const bool normal_shading = (P.flags & F_NORMAL_SHADING) != 0;
  const double* __restrict__ G = reinterpret_cast<const double*>(P.ctab);  // [n][cx, cy, cz, r]
  const int n = P.n;
  unsigned n_samples = 0;

  for (;;) {
    // 32 consecutive work units per warp and ticket (replaces the row-chunk pool, raytracing.clj:157-171)
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(P.queue, 32ull);
    base = __shfl_sync(FULL, base, 0);
    // (listed: the count is read again per ticket -- an L1 hit; held across the sample loop it costs a spill at
    // the 80 registers of three CTAs per SM)
    const unsigned long long total_units = total_units_of<kListed>(P);
    if (base >= total_units) break;
    const unsigned long long ticket = base + (unsigned long long)lane;
    if (ticket >= total_units) continue;  // (tail of the last ticket: the lane waits at the next shuffle, which ends the loop)

    unsigned unit = (unsigned)ticket;
    const unsigned frame = kFrames ? unit / FP->frame_units : 0u;
    const unsigned frame_unit = kFrames ? unit - frame * FP->frame_units : unit;  // the unit within its frame
    const unsigned p_local = kListed ? unit_of_listed_ticket(P, (unsigned)ticket, unit) : frame_unit / (unsigned)P.nchunks;
    const int chunk = (int)((kListed ? unit : frame_unit) - p_local * (unsigned)P.nchunks);
    const int lr = (int)(p_local / (unsigned)P.W);
    const int pi = (int)(p_local - (unsigned)lr * (unsigned)P.W);
    const int tile = lr / P.shard_rows;
    const int pj = (tile * P.shard_count + P.shard_index) * P.shard_rows + (lr - tile * P.shard_rows);
    const unsigned pixel = (unsigned)pj * (unsigned)P.W + (unsigned)pi;
    const int k_begin = P.sample_base + chunk * P.spu;
    const int k_end = min(k_begin + P.spu, P.spp);
    double sum_r = 0.0, sum_g = 0.0, sum_b = 0.0;
    if (kSeeded) { const double* a = P.acc + (size_t)p_local * 3u; sum_r = a[0]; sum_g = a[1]; sum_b = a[2]; }
    double sq_r = 0.0, sq_g = 0.0, sq_b = 0.0;
    if (kMoments) { const double* a = P.acc2 + (size_t)p_local * 3u; sq_r = a[0]; sq_g = a[1]; sq_b = a[2]; }

#pragma unroll 1
    for (int k = k_begin; k < k_end; ++k) {
      // ---- camera ray: raytracing.clj:144-151, realm/raytracing.clj:332-339, raytracing_i.clj:150-158
      uint4 w = RTCLJ_PHILOX(P, pixel, (unsigned)k, 0u, 0u);
      d3 O, D;
      if (kFrames) {
        frame_camera_ray<kDefocus>(P, FP->cam[frame], pixel, pi, pj, k, w, O, D);
      } else {
        const double sx = (double)pi + (u24(w.x) - 0.5);
        const double sy = (double)pj + (u24(w.y) - 0.5);
        const d3 ps = add(add(ld3(P.p00), muls(ld3(P.du), sx)), muls(ld3(P.dv), sy));
        O = ld3(P.center);
        if (kDefocus) {  // vec3a/random-in-unit-disk, vec3a.clj:81-86
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

      // ---- closest hit over every sphere in list order (hit-anything, raytracing.clj:33-43;
      // raytracing_i.clj:48-57): the operations of exact_test_lex, geometry from the parameters, with the
      // reference's acceptance of a NaN root (scan_all_ni)
      const double a = lensq(D);
      const double ya = recip_refined(a);
      const bool a_ok = recip_safe(a);
      int best = -1;
      double closest = __longlong_as_double(0x7ff0000000000000LL);
#if RTCLJ_PRIM_UNROLL
#pragma unroll
      for (int i = 0; i < kPrimarySpheres; ++i) {
        if (i >= n) break;
#else
#pragma unroll 1
      for (int i = 0; i < n; ++i) {
#endif
        const double gr = G[4 * i + 3];
        const d3 oc = mk(G[4 * i] - O.x, G[4 * i + 1] - O.y, G[4 * i + 2] - O.z);
        const double h = dot(D, oc);
        const double c = lensq(oc) - gr * gr;
        const double disc = h * h - a * c;
        if (disc < 0.0) continue;
        const double sq = sqrt(disc);
        double root = div_by(h - sq, a, ya, a_ok);
        if (root <= 1e-3) {
          root = div_by(h + sq, a, ya, a_ok);
          if (root <= 1e-3) continue;
        }
        // list order: on an exact tie the earlier sphere stays.  `!(closest <= root)`, not `root < closest`: the
        // reference accepts a NaN root (|d|^2 = 0 or inf), and once closest is NaN every later sphere wins
        if (!(closest <= root)) { closest = root; best = i; }
      }

      // ---- colour of the sample
      d3 color = mk(0.0, 0.0, 0.0);  // a hit at max-depth 1 ends black (raytracing.clj:46-47)
      if (best < 0) {  // sky, raytracing.clj:55-58 / realm/raytracing.clj:229-236 / raytracing_i.clj:67-73
        const d3 U = divs_by(D, sqrt(a));
        const double g = 0.5 * (U.y + 1.0);
        color = mk((1.0 - g) * 1.0 + g * 0.5, (1.0 - g) * 1.0 + g * 0.7, (1.0 - g) * 1.0 + g * 1.0);
      } else if (normal_shading) {  // raytracing_i.clj:62-66
        const d3 Pt = add(O, muls(D, closest));                                                   // ray/at, ray.clj:7-8
        const d3 outward = divs_by(sub(Pt, mk(G[4 * best], G[4 * best + 1], G[4 * best + 2])), G[4 * best + 3]);  // hittable.clj:25
        const bool front = dot(D, outward) < 0.0;                                                 // hit.clj:14-15
        const d3 N = front ? outward : neg(outward);
        color = muls(add(N, mk(1.0, 1.0, 1.0)), 0.5);
      }
      sum_r = sum_r + color.x; sum_g = sum_g + color.y; sum_b = sum_b + color.z;  // raytracing.clj:153
      if (kMoments) { sq_r = sq_r + color.x * color.x; sq_g = sq_g + color.y * color.y; sq_b = sq_b + color.z * color.z; }
      n_samples++;
    }
    if (kListed) {  // the unit again from the ticket: one load per unit instead of a register (a spill) over the loop
      const unsigned q = (unsigned)ticket / (unsigned)P.nchunks;
      unit = *(volatile const unsigned*)(P.list + q) * (unsigned)P.nchunks + ((unsigned)ticket - q * (unsigned)P.nchunks);
    }
    double* out = P.partial + (size_t)unit * 3u;
    out[0] = sum_r; out[1] = sum_g; out[2] = sum_b;
    if (kMoments) { double* a = P.acc2 + (size_t)p_local * 3u; a[0] = sq_r; a[1] = sq_g; a[2] = sq_b; }
  }

  // ---- counters: samples = segments; every sphere is tested for every segment
  {
    const unsigned lo = __reduce_add_sync(FULL, n_samples & 0xffffu), hi = __reduce_add_sync(FULL, n_samples >> 16);
    if (lane == 0) {
      const unsigned long long s = (unsigned long long)lo + ((unsigned long long)hi << 16);
      atomicAdd(P.stats + 0, s);
      atomicAdd(P.stats + 1, s);
      atomicAdd(P.stats + 2, s * (unsigned long long)n);
    }
  }
}

template <bool kDefocus>  // (as a run-time branch the unused disk draw still costs its conversions: 3 % of a sample)
__global__ void __launch_bounds__(kPrimaryThreads, RTCLJ_PRIM_MINB) render_primary_kernel(const __grid_constant__ KParams P) {
  render_primary_body<kDefocus, false>(P);
}

template <bool kDefocus>
__global__ void __launch_bounds__(kPrimaryThreads, RTCLJ_PRIM_MINB) render_primary_seeded_kernel(const __grid_constant__ KParams P) {
  render_primary_body<kDefocus, true>(P);
}

template <bool kDefocus>
__global__ void __launch_bounds__(kPrimaryThreads, RTCLJ_PRIM_MINB) render_primary_listed_kernel(const __grid_constant__ KParams P) {
  render_primary_body<kDefocus, false, true>(P);
}

template <bool kDefocus>
__global__ void __launch_bounds__(kPrimaryThreads, RTCLJ_PRIM_MINB) render_primary_seeded_listed_kernel(const __grid_constant__ KParams P) {
  render_primary_body<kDefocus, true, true>(P);
}

template <bool kDefocus>
__global__ void __launch_bounds__(kPrimaryThreads, RTCLJ_PRIM_MINB) render_primary_frames_kernel(const __grid_constant__ FrameKParams FP) {
  render_primary_body<kDefocus, false, false, true>(FP.P, &FP);
}

}  // namespace rtclj
