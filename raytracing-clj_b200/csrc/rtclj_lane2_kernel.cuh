// rtclj_lane2_kernel.cuh -- render_kernel<true> (one path per lane, rtclj_kernels.cuh) with TWO paths per
// lane, for scenes of <= 512 spheres (BASELINE.json configs 1-4).
//
// Why: the cull is 62 % of the instructions of a frame, and a quarter of the cull's instructions are
// the uniform loads that bring a sphere pair into uniform registers (32 LDCU.64 per 16 spheres).  With two
// rays per lane every loaded pair feeds two rays: 103 instead of 123 instructions per 16 spheres x 32 rays
// (tools/microbench/cull_loop8), and the two independent FFMA2 chains let a single warp keep the FMA
// pipe busy (one warp culling alone reaches only half the FFMA2 rate).  Resolve / shade / sampling stay
// exactly the code of render_kernel<true>, run for path 0 and then for path 1: the path that is not being
// processed waits in shared memory (76 bytes), the two are swapped between the passes.
// The cull has two levels (DESIGN.md 4.2): both lines against one bounding record per group of 16 spheres (uniform
// operands), then each lane against the members of the groups its lines reach -- the flat cull's survivors.  The
// camera-sequence twins keep the flat cull.
//
// Reference: src/raytracing.clj:141-171, src/realm/raytracing.clj:325-346 and the functions they call
// (cited at each step below).  Arithmetic, draw order and results are those of render_kernel<true>.
#pragma once
#include "rtclj_path_step.cuh"

namespace rtclj {

#ifndef RTCLJ_LANE2_THREADS
#define RTCLJ_LANE2_THREADS 640
#endif
constexpr int kT2 = RTCLJ_LANE2_THREADS;


// dynamic shared memory layout (bytes)
// (unit sums accumulating in global memory instead -- 30 KB less shared memory, 96 instead of 64 KB of L1 --
// were measured: 552.5 against 543.7 ms per bench frame)
struct Lane2Smem {
  static constexpr size_t masks = 0;                                   // 32 blocks x kT2 x u32: path 0 low half, path 1 high half
  static constexpr size_t sums = masks + (size_t)32 * kT2 * 4;         // 2 paths x 3 x kT2 doubles: unit sums
  static constexpr size_t f64 = sums + (size_t)2 * 3 * kT2 * 8;        // 6 x kT2 doubles: O, D of the waiting path
  static constexpr size_t u32 = f64 + (size_t)6 * kT2 * 8;             // 7 x kT2 words: its bookkeeping
  static constexpr size_t table = u32 + (size_t)7 * kT2 * 4;           // KParams::ltab: the groups, then the slot -> index map
  static constexpr size_t total = table + (size_t)kLtabUint4 * 16;
};

// kSampleBuf: strict order through the per-sample buffer, its own instantiation (rtclj_kernels.cuh); kListed: the
// pixels of KParams::list only (render_lane2_listed_kernel); kFrames: a camera sequence, P = FP->P
// (render_lane2_frames_kernel)
template <bool kSampleBuf, bool kListed, bool kFrames = false>
__device__ __forceinline__ void render_lane2_body(const KParams& P, const FrameKParams* FP = nullptr) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31;
  const unsigned gtid = blockIdx.x * kT2 + tid;
  unsigned* const my_mask = reinterpret_cast<unsigned*>(smem_raw + Lane2Smem::masks) + tid;       // [block * kT2]
  double* const my_sums = reinterpret_cast<double*>(smem_raw + Lane2Smem::sums) + tid;            // [(path * 3 + c) * kT2]
  double* const wO = reinterpret_cast<double*>(smem_raw + Lane2Smem::f64) + tid;                  // [c * kT2]: Ox Oy Oz Dx Dy Dz
  unsigned* const wU = reinterpret_cast<unsigned*>(smem_raw + Lane2Smem::u32) + tid;              // [c * kT2]
  const unsigned short* const slot_index = reinterpret_cast<const unsigned short*>(smem_raw + Lane2Smem::table) + kLtabSlots * 8;
  const unsigned flags = P.flags;
  const unsigned FULL = 0xffffffffu;
  const unsigned long long total_units = kListed ? total_units_of<true>(P) : 0ull;

  // the path in registers
  PathRegs pr;
  pr.O = mk(0.0, 0.0, 0.0); pr.D = mk(0.0, 0.0, 1.0);
  pr.pixel = 0; pr.unit = 0; pr.k = 0; pr.k_end = 0; pr.depth_left = 0; pr.nstack = 0; pr.status = PS_FRESH;
  PathCounters pc = {0u, 0u, 0u, 0u};
  d3& O = pr.O; d3& D = pr.D;
  unsigned& pixel = pr.pixel; unsigned& unit = pr.unit;
  int& k = pr.k; int& k_end = pr.k_end; int& depth_left = pr.depth_left; int& nstack = pr.nstack; int& status = pr.status;
  // the waiting path starts FRESH as well
  wU[6 * kT2] = (unsigned)PS_FRESH;
  if (!kFrames) {  // the spatially ordered cull table, for level 2 of the cull
    uint4* const tab = reinterpret_cast<uint4*>(smem_raw + Lane2Smem::table);
    static_assert(kLtabUint4 <= kT2, "one uint4 of the table per thread");
    if (tid < kLtabUint4) tab[tid] = __ldg(reinterpret_cast<const uint4*>(P.ltab) + tid);
    __syncthreads();
  }

#ifdef RTCLJ_TAIL_PROBE  // tuning builds only (tools/tail_probe.py): when does each warp start, first run dry, end?
  unsigned long long t_start, t_dry = 0, t_end;
  unsigned n_iter = 0, n_iter_dry = 0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_start));
#endif
  for (;;) {
#ifdef RTCLJ_TAIL_PROBE
    n_iter++;
    if (t_dry == 0 && __any_sync(FULL, status == PS_DEAD || wU[6 * kT2] == (unsigned)PS_DEAD)) {
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_dry));
      n_iter_dry = n_iter;
    }
#endif
    // ================================================================ (A) cull, both paths at once
    unsigned bany0 = 0, bany1 = 0;  // which blocks have a survivor (block j at bit 32 - nconst + j)
    {
      const bool ray1 = wU[6 * kT2] == (unsigned)PS_RAY;
      d3 O1 = mk(0.0, 0.0, 0.0), D1 = mk(0.0, 0.0, 1.0);
      if (ray1) { O1 = mk(wO[0], wO[kT2], wO[2 * kT2]); D1 = mk(wO[3 * kT2], wO[4 * kT2], wO[5 * kT2]); }
      if (!(flags & F_NO_CULL) && __any_sync(FULL, status == PS_RAY || ray1)) {
        const RayView a = make_view(P, O, D), b = make_view(P, O1, D1);
        const f32x2 a_nb = splat2(a.nbetaf), a_kq = splat2(a.kqf), b_nb = splat2(b.nbetaf), b_kq = splat2(b.kqf);
        const f32x2 a_ox = splat2(2.0f * a.ofx), a_oy = splat2(2.0f * a.ofy), a_oz = splat2(2.0f * a.ofz);
        const f32x2 b_ox = splat2(2.0f * b.ofx), b_oy = splat2(2.0f * b.ofy), b_oz = splat2(2.0f * b.ofz);
        const f32x2 a_dx = splat2(a.dhx), a_dy = splat2(a.dhy), a_dz = splat2(a.dhz);
        const f32x2 b_dx = splat2(b.dhx), b_dy = splat2(b.dhy), b_dz = splat2(b.dhz);
        // one pair of cull records against both lines: record s of a block -> sign bit 2 kCBP - 1 - s of acc0 / acc1
        auto pair = [&](const f32x2 cx, const f32x2 cy, const f32x2 cz, const f32x2 rs, f32x2 akq, f32x2 bkq, unsigned& acc0,
                        unsigned& acc1) {
          {
            const f32x2 bb = fma2(cz, a_dz, fma2(cy, a_dy, fma2(cx, a_dx, a_nb)));
            const f32x2 ss = fma2(cz, a_oz, fma2(cy, a_oy, fma2(cx, a_ox, add2(rs, akq))));
            const f32x2 dd = fma2(bb, bb, ss);
            acc0 = __funnelshift_l((unsigned)dd, acc0, 1);
            acc0 = __funnelshift_l((unsigned)(dd >> 32), acc0, 1);
          }
          {
            const f32x2 bb = fma2(cz, b_dz, fma2(cy, b_dy, fma2(cx, b_dx, b_nb)));
            const f32x2 ss = fma2(cz, b_oz, fma2(cy, b_oy, fma2(cx, b_ox, add2(rs, bkq))));
            const f32x2 dd = fma2(bb, bb, ss);
            acc1 = __funnelshift_l((unsigned)dd, acc1, 1);
            acc1 = __funnelshift_l((unsigned)(dd >> 32), acc1, 1);
          }
        };
        const int ng = P.nconst;
        if constexpr (kFrames) {
          // the camera-sequence twins keep the flat cull: every block of the list-order table, stored unconditionally
          // (their chunked instantiation has no room for the second level in the 34 KB instruction-cache budget)
#pragma unroll 1
          for (int ub = 0; ub < ng; ++ub) {
            unsigned acc0 = 0xffffffffu, acc1 = 0xffffffffu;
#pragma unroll
            for (int p = 0; p < kCBP; ++p) {
              const uint4 u = P.ctab[2 * (ub * kCBP + p)], v = P.ctab[2 * (ub * kCBP + p) + 1];
              pair(((f32x2)u.y << 32) | u.x, ((f32x2)u.w << 32) | u.z, ((f32x2)v.y << 32) | v.x, ((f32x2)v.w << 32) | v.z,
                   a_kq, b_kq, acc0, acc1);
            }
            my_mask[ub * kT2] = __byte_perm(acc0, acc1, 0x5410);
            bany0 = (bany0 >> 1) | (acc0 != 0xffffffffu ? 0x80000000u : 0u);
            bany1 = (bany1 >> 1) | (acc1 != 0xffffffffu ? 0x80000000u : 0u);
          }
        } else {
          // level 1: the sign bits of the group records for each line, from uniform operands; one running word per line
          // (group g at bit 16 nb - 1 - g after nb blocks, set = the record rejects the line, ones above)
          unsigned rej0 = 0xffffffffu, rej1 = 0xffffffffu;
          {
            const f32x2 a_kg = splat2(a.kqf * kGroupKq), b_kg = splat2(b.kqf * kGroupKq);
#pragma unroll 1
            for (int ub = 0; ub * kGroupSpheres < ng; ++ub) {
#pragma unroll
              for (int p = 0; p < kCBP; ++p) {
                const uint4 u = P.gtab[2 * (ub * kCBP + p)], v = P.gtab[2 * (ub * kCBP + p) + 1];
                pair(((f32x2)u.y << 32) | u.x, ((f32x2)u.w << 32) | u.z, ((f32x2)v.y << 32) | v.x, ((f32x2)v.w << 32) | v.z,
                     a_kg, b_kg, rej0, rej1);
              }
            }
          }
          // level 2: each lane culls the groups either of its lines reaches, both lines at once, from the shared-memory
          // table.  A group one line does not reach yields no survivor for it: the same masks as culling every group.
          const ulonglong2* const tab = reinterpret_cast<const ulonglong2*>(smem_raw + Lane2Smem::table);
          // (the groups either line reaches, group g at bit 32 - ng + g as in bany; padding groups shift out)
          const int nb = (ng + kGroupSpheres - 1) / kGroupSpheres;
          unsigned todo = __brev(~(rej0 & rej1)) << (kGroupSpheres * nb - ng);
#pragma unroll 1
          while (todo) {
            const unsigned bit = todo & (0u - todo);
            todo ^= bit;
            const int g = ng - 1 - __clz(bit);
            const ulonglong2* const t = tab + g * kGroupStride;
            unsigned acc0 = 0xffffffffu, acc1 = 0xffffffffu;
#pragma unroll 1
            for (const ulonglong2* q = t; q != t + 2 * kCBP; q += 2) {
              const ulonglong2 u = q[0], v = q[1];
              pair(u.x, u.y, v.x, v.y, a_kq, b_kq, acc0, acc1);
            }
            // slot s of the group -> bit 15 - s (path 0) / 31 - s (path 1); clear = survivor
            my_mask[g * kT2] = __byte_perm(acc0, acc1, 0x5410);
            bany0 |= acc0 != 0xffffffffu ? bit : 0u;
            bany1 |= acc1 != 0xffffffffu ? bit : 0u;
          }
          __syncwarp();  // (without it ptxas demotes the next segment's level-1 loads to per-lane LDC)
        }
      }
    }

    // ================================================================ (B)+(C) the two paths in turn
#pragma unroll 1
    for (int path = 0; path < 2; ++path) {
      const unsigned mask_shift = path ? 16u : 0u;
      path_step<kSampleBuf, kT2, kListed, kFrames>(P, pr, pc, path ? bany1 : bany0,
                                                   [&](int j) { return ~(my_mask[j * kT2] >> mask_shift) & 0xffffu; },
                                                   my_sums + path * 3 * kT2, (size_t)gtid * 2u + (size_t)path, lane, total_units, FP,
                                                   [&](int s) { return kFrames ? s : (int)slot_index[s]; });

      // ---- swap: this path waits in shared memory while the other one is processed / both are culled
      {
        const d3 tO = mk(wO[0], wO[kT2], wO[2 * kT2]), tD = mk(wO[3 * kT2], wO[4 * kT2], wO[5 * kT2]);
        const unsigned t_pixel = wU[0], t_unit = wU[kT2], t_k = wU[2 * kT2], t_kend = wU[3 * kT2];
        const unsigned t_depth = wU[4 * kT2], t_nstack = wU[5 * kT2], t_status = wU[6 * kT2];
        wO[0] = O.x; wO[kT2] = O.y; wO[2 * kT2] = O.z; wO[3 * kT2] = D.x; wO[4 * kT2] = D.y; wO[5 * kT2] = D.z;
        wU[0] = pixel; wU[kT2] = unit; wU[2 * kT2] = (unsigned)k; wU[3 * kT2] = (unsigned)k_end;
        wU[4 * kT2] = (unsigned)depth_left; wU[5 * kT2] = (unsigned)nstack; wU[6 * kT2] = (unsigned)status;
        O = tO; D = tD;
        pixel = t_pixel; unit = t_unit; k = (int)t_k; k_end = (int)t_kend;
        depth_left = (int)t_depth; nstack = (int)t_nstack; status = (int)t_status;
      }
    }
    // after two swaps the path that was in registers is in registers again
    if (!__any_sync(FULL, status != PS_DEAD || wU[6 * kT2] != (unsigned)PS_DEAD)) break;
  }

#ifdef RTCLJ_TAIL_PROBE
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_end));
  if (lane == 0 && P.arrive) {
    unsigned long long* rec = reinterpret_cast<unsigned long long*>(P.arrive) + ((size_t)blockIdx.x * (kT2 / 32) + (tid >> 5)) * 4;
    rec[0] = t_start; rec[1] = t_dry; rec[2] = t_end; rec[3] = ((unsigned long long)n_iter << 32) | n_iter_dry;
  }
#endif
  // ---- counters: REDUX on 16-bit halves (each lane's count fits 32 bits), one atomic per warp
  {
    const unsigned v[5] = {pc.samples, pc.seg, pc.exact, 0u, pc.pref};
#pragma unroll 1
    for (int q = 0; q < 5; ++q) {
      const unsigned lo = __reduce_add_sync(FULL, v[q] & 0xffffu), hi = __reduce_add_sync(FULL, v[q] >> 16);
      if (lane == 0) atomicAdd(P.stats + q, (unsigned long long)lo + ((unsigned long long)hi << 16));
    }
  }
}

template <bool kSampleBuf>
__global__ void __launch_bounds__(kT2, 1) render_lane2_kernel(const __grid_constant__ KParams P) {
  render_lane2_body<kSampleBuf, false>(P);
}

template <bool kSampleBuf>
__global__ void __launch_bounds__(kT2, 1) render_lane2_listed_kernel(const __grid_constant__ KParams P) {
  render_lane2_body<kSampleBuf, true>(P);
}

template <bool kSampleBuf>
__global__ void __launch_bounds__(kT2, 1) render_lane2_frames_kernel(const __grid_constant__ FrameKParams FP) {
  render_lane2_body<kSampleBuf, false, true>(FP.P, &FP);
}

template <bool kSampleBuf>
__global__ void __launch_bounds__(kT2, 1) render_lane2_listed_frames_kernel(const __grid_constant__ FrameKParams FP) {
  render_lane2_body<kSampleBuf, true, true>(FP.P, &FP);
}

// (The same loop with ONE path per lane built on path_step() was measured against render_kernel<true>: equal on
// the cover scene, 6 % slower on realm's forward product -- formed from the stack instead of a running product
// in registers -- and on primary-ray renders, which pay path_step's pixel / W division per sample.  So short
// renders and tiny scenes stay on render_kernel<true>.)

}  // namespace rtclj
