// Edge-avoiding a-trous filter of a linear image, guided by a second image (the normal-shaded primary render):
// the device side of rtclj_ctx_denoise.  The definition is in include/rtclj_b200.h; tests/denoise_model.py reproduces
// it bit for bit, so every operation below is an IEEE float32 + - * / or fmaxf in the order the header states
// (rtclj_abi.cu is compiled with --fmad=false and IEEE division).  DESIGN.md section 4.13.
#pragma once

#include "rtclj_kernels.cuh"

namespace rtclj {

constexpr int kDenoiseTileW = 32, kDenoiseTileH = 8;  // one CTA: a 32 x 8 pixel tile, one thread per pixel
constexpr unsigned kDenoiseMaxBlocks = 1u << 20;      // grid-stride over tiles beyond this (64-bit tile index)

struct DenoiseParams {
  const double* lin64;    // level 0: the caller's colour C (W*H*3 doubles); the last level: its non-finite fallback
  const double* guide64;  // level 0: the caller's guide G
  const float4* src;      // levels > 0: c_i
  float4* dst;            // levels < L-1: c_(i+1)
  float4* guide;          // level 0 writes float32(G) here (L > 1); later levels read it
  double* out_linear;     // the last level: (double)c_L, or C where the pixel was not filtered; may be nullptr
  unsigned char* out_rgb8;  // the last level: write-color! of out_linear; may be nullptr
  long long W, H;
  int step;               // 2^i
  float sigma2_c;         // (sigma_c * 2^-i)^2
  float sigma2_g;         // sigma_g^2
  int quant_linear;
};

__device__ __forceinline__ bool finite3(float4 v) { return isfinite(v.x) && isfinite(v.y) && isfinite(v.z); }

__device__ __forceinline__ float4 load64(const double* p, long long i) {
  const double* q = p + 3 * i;
  return make_float4((float)q[0], (float)q[1], (float)q[2], 0.f);
}

// k(x) = t * t, t = fmax(1 - x, 0)
__device__ __forceinline__ float denoise_k(float x) {
  const float t = fmaxf(1.0f - x, 0.0f);
  return t * t;
}

__device__ __forceinline__ float sqdist(float4 a, float4 b) {
  const float dr = a.x - b.x, dg = a.y - b.y, db = a.z - b.z;
  return (dr * dr + dg * dg) + db * db;
}

// One level of the filter.  First: taps read the caller's f64 images (the float32 conversion folded in) and the
// guide is written as float32 for the later levels.  Last: the f64 and 8-bit outputs are written instead of c_(i+1).
// First && Last reads C's neighbours while writing out_linear: the host never launches it with the two overlapping.
template <bool First, bool Last>
__global__ void __launch_bounds__(kDenoiseTileW * kDenoiseTileH) denoise_level_kernel(const DenoiseParams P) {
  const long long tiles_x = (P.W + kDenoiseTileW - 1) / kDenoiseTileW;
  const long long tiles = tiles_x * ((P.H + kDenoiseTileH - 1) / kDenoiseTileH);
  const float h[5] = {1.0f / 16.0f, 1.0f / 4.0f, 3.0f / 8.0f, 1.0f / 4.0f, 1.0f / 16.0f};
  for (long long t = blockIdx.x; t < tiles; t += gridDim.x) {
    const long long ty = t / tiles_x;
    const long long x = (t - ty * tiles_x) * kDenoiseTileW + threadIdx.x;
    const long long y = ty * kDenoiseTileH + threadIdx.y;
    if (x >= P.W || y >= P.H) continue;
    const long long p = y * P.W + x;
    const float4 cp = First ? load64(P.lin64, p) : P.src[p];
    const float4 gp = First ? load64(P.guide64, p) : P.guide[p];
    if (First && !Last) P.guide[p] = gp;
    float4 out = cp;
    const bool filtered = finite3(cp) && finite3(gp);
    if (filtered) {
      float ar = 0.f, ag = 0.f, ab = 0.f, wsum = 0.f;
#pragma unroll
      for (int dy = -2; dy <= 2; ++dy) {
        const long long qy = y + (long long)P.step * dy;
        if (qy < 0 || qy >= P.H) continue;
#pragma unroll
        for (int dx = -2; dx <= 2; ++dx) {
          const long long qx = x + (long long)P.step * dx;
          if (qx < 0 || qx >= P.W) continue;
          const long long q = qy * P.W + qx;
          const float4 cq = First ? load64(P.lin64, q) : P.src[q];
          const float4 gq = First ? load64(P.guide64, q) : P.guide[q];
          if (!finite3(cq) || !finite3(gq)) continue;
          const float dc = sqdist(cq, cp), dg = sqdist(gq, gp);
          const float w = ((h[dx + 2] * h[dy + 2]) * denoise_k(dc / P.sigma2_c)) * denoise_k(dg / P.sigma2_g);
          ar = ar + w * cq.x; ag = ag + w * cq.y; ab = ab + w * cq.z;
          wsum = wsum + w;
        }
      }
      out = make_float4(ar / wsum, ag / wsum, ab / wsum, 0.f);
    }
    if (!Last) {
      P.dst[p] = out;
    } else {
      double r = (double)out.x, g = (double)out.y, b = (double)out.z;
      // a pixel whose float32 colour or guide is not finite was never filtered: it keeps its input value.  (A
      // pixel filtered into a non-finite value, by float32 overflow, keeps the non-finite float.)
      // c_i of a pixel with a non-finite c_0 stays c_0: C is read again only where c_(L-1) is not finite.
      if (!finite3(gp) || (!finite3(cp) && (First || !finite3(load64(P.lin64, p))))) {
        r = P.lin64[3 * p]; g = P.lin64[3 * p + 1]; b = P.lin64[3 * p + 2];
      }
      if (P.out_linear) { P.out_linear[3 * p] = r; P.out_linear[3 * p + 1] = g; P.out_linear[3 * p + 2] = b; }
      if (P.out_rgb8) {
        const bool lin = P.quant_linear != 0;
        P.out_rgb8[3 * p] = quantise(r, lin); P.out_rgb8[3 * p + 1] = quantise(g, lin); P.out_rgb8[3 * p + 2] = quantise(b, lin);
      }
    }
  }
}

// float32(C) and float32(G) as float4 images: level 0 of an in-place call with L = 1, where the folded conversion
// would read C's neighbours after other threads overwrote them.
__global__ void __launch_bounds__(256) denoise_convert_kernel(const double* lin64, const double* guide64, float4* c,
                                                              float4* g, long long npix) {
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < npix; p += (long long)gridDim.x * blockDim.x) {
    c[p] = load64(lin64, p);
    g[p] = load64(guide64, p);
  }
}

}  // namespace rtclj
