// rtclj_adaptive.cuh -- adaptive accumulation (rtclj_ctx_accum_begin_adaptive, DESIGN.md section 4.10): the fold
// that also keeps each pixel's sum of squared unit sums and decides which pixels the next pass traces, the
// compaction that lists them, and the export of the noise estimate.  Off the hot path: one thread per pixel, once
// per pass.  The render kernels only change how a ticket finds its pixel (the listed kernels).
#pragma once
#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>
#include "rtclj_kernels.cuh"

namespace rtclj {

// The noise estimate of one channel from the pixel's moments over m = ceil(n / u) units of u samples: the
// standard error of the pixel mean, ((S2 - S1^2 / m) / (m (m - 1))) / u^2, clamped at 0.  Plain IEEE operations
// in this order (the file is compiled without FMA contraction), so that a test can recompute them bit for bit.
__device__ __forceinline__ double unit_stderr(double s1, double s2, int n, int u) {
  const double m = (double)((n + u - 1) / u);
  double q = s1 * s1;
  q = q / m;
  double v = s2 - q;
  v = v / (m * (m - 1.0));
  v = v / ((double)u * (double)u);
  v = fmax(v, 0.0);
  return sqrt(v);
}

// Moments that overflowed: S1^2 or S2 is not finite, so the variance above is inf - inf = NaN or -inf, which the
// clamp would turn into 0.  The stopping rule counts such a channel as noisy instead (a bright pixel is not a
// converged one).  With finite moments both terms are finite and >= 0, so the variance is finite for m >= 2.
__device__ __forceinline__ bool moments_overflow(double s1, double s2) {
  return !(isfinite(s1 * s1) && isfinite(s2));
}

struct AParams {
  const double* sample_buf;      // strict order: per-sample colours [k][local pixel][4], or nullptr
  unsigned long long sample_stride;
  const double* partial;         // unit sums [local pixel][nchunks][3] (chunked order, seeded)
  double* out_linear;            // full image or nullptr
  unsigned char* out_rgb8;       // full image or nullptr
  int W, spp, nchunks, shard_index, shard_count, shard_rows;  // spp: the samples in sample_buf
  unsigned flags;
  unsigned long long local_pixels;
  double* acc;                   // S1 [local pixel][3]
  double* acc2;                  // S2 [local pixel][3]
  int* samples;                  // n_p [local pixel]
  unsigned char* live;           // [local pixel] 1: traced by the passes, 0: stopped for good
  int seeded;                    // render_primary_seeded_listed_kernel: S1 in partial, S2 already in acc2
  int strict;                    // pass unit 1: the mean is formed from 0.0 + S1, as the strict one-shot fold does
  int mean_n;                    // samples per pixel after this pass
  int decide;                    // 0: a sub-pass of a strict pass (fold only)
  int unit, target, min_samples; // the stopping rule
  double abs_tol, rel_tol;
};

// One pass of an adaptive accumulation, per local pixel.  A pixel traced in this pass folds its unit sums in
// unit order onto S1 (as finalize_kernel does) and their squares onto S2, then is tested; a stopped pixel keeps
// its sums and count.  Every pixel's images are written from S1 and its own count with the operations of a
// one-shot finalize_kernel, so the image is the one-shot image of n_p samples pixel by pixel.
__global__ void finalize_adaptive_kernel(const AParams A) {
  const unsigned long long p = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= A.local_pixels) return;
  double* const acc = A.acc + 3ull * p;
  double* const acc2 = A.acc2 + 3ull * p;
  const bool traced = A.live[p] != 0;
  if (!traced && !A.decide) return;
  double s1[3] = {acc[0], acc[1], acc[2]};
  double s2[3] = {acc2[0], acc2[1], acc2[2]};
  if (traced) {
    if (A.sample_buf) {  // strict order: every sample is a unit
      const double2* src = reinterpret_cast<const double2*>(A.sample_buf) + p * 2ull;
#pragma unroll 4
      for (int k = 0; k < A.spp; ++k) {
        const double2 xy = __ldcs(src + (unsigned long long)k * A.sample_stride * 2ull);
        const double2 z = __ldcs(src + (unsigned long long)k * A.sample_stride * 2ull + 1);
        s1[0] = s1[0] + xy.x; s1[1] = s1[1] + xy.y; s1[2] = s1[2] + z.x;
        s2[0] = s2[0] + xy.x * xy.x; s2[1] = s2[1] + xy.y * xy.y; s2[2] = s2[2] + z.x * z.x;
      }
    } else if (A.seeded) {  // one unit that continued S1 (and S2, in place) sample by sample
      const double* src = A.partial + p * 3ull;
      s1[0] = src[0]; s1[1] = src[1]; s1[2] = src[2];
    } else {
      const double* src = A.partial + p * (unsigned long long)A.nchunks * 3ull;
      for (int c = 0; c < A.nchunks; ++c) {
        const double ur = src[3 * c], ug = src[3 * c + 1], ub = src[3 * c + 2];
        s1[0] = s1[0] + ur; s1[1] = s1[1] + ug; s1[2] = s1[2] + ub;
        s2[0] = s2[0] + ur * ur; s2[1] = s2[1] + ug * ug; s2[2] = s2[2] + ub * ub;
      }
    }
    acc[0] = s1[0]; acc[1] = s1[1]; acc[2] = s1[2];
    if (!A.seeded) { acc2[0] = s2[0]; acc2[1] = s2[1]; acc2[2] = s2[2]; }
    if (!A.decide) return;
    A.samples[p] = A.mean_n;
  }
  const int n = traced ? A.mean_n : A.samples[p];
  double mean[3];
  for (int c = 0; c < 3; ++c) mean[c] = A.strict ? 0.0 + s1[c] : s1[c];
  if (A.flags & F_MEAN_DIVIDE) {
    const double s = (double)n;
    for (int c = 0; c < 3; ++c) mean[c] = mean[c] / s;
  } else {
    const double s = 1.0 / (double)n;
    for (int c = 0; c < 3; ++c) mean[c] = mean[c] * s;
  }
  const int lr = (int)(p / (unsigned)A.W);
  const int i = (int)(p - (unsigned long long)lr * (unsigned)A.W);
  const int tile = lr / A.shard_rows;
  const int j = (tile * A.shard_count + A.shard_index) * A.shard_rows + (lr - tile * A.shard_rows);
  const size_t o = 3ull * ((size_t)j * (size_t)A.W + (size_t)i);
  if (A.out_linear) { A.out_linear[o] = mean[0]; A.out_linear[o + 1] = mean[1]; A.out_linear[o + 2] = mean[2]; }
  if (A.out_rgb8) {
    const bool lin = (A.flags & F_QUANT_LINEAR) != 0;
    A.out_rgb8[o] = quantise(mean[0], lin); A.out_rgb8[o + 1] = quantise(mean[1], lin); A.out_rgb8[o + 2] = quantise(mean[2], lin);
  }
  if (traced) {  // the stopping rule: the pixel stays active iff below the target and (below min_samples or noisy)
    bool noisy = n < A.min_samples;
    for (int c = 0; c < 3; ++c) {
      const double t = A.abs_tol + A.rel_tol * fabs(mean[c]);
      noisy = noisy || moments_overflow(s1[c], s2[c]) || unit_stderr(s1[c], s2[c], n, A.unit) > t;
    }
    A.live[p] = (n < A.target && noisy) ? 1 : 0;
  }
}

// The sample-count map (int32) and the noise estimate (3 doubles) of the shard's pixels, at their full-image
// positions: the numbers the stopping rule compared.
__global__ void noise_export_kernel(const AParams A, int* out_samples, double* out_stderr) {
  const unsigned long long p = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= A.local_pixels) return;
  const int lr = (int)(p / (unsigned)A.W);
  const int i = (int)(p - (unsigned long long)lr * (unsigned)A.W);
  const int tile = lr / A.shard_rows;
  const int j = (tile * A.shard_count + A.shard_index) * A.shard_rows + (lr - tile * A.shard_rows);
  const size_t o = (size_t)j * (size_t)A.W + (size_t)i;
  const int n = A.samples[p];
  if (out_samples) out_samples[o] = n;
  if (out_stderr)
    for (int c = 0; c < 3; ++c) out_stderr[3 * o + c] = unit_stderr(A.acc[3 * p + c], A.acc2[3 * p + c], n, A.unit);
}

// ---- compaction: the live pixels in descending order into list[0, *count).  Three launches: count per tile,
// scan of the tile counts (one CTA), scatter.  Tile t covers positions [t * kListTile, (t + 1) * kListTile) of
// the descending order (position s is pixel local_pixels - 1 - s), so the list is ordered like the tickets of
// unit_of_ticket.
constexpr int kListThreads = 256, kListPer = 8, kListTile = kListThreads * kListPer;

__device__ __forceinline__ int live_run(const unsigned char* live, unsigned long long n, unsigned long long s0) {
  int cnt = 0;
#pragma unroll
  for (int e = 0; e < kListPer; ++e) {
    const unsigned long long s = s0 + (unsigned long long)e;
    if (s < n && live[n - 1 - s]) ++cnt;
  }
  return cnt;
}

__global__ void __launch_bounds__(kListThreads) list_count_kernel(const unsigned char* live, unsigned long long n,
                                                                  unsigned* tile_counts) {
  typedef cub::BlockReduce<int, kListThreads> Reduce;
  __shared__ typename Reduce::TempStorage tmp;
  const unsigned long long s0 = (unsigned long long)blockIdx.x * kListTile + (unsigned long long)threadIdx.x * kListPer;
  const int total = Reduce(tmp).Sum(live_run(live, n, s0));
  if (threadIdx.x == 0) tile_counts[blockIdx.x] = (unsigned)total;
}

__global__ void __launch_bounds__(1024) list_scan_kernel(unsigned* tile_counts, unsigned ntiles, unsigned* count) {
  typedef cub::BlockScan<unsigned, 1024> Scan;
  __shared__ typename Scan::TempStorage tmp;
  unsigned carry = 0;
  for (unsigned b = 0; b < ntiles; b += 1024) {
    const unsigned t = b + threadIdx.x;
    const unsigned v = t < ntiles ? tile_counts[t] : 0u;
    unsigned excl, sum;
    Scan(tmp).ExclusiveSum(v, excl, sum);
    __syncthreads();  // tmp is reused by the next round
    if (t < ntiles) tile_counts[t] = carry + excl;
    carry += sum;
  }
  if (threadIdx.x == 0) *count = carry;
}

__global__ void __launch_bounds__(kListThreads) list_scatter_kernel(const unsigned char* live, unsigned long long n,
                                                                    const unsigned* tile_offsets, unsigned* list) {
  typedef cub::BlockScan<int, kListThreads> Scan;
  __shared__ typename Scan::TempStorage tmp;
  const unsigned long long s0 = (unsigned long long)blockIdx.x * kListTile + (unsigned long long)threadIdx.x * kListPer;
  int at = 0;
  Scan(tmp).ExclusiveSum(live_run(live, n, s0), at);
  unsigned o = tile_offsets[blockIdx.x] + (unsigned)at;
#pragma unroll
  for (int e = 0; e < kListPer; ++e) {
    const unsigned long long s = s0 + (unsigned long long)e;
    if (s < n && live[n - 1 - s]) list[o++] = (unsigned)(n - 1 - s);
  }
}

// The compaction of n pixels' live flags: list[0, aux[0]) gets the live pixels in descending order, aux[0] their
// count; aux[1, 1 + tiles) is the scan's scratch.  Asynchronous on `stream`; n == 0 launches nothing.
inline cudaError_t launch_relist(const unsigned char* live, unsigned long long n, unsigned* aux, unsigned* list,
                                 cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  const unsigned tiles = (unsigned)((n + kListTile - 1) / kListTile);
  list_count_kernel<<<tiles, kListThreads, 0, stream>>>(live, n, aux + 1);
  list_scan_kernel<<<1, 1024, 0, stream>>>(aux + 1, tiles, aux);
  list_scatter_kernel<<<tiles, kListThreads, 0, stream>>>(live, n, aux + 1, list);
  return cudaGetLastError();
}

}  // namespace rtclj
