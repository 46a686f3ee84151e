// Test harness for the adaptive-sampling kernels of rtclj_adaptive.cuh, which it includes unchanged: C wrappers
// that launch the compaction, unit_stderr over arrays and finalize_adaptive_kernel on device pointers (torch
// tensors) and a stream, so that tests/test_gpu_adaptive_kernels.py can compare them with numpy at sizes and edges
// the public API does not reach.  Built on first use by tests/adaptive_kernels.py with the library's flags.
#include <cstddef>
#include "rtclj_adaptive.cuh"

using rtclj::AParams;

namespace {

__global__ void unit_stderr_kernel(const double* s1, const double* s2, const int* n, int u, unsigned long long count,
                                   double* out, unsigned char* overflow) {
  const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  out[i] = rtclj::unit_stderr(s1[i], s2[i], n[i], u);
  overflow[i] = rtclj::moments_overflow(s1[i], s2[i]) ? 1 : 0;
}

}  // namespace

extern "C" {

// the compaction of the library (launch_relist): list[0, aux[0]) the live pixels in descending order
int ak_relist(const unsigned char* live, unsigned long long n, unsigned* aux, unsigned* list, void* stream) {
  return (int)rtclj::launch_relist(live, n, aux, list, (cudaStream_t)stream);
}

// out[i] = unit_stderr(s1[i], s2[i], n[i], u); overflow[i] = moments_overflow(s1[i], s2[i])
int ak_unit_stderr(const double* s1, const double* s2, const int* n, int u, unsigned long long count, double* out,
                   unsigned char* overflow, void* stream) {
  if (count == 0) return 0;
  unit_stderr_kernel<<<(unsigned)((count + 255) / 256), 256, 0, (cudaStream_t)stream>>>(s1, s2, n, u, count, out,
                                                                                          overflow);
  return (int)cudaGetLastError();
}

// finalize_adaptive_kernel on a caller-filled AParams, one thread per local pixel as the library launches it
int ak_finalize(const AParams* A, void* stream) {
  if (A->local_pixels == 0) return 0;
  const unsigned blocks = (unsigned)((A->local_pixels + 255) / 256);
  rtclj::finalize_adaptive_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(*A);
  return (int)cudaGetLastError();
}

// sizeof(AParams) and the offset of each field, in declaration order: the Python mirror checks its layout
int ak_aparams_layout(unsigned long long* out, int cap) {
  const unsigned long long v[] = {
      sizeof(AParams),
      offsetof(AParams, sample_buf), offsetof(AParams, sample_stride), offsetof(AParams, partial),
      offsetof(AParams, out_linear), offsetof(AParams, out_rgb8), offsetof(AParams, W), offsetof(AParams, spp),
      offsetof(AParams, nchunks), offsetof(AParams, shard_index), offsetof(AParams, shard_count),
      offsetof(AParams, shard_rows), offsetof(AParams, flags), offsetof(AParams, local_pixels),
      offsetof(AParams, acc), offsetof(AParams, acc2), offsetof(AParams, samples), offsetof(AParams, live),
      offsetof(AParams, seeded), offsetof(AParams, strict), offsetof(AParams, mean_n), offsetof(AParams, decide),
      offsetof(AParams, unit), offsetof(AParams, target), offsetof(AParams, min_samples),
      offsetof(AParams, abs_tol), offsetof(AParams, rel_tol)};
  const int n = (int)(sizeof v / sizeof v[0]);
  for (int i = 0; i < n && i < cap; ++i) out[i] = v[i];
  return n;
}

// the compaction's tile size (kListTile)
int ak_list_tile() { return rtclj::kListTile; }

}  // extern "C"
