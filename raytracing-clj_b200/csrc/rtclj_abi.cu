// rtclj_abi.cu -- the C ABI (include/rtclj_b200.h) over the sm_100a kernels.
// Host side of the render loop: scene preparation (fp64 tables + the inflated fp32 cull
// table), work-unit sizing, launches, copies.  No CPU fallback anywhere in this file.
#include "../../include/rtclj_b200.h"
#include "rtclj_kernels.cuh"
#include "rtclj_wave_kernel.cuh"
#include "rtclj_lane2_kernel.cuh"
#include "rtclj_primary_kernel.cuh"
#include "rtclj_split_kernel.cuh"
#include "rtclj_p3_kernels.cuh"
#include "rtclj_png_kernels.cuh"
#include "rtclj_adaptive.cuh"
#include "rtclj_error.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

using namespace rtclj;


namespace {

#define fail rtclj_fail  // the thread-local message lives in rtclj_host.cpp (rtclj_error.h)

#define CU(call)                                                                          \
  do {                                                                                    \
    cudaError_t e_ = (call);                                                              \
    if (e_ != cudaSuccess)                                                                \
      return fail(e_ == cudaErrorNoDevice || e_ == cudaErrorInsufficientDriver            \
                      ? RTCLJ_E_NO_DEVICE : RTCLJ_E_CUDA,                                 \
                  "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;  // elements
  cudaError_t reserve(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    cudaError_t e = cudaMalloc(&p, n * sizeof(T));
    if (e == cudaSuccess) cap = n;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

float round_up_to_float(double v) {
  float f = (float)v;
  if ((double)f < v) f = std::nextafterf(f, INFINITY);
  return f;
}

}  // namespace

struct rtclj_ctx {
  int device = 0;
  int sm_count = 0;
  size_t smem_optin = 0;
  int n = 0, nhalf = 0;  // spheres; 16-sphere half blocks of the padded cull table
  double shift[3] = {0, 0, 0};
  DevBuf<float4> geom32;
  DevBuf<float4> geomA;                 // one {cx, cy, cz, Ws} per sphere: what the fp32 prefilter loads
  DevBuf<Geom64> geom64;
  DevBuf<MatRec> mat;
  DevBuf<double> partial;
  DevBuf<unsigned long long> counters;  // [0] queue, [1..4] stats
  DevBuf<unsigned short> stack;
  DevBuf<unsigned> arrive;              // wavefront kernel: chunk arrival counters per pixel
  DevBuf<double> sample_buf;            // strict order on long paths: one colour per sample (kept between renders)
  std::vector<float> ctab_host;         // the cull table of a small scene: launched as a kernel parameter
  KParams kparams;                      // launch parameters of the last render (8.4 KB with the table)
  FrameKParams fparams;                 // launch parameters of the last camera-sequence launch (28 KB)
  DevBuf<double> out_linear;            // used by the host-buffer entry points
  DevBuf<unsigned char> out_rgb8;
  DevBuf<unsigned long long> p3_state;  // P3 writer: ticket, total, text bytes per CTA run
  int p3_ctas_per_sm = 0;
  DevBuf<unsigned char> p3_in, p3_text; // staging for the host-buffer entry point
  float p3_count_ms = 0.f, p3_write_ms = 0.f;
  // PNG writer: the filtered stream F, one staging slot and one record per 64 KiB segment, the total length
  DevBuf<unsigned char> png_f, png_stage;
  DevBuf<PngSegRec> png_rec;
  DevBuf<unsigned long long> png_state;
  DevBuf<unsigned char> png_in, png_out;  // staging for the host-buffer entry points
  bool png_attr = false;                   // the PNG kernels' shared-memory limit is raised
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;  // render: start, kernel end, finalize end
  cudaEvent_t p3_ev0 = nullptr, p3_ev1 = nullptr;           // the P3 writer's own timing events
  cudaStream_t own_stream = nullptr;
  int last_spu = 0;
  // the accumulation in progress (rtclj_ctx_accum_begin / _step); rtclj_ctx_set_scene ends it
  struct Accum {
    bool active = false;
    bool strict = false;     // one sequential sum per pixel (pass_unit 1)
    rtclj_camera cam;
    rtclj_params prm;        // prm.spp: the target
    int done = 0;            // samples per pixel so far
    int pass_unit = 1;
    // adaptive accumulation (rtclj_ctx_accum_begin_adaptive): the stopping rule, DESIGN.md section 4.10
    bool adaptive = false;
    double abs_tol = 0.0, rel_tol = 0.0;
    int min_samples = 0;
  } accum;
  DevBuf<double> acc;                   // the accumulation's running sums: 3 per local pixel
  // adaptive accumulation, per local pixel: sums of squared unit sums (3 doubles), sample count, live flag, and
  // the list of the live pixels (descending) that the listed kernels trace; list_aux = [count, tile counts...]
  DevBuf<double> acc2;
  DevBuf<int> nsamp;
  DevBuf<unsigned char> live;
  DevBuf<unsigned> list, list_aux;
  DevBuf<int> noise_samples;            // rtclj_progressive_noise: full-size staging of the exported images
  DevBuf<double> noise_stderr;
  double prim_geom[4 * kPrimarySpheres] = {};  // exact geometry of the first spheres: parameters of render_primary_kernel
  bool have_scene = false;
  bool render_pending = false;  // a render has been enqueued since the last scene upload / stats
  // pinned staging for downloads into PAGEABLE caller memory (two buffers, pipelined)
  void* pin[2] = {nullptr, nullptr};
  size_t pin_cap = 0;
  cudaEvent_t pin_ev[2] = {nullptr, nullptr};
};

namespace {

// shared memory: [table (large scenes only)] [survivor lists, or 33 per-block masks per lane on the
// constant-table path] [mbarrier] [unit sums]
// 16-pair blocks (512 B) of the table that fit in shared memory next to the lists and the sums
int smem_table_blocks(size_t smem_optin) {
  const size_t fixed = (size_t)kListCap * threads_of(false) * 4 + 16 + (size_t)threads_of(false) * 24;
  return smem_optin > fixed ? (int)((smem_optin - fixed) / 512) : 0;
}
size_t smem_needed(int nhalf, bool const_tab, size_t smem_optin, bool few = false) {
  const size_t table = const_tab ? 0 : std::min((size_t)nhalf * 256, (size_t)smem_table_blocks(smem_optin) * 512);
  const size_t threads = (size_t)threads_of(const_tab, few);
  const size_t lists = (size_t)(const_tab ? 33 : kListCap) * threads * 4;
  return table + lists + 16 + threads * 24;
}
bool use_const_table(int nhalf) { return nhalf * 16 <= 512; }  // <= 32 blocks on that path either way

int local_rows_of(int H, int shard_index, int shard_count, int shard_rows) {
  if (shard_count <= 1) return H;
  int rows = 0;
  const int ntiles = (H + shard_rows - 1) / shard_rows;
  for (int t = shard_index; t < ntiles; t += shard_count)
    rows += std::min(shard_rows, H - t * shard_rows);
  return rows;
}

// Unit size chosen from the image alone (not from the GPU count), so that an image is
// bit-identical however many GPUs share it: aim at >= 64 units per lane of an 8-GPU box.  The kernel's
// tail lasts about one unit (lanes drain once the queue is empty): measured on the bench workload at
// 8 GPUs, 100 / 50 / 25 / 10 samples per unit give 79.7 / 72.5 / 71.8 / 72.2 ms per frame.
int auto_samples_per_unit(int W, int H, int spp) {
  const double want_units = 64.0 * 148.0 * 512.0 * 8.0;
  const double pixels = (double)W * (double)H;
  int nchunks = (int)std::ceil(want_units / pixels);
  nchunks = std::max(1, std::min(nchunks, std::max(1, spp / 8)));
  return (spp + nchunks - 1) / nchunks;
}

int validate(const rtclj_camera* cam, const rtclj_params* prm) {
  if (!cam || !prm) return fail(RTCLJ_E_INVALID, "null camera or params");
  if (cam->width <= 0 || cam->height <= 0) return fail(RTCLJ_E_INVALID, "image size must be positive");
  {
    bool finite = std::isfinite(cam->defocus_angle);
    for (int a = 0; a < 3; ++a)
      finite = finite && std::isfinite(cam->pixel00[a]) && std::isfinite(cam->pixel_du[a]) && std::isfinite(cam->pixel_dv[a]) &&
               std::isfinite(cam->center[a]) && std::isfinite(cam->defocus_u[a]) && std::isfinite(cam->defocus_v[a]);
    if (!finite) return fail(RTCLJ_E_INVALID, "non-finite camera value");
    for (int a = 0; a < 3; ++a)
      if (!(std::fabs(cam->center[a]) + std::fabs(cam->defocus_u[a]) + std::fabs(cam->defocus_v[a]) < 1e18))
        return fail(RTCLJ_E_INVALID, "camera coordinates beyond 1e18 are not supported");
  }
  if ((uint64_t)cam->width * (uint64_t)cam->height > 0xffffffffull)
    return fail(RTCLJ_E_INVALID, "more than 2^32 pixels");
  if (prm->spp <= 0) return fail(RTCLJ_E_INVALID, "spp must be positive");
  if (prm->shard_count > 1 && (prm->shard_index < 0 || prm->shard_index >= prm->shard_count || prm->shard_rows <= 0))
    return fail(RTCLJ_E_INVALID, "bad shard (%d of %d, %d rows)", prm->shard_index, prm->shard_count, prm->shard_rows);
  return RTCLJ_OK;
}

// Every instantiation of the render kernels, indexed by its template flags: launch_pass launches from these tables
// and rtclj_ctx_create raises the dynamic shared memory limit of every entry that takes some (kSmemLimits).
using KernelFn = void (*)(KParams);
// render_kernel and render_listed_kernel, [listed][const_tab][sample_buf][packed]: threads_of(const_tab, packed)
// threads, smem_needed() bytes.  The packed instantiation exists with the constant table only.
const KernelFn kRenderFns[2][2][2][2] = {
    {{{render_kernel<false, false, false>, nullptr}, {render_kernel<false, true, false>, nullptr}},
     {{render_kernel<true, false, false>, render_kernel<true, false, true>},
      {render_kernel<true, true, false>, render_kernel<true, true, true>}}},
    {{{render_listed_kernel<false, false, false>, nullptr}, {render_listed_kernel<false, true, false>, nullptr}},
     {{render_listed_kernel<true, false, false>, render_listed_kernel<true, false, true>},
      {render_listed_kernel<true, true, false>, render_listed_kernel<true, true, true>}}}};
// render_lane2_kernel and render_lane2_listed_kernel, [listed][sample_buf]: kT2 threads, Lane2Smem::total bytes
const KernelFn kLane2Fns[2][2] = {{render_lane2_kernel<false>, render_lane2_kernel<true>},
                                  {render_lane2_listed_kernel<false>, render_lane2_listed_kernel<true>}};
// render_split_kernel, [sample_buf]: kSplitThreads threads, SplitSmem::total bytes
const KernelFn kSplitFns[2] = {render_split_kernel<false>, render_split_kernel<true>};
// render_wave_kernel: kWT threads, WaveSmem::total bytes
const KernelFn kWaveFns[1] = {render_wave_kernel};
// the primary-ray kernels, [listed][seeded][defocus]: kPrimaryThreads threads, no dynamic shared memory
const KernelFn kPrimaryFns[2][2][2] = {
    {{render_primary_kernel<false>, render_primary_kernel<true>},
     {render_primary_seeded_kernel<false>, render_primary_seeded_kernel<true>}},
    {{render_primary_listed_kernel<false>, render_primary_listed_kernel<true>},
     {render_primary_seeded_listed_kernel<false>, render_primary_seeded_listed_kernel<true>}}};

// The frame twins of a camera sequence (FrameKParams), one per instantiation the library can choose for it:
// render_frames_kernel [const_tab][sample_buf][packed] as kRenderFns[0], render_lane2_frames_kernel [sample_buf],
// render_primary_frames_kernel [some frame has the defocus disk].  (The wave and split kernels render no sequences.)
using FramesFn = void (*)(FrameKParams);
const FramesFn kRenderFramesFns[2][2][2] = {
    {{render_frames_kernel<false, false, false>, nullptr}, {render_frames_kernel<false, true, false>, nullptr}},
    {{render_frames_kernel<true, false, false>, render_frames_kernel<true, false, true>},
     {render_frames_kernel<true, true, false>, render_frames_kernel<true, true, true>}}};
const FramesFn kLane2FramesFns[2] = {render_lane2_frames_kernel<false>, render_lane2_frames_kernel<true>};
const FramesFn kPrimaryFramesFns[2] = {render_primary_frames_kernel<false>, render_primary_frames_kernel<true>};

// the tables of kernels with dynamic shared memory, and the most a launch asks for (0: the device's opt-in limit)
template <class Fn> struct SmemLimit { const Fn* fns; size_t count; size_t bytes; };
const SmemLimit<KernelFn> kSmemLimits[] = {
    {&kRenderFns[0][0][0][0], sizeof kRenderFns / sizeof(KernelFn), 0},
    {&kLane2Fns[0][0], sizeof kLane2Fns / sizeof(KernelFn), Lane2Smem::total},
    {kSplitFns, sizeof kSplitFns / sizeof(KernelFn), SplitSmem::total},
    {kWaveFns, sizeof kWaveFns / sizeof(KernelFn), WaveSmem::total}};
const SmemLimit<FramesFn> kFramesSmemLimits[] = {
    {&kRenderFramesFns[0][0][0], sizeof kRenderFramesFns / sizeof(FramesFn), 0},
    {kLane2FramesFns, sizeof kLane2FramesFns / sizeof(FramesFn), Lane2Smem::total}};

}  // namespace

// ---- arithmetic-peak calibration (pure FMA loops, 8 independent chains per thread)
namespace {
template <int MODE>
__global__ void __launch_bounds__(512) peak_kernel(float* out, int iters, float seed) {
  if (MODE == 2) {
    double a0 = seed, a1 = seed + 1, a2 = seed + 2, a3 = seed + 3, a4 = seed + 4, a5 = seed + 5, a6 = seed + 6, a7 = seed + 7;
    const double m = 0.999999, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
      a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
      a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = (float)(a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7);
  } else if (MODE == 1) {
    f32x2 a0 = splat2(seed), a1 = splat2(seed + 1), a2 = splat2(seed + 2), a3 = splat2(seed + 3);
    f32x2 a4 = splat2(seed + 4), a5 = splat2(seed + 5), a6 = splat2(seed + 6), a7 = splat2(seed + 7);
    const f32x2 m = splat2(0.999999f), c = splat2(1e-9f);
    for (int i = 0; i < iters; ++i) {
      a0 = fma2(a0, m, c); a1 = fma2(a1, m, c); a2 = fma2(a2, m, c); a3 = fma2(a3, m, c);
      a4 = fma2(a4, m, c); a5 = fma2(a5, m, c); a6 = fma2(a6, m, c); a7 = fma2(a7, m, c);
    }
    float lo, hi, s = 0.f;
    unpack2(a0, lo, hi); s += lo + hi; unpack2(a1, lo, hi); s += lo + hi; unpack2(a2, lo, hi); s += lo + hi;
    unpack2(a3, lo, hi); s += lo + hi; unpack2(a4, lo, hi); s += lo + hi; unpack2(a5, lo, hi); s += lo + hi;
    unpack2(a6, lo, hi); s += lo + hi; unpack2(a7, lo, hi); s += lo + hi;
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
  } else {
    float a0 = seed, a1 = seed + 1, a2 = seed + 2, a3 = seed + 3, a4 = seed + 4, a5 = seed + 5, a6 = seed + 6, a7 = seed + 7;
    const float m = 0.999999f, c = 1e-9f;
    for (int i = 0; i < iters; ++i) {
      a0 = fmaf(a0, m, c); a1 = fmaf(a1, m, c); a2 = fmaf(a2, m, c); a3 = fmaf(a3, m, c);
      a4 = fmaf(a4, m, c); a5 = fmaf(a5, m, c); a6 = fmaf(a6, m, c); a7 = fmaf(a7, m, c);
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
  }
}
}  // namespace


extern "C" {

int rtclj_abi_version(void) { return RTCLJ_ABI_VERSION; }

int rtclj_device_count(int* count) {
  if (!count) return fail(RTCLJ_E_INVALID, "null count");
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) { *count = 0; cudaGetLastError(); return fail(RTCLJ_E_NO_DEVICE, "no CUDA device: %s", cudaGetErrorString(e)); }
  *count = n;
  return RTCLJ_OK;
}

void rtclj_ctx_destroy(rtclj_ctx* c);

int rtclj_ctx_create(int32_t device, rtclj_ctx** out) {
  if (!out) return fail(RTCLJ_E_INVALID, "null out");
  *out = nullptr;
  int ndev = 0;
  int rc = rtclj_device_count(&ndev);
  if (rc) return rc;
  if (ndev == 0) return fail(RTCLJ_E_NO_DEVICE, "no CUDA device (this library has no CPU fallback)");
  if (device < 0 || device >= ndev) return fail(RTCLJ_E_INVALID, "device %d out of range [0,%d)", device, ndev);
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10)
    return fail(RTCLJ_E_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
  // owned until every CUDA call below has succeeded: a failure frees what was created
  std::unique_ptr<rtclj_ctx, void (*)(rtclj_ctx*)> guard(new (std::nothrow) rtclj_ctx(), rtclj_ctx_destroy);
  rtclj_ctx* c = guard.get();
  if (!c) return fail(RTCLJ_E_CUDA, "out of host memory");
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  c->smem_optin = prop.sharedMemPerBlockOptin;
  CU(cudaEventCreate(&c->ev0));
  CU(cudaEventCreate(&c->ev1));
  CU(cudaEventCreate(&c->ev2));
  CU(cudaEventCreate(&c->p3_ev0));
  CU(cudaEventCreate(&c->p3_ev1));
  CU(cudaEventCreateWithFlags(&c->pin_ev[0], cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&c->pin_ev[1], cudaEventDisableTiming));
  CU(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
  CU(c->counters.reserve(8));
  for (const SmemLimit<KernelFn>& t : kSmemLimits)
    for (size_t i = 0; i < t.count; ++i)
      if (t.fns[i])
        CU(cudaFuncSetAttribute(t.fns[i], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(t.bytes ? t.bytes : c->smem_optin)));
  for (const SmemLimit<FramesFn>& t : kFramesSmemLimits)
    for (size_t i = 0; i < t.count; ++i)
      if (t.fns[i])
        CU(cudaFuncSetAttribute(t.fns[i], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(t.bytes ? t.bytes : c->smem_optin)));
  *out = guard.release();
  return RTCLJ_OK;
}

void rtclj_ctx_destroy(rtclj_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->own_stream) cudaStreamSynchronize(c->own_stream);
  c->geom32.release(); c->geomA.release(); c->geom64.release(); c->mat.release(); c->partial.release();
  c->counters.release(); c->stack.release(); c->arrive.release(); c->sample_buf.release(); c->out_linear.release(); c->out_rgb8.release();
  c->acc.release(); c->acc2.release(); c->nsamp.release(); c->live.release(); c->list.release(); c->list_aux.release();
  c->noise_samples.release(); c->noise_stderr.release();
  c->p3_state.release(); c->p3_in.release(); c->p3_text.release();
  c->png_f.release(); c->png_stage.release(); c->png_rec.release(); c->png_state.release(); c->png_in.release(); c->png_out.release();
  for (cudaEvent_t e : {c->ev0, c->ev1, c->ev2, c->p3_ev0, c->p3_ev1, c->pin_ev[0], c->pin_ev[1]})
    if (e) cudaEventDestroy(e);
  for (void* h : c->pin) if (h) cudaFreeHost(h);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  delete c;
}

int rtclj_ctx_set_scene(rtclj_ctx* c, const rtclj_scene* s) {
  if (!c || !s) return fail(RTCLJ_E_INVALID, "null ctx or scene");
  c->accum.active = false;  // an accumulation belongs to the scene it began with
  const int n = s->n;
  if (n < 0) return fail(RTCLJ_E_INVALID, "negative sphere count");
  if (n > 0 && (!s->center_xyz || !s->radius || !s->material || !s->albedo_rgb || !s->fuzz || !s->ior))
    return fail(RTCLJ_E_INVALID, "null scene array");
  if (n > 65532) return fail(RTCLJ_E_TOO_LARGE, "%d spheres: survivor lists hold 16-bit indices", n);
  const int nhalf = (n + 15) / 16;  // the cull table is padded to 16-sphere half blocks
  const int npad = ((n + 31) / 32) * 32;  // table padded to 32 spheres (the constant-table path may use 16-pair blocks)
  for (int i = 0; i < n; ++i) {
    const int k = s->material[i];
    if (k != RTCLJ_LAMBERTIAN && k != RTCLJ_METAL && k != RTCLJ_DIELECTRIC)
      return fail(RTCLJ_E_INVALID, "sphere %d: unknown material id %d", i, k);
    // NaN / infinity: the reference's sequential scan degenerates (a NaN root is "accepted" and every
    // later body then wins); that is garbage in either implementation, so it is refused here
    bool finite = std::isfinite(s->radius[i]) && std::isfinite(s->fuzz[i]) && std::isfinite(s->ior[i]);
    for (int a = 0; a < 3; ++a) finite = finite && std::isfinite(s->center_xyz[3 * i + a]) && std::isfinite(s->albedo_rgb[3 * i + a]);
    if (!finite) return fail(RTCLJ_E_INVALID, "sphere %d: non-finite parameter", i);
    // the fp32 cull squares coordinates of ray origins, which lie on sphere surfaces: keep them below 1e18
    double reach = std::fabs(s->radius[i]);
    for (int a = 0; a < 3; ++a) reach = std::max(reach, std::fabs(s->center_xyz[3 * i + a]));
    if (!(reach < 1e18)) return fail(RTCLJ_E_INVALID, "sphere %d: coordinates beyond 1e18 are not supported", i);
  }
  CU(cudaSetDevice(c->device));
  // rtclj_ctx_render is asynchronous and may run on a non-blocking stream, which the blocking copies
  // below do not wait for: let the last render finish before its tables change
  if (c->render_pending) { CU(cudaEventSynchronize(c->ev2)); c->render_pending = false; }

  // translation for the fp32 cull: per-axis median of the centres keeps |C - shift|
  // (and with it the inflation of the conservative test) small where the spheres are
  double shift[3] = {0, 0, 0};
  if (n > 0) {
    std::vector<double> tmp((size_t)n);
    for (int a = 0; a < 3; ++a) {
      for (int i = 0; i < n; ++i) tmp[(size_t)i] = s->center_xyz[3 * i + a];
      std::nth_element(tmp.begin(), tmp.begin() + n / 2, tmp.end());
      shift[a] = tmp[(size_t)(n / 2)];
    }
  }
  std::vector<Geom64> g64((size_t)std::max(n, 1));
  std::vector<MatRec> mats((size_t)std::max(n, 1));
  std::vector<float> g32((size_t)std::max(npad, 2) * 4);
  std::vector<float4> gA((size_t)std::max(n, 1));
  for (int i = 0; i < npad; ++i) {
    float cx = 0.f, cy = 0.f, cz = 0.f, r2s = -1e30f;  // padding never survives the cull
    if (i < n) {
      const double* C = s->center_xyz + 3 * i;
      const double r = s->radius[i];
      g64[(size_t)i] = Geom64{C[0], C[1], C[2], r};
      MatRec m;
      m.albedo[0] = s->albedo_rgb[3 * i]; m.albedo[1] = s->albedo_rgb[3 * i + 1]; m.albedo[2] = s->albedo_rgb[3 * i + 2];
      m.kind = s->material[i];
      m.param = m.kind == RTCLJ_METAL ? s->fuzz[i] : s->ior[i];
      if (m.kind == RTCLJ_DIELECTRIC) {
        // material.clj:37 (/ 1.0 refraction-index) and material.clj:31 (/ (- 1.0 ri) (+ 1.0 ri)),
        // the same IEEE double operations the reference performs per hit, done once here
        const double ior = s->ior[i], inv = 1.0 / ior;
        m.albedo[0] = inv;
        m.albedo[1] = (1.0 - inv) / (1.0 + inv);
        m.albedo[2] = (1.0 - ior) / (1.0 + ior);
      }
      m.pad = 0;
      mats[(size_t)i] = m;
      const double far = std::max(std::max(std::fabs(C[0] - shift[0]), std::fabs(C[1] - shift[1])),
                                  std::max(std::fabs(C[2] - shift[2]), std::fabs(r)));
      if (far < 1e15) {
        cx = (float)(C[0] - shift[0]); cy = (float)(C[1] - shift[1]); cz = (float)(C[2] - shift[2]);
        // Ws = r^2 (1 + 8 eps) - |c|^2 (1 - 96 eps), c = the fp32-rounded shifted centre; rounded UP
        const double eps = (double)kEps32;
        const double c2 = (double)cx * cx + (double)cy * cy + (double)cz * cz;
        r2s = round_up_to_float(r * r * (1.0 + 8.0 * eps) - c2 * (1.0 - 96.0 * eps));
      } else {
        // squares beyond the fp32 range: the sphere is never culled (c = 0, Ws huge) and never
        // dropped by the fp32 prefilter; the fp64 test decides
        r2s = 3.0e38f;
      }
    }
    // pair-packed: pair p = i/2, half h = i&1 -> {cx[h], cy[2+h]} in vec0, {cz[h], r2s[2+h]} in vec1
    const int p = i >> 1, h = i & 1;
    float* v = g32.data() + (size_t)p * 8;
    v[0 + h] = cx; v[2 + h] = cy; v[4 + h] = cz; v[6 + h] = r2s;
    if (i < n) gA[(size_t)i] = make_float4(cx, cy, cz, r2s);
  }
  CU(c->geom64.reserve((size_t)std::max(n, 1)));
  CU(c->mat.reserve((size_t)std::max(n, 1)));
  CU(c->geom32.reserve((size_t)std::max(npad, 2)));
  CU(c->geomA.reserve((size_t)std::max(n, 1)));
  if (n > 0) {
    CU(cudaMemcpy(c->geom64.p, g64.data(), sizeof(Geom64) * (size_t)n, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->mat.p, mats.data(), sizeof(MatRec) * (size_t)n, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->geom32.p, g32.data(), sizeof(float) * 4 * (size_t)npad, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(c->geomA.p, gA.data(), sizeof(float4) * (size_t)n, cudaMemcpyHostToDevice));
  }
  c->n = n; c->nhalf = nhalf;
  for (int i = 0; i < std::min(n, kPrimarySpheres); ++i) {
    c->prim_geom[4 * i] = g64[(size_t)i].cx; c->prim_geom[4 * i + 1] = g64[(size_t)i].cy;
    c->prim_geom[4 * i + 2] = g64[(size_t)i].cz; c->prim_geom[4 * i + 3] = g64[(size_t)i].r;
  }
  c->ctab_host.clear();
  if (use_const_table(nhalf)) c->ctab_host.assign(g32.begin(), g32.begin() + (size_t)npad * 4);
  std::memcpy(c->shift, shift, sizeof shift);
  c->have_scene = true;
  return RTCLJ_OK;
}

}  // extern "C"

namespace {

// Scenes of <= 512 spheres: four kernels produce the same image (tests); the default is the fastest measured on
// the bench workload (DESIGN.md section 7), the flags select the others for A/B timing
enum { SMALL_LANE1, SMALL_LANE2, SMALL_WAVE, SMALL_SPLIT };
// the kernel a launch runs: none (max_depth <= 0, black), render_kernel with the table in shared memory or as a
// kernel parameter, and the other constant-table kernels
enum class Kernel { none, render_smem, render_const, lane2, wave, split, primary };
struct KernelChoice {
  Kernel kernel;
  bool primary_only;   // max_depth 1 or normal shading
  bool no_cull;        // the library adds RTCLJ_F_NO_CULL: the exhaustive fp64 scan
  bool packed;         // render_kernel's instantiation for scenes of fewer than 64 spheres
  bool finishes;       // the kernel writes the pixels itself, without finalize_kernel (wave)
  bool sample_buf_ok;  // the kernel can store every sample's colour (sample_buf)
};

bool primary_only(const rtclj_params* prm) { return prm->max_depth == 1 || (prm->flags & RTCLJ_F_NORMAL_SHADING); }

// the kernel of a launch that traces `total_samples` samples of this shard
KernelChoice choose_kernel(const rtclj_ctx* c, const rtclj_params* prm, double total_samples) {
  KernelChoice k;
  const bool const_tab = use_const_table(c->nhalf) && !(prm->flags & RTCLJ_F_SMEM_TABLE);
  // Two paths per lane pay when the cull dominates (many spheres) and the render is long enough to hide
  // the longer tail of twice as many work units in flight: measured on a B200 (profiles/r2_kernel_ab.md),
  // cover scene 1920x1080: 500 spp 543.7 vs 561.6 ms, one eighth of it (an 8-GPU shard, 1.3e8 samples) 70.85 vs
  // 71.40 ms, 16 spp (3.3e7 samples) 19.6 vs 18.6 ms; 5 spheres: 11.7 vs 11.0 ms.  Break-even near 9e7 samples.
  // (final build of round 2, 16 / 24 / 32 / 48 spp at 1920x1080: 18.48 / 26.71 / 34.86 / 51.25 against 18.50 / 27.23 /
  // 35.77 / 53.28 ms -- the break-even moved down to 3.3e7 samples; at 2e6 samples the single-path kernel is 30 % faster)
  int small = (c->n >= 64 && total_samples >= 4.0e7) ? SMALL_LANE2 : SMALL_LANE1;
#ifdef RTCLJ_DEFAULT_SMALL_KERNEL
  small = RTCLJ_DEFAULT_SMALL_KERNEL;
#endif
  if (prm->flags & RTCLJ_F_LANE_KERNEL) small = SMALL_LANE1;
  if (prm->flags & RTCLJ_F_LANE2_KERNEL) small = SMALL_LANE2;
  if (prm->flags & RTCLJ_F_WAVE_KERNEL) small = SMALL_WAVE;
  if (prm->flags & RTCLJ_F_SPLIT_KERNEL) small = SMALL_SPLIT;
  const bool lane1 = const_tab && small == SMALL_LANE1;  // one path per lane: the primary kernel or render_kernel<true>
  k.primary_only = primary_only(prm);
  if (prm->max_depth <= 0) k.kernel = Kernel::none;
  else if (!const_tab) k.kernel = Kernel::render_smem;
  else if (small == SMALL_LANE2) k.kernel = Kernel::lane2;
  else if (small == SMALL_WAVE) k.kernel = Kernel::wave;
  else if (small == SMALL_SPLIT) k.kernel = Kernel::split;
  // primary rays only and a handful of spheres (config 4): a kernel without the path machinery, 1.6x faster
  // (rtclj_primary_kernel.cuh); RTCLJ_F_LANE_KERNEL / RTCLJ_F_NO_CULL keep render_kernel for A/B and tests
  else if (lane1 && k.primary_only && c->n <= kPrimarySpheres && !(prm->flags & (RTCLJ_F_LANE_KERNEL | RTCLJ_F_NO_CULL)))
    k.kernel = Kernel::primary;
  else k.kernel = Kernel::render_const;
  // A handful of spheres: the exhaustive fp64 scan (the same lexicographic minimum, tests) beats cull +
  // prefilter.  Measured at 1920x1080 x 16 spp on prefixes of the default scene: path tracing 1 / 2 / 3 / 4
  // spheres 2.24 / 4.86 / 7.08 / 9.43 ms against 2.78 / 5.24 / 7.12 / 9.31 with the cull; primary rays only
  // 2 / 5 / 6 / 8 spheres 0.96 / 1.16 / 1.20 / 1.30 ms against 1.19 / 1.26 / 1.25 / 1.26.
  k.no_cull = lane1 && (c->n <= 2 || (k.primary_only && c->n <= kPrimarySpheres));
  // scenes of fewer than 64 spheres: their own instantiation (packed prefilter candidates, 768 threads), measured
  // per regime -- rtclj_kernels.cuh, render_kernel / threads_of
  k.packed = RTCLJ_PACKED_CANDS && k.kernel == Kernel::render_const && c->n < 64;
  k.finishes = k.kernel == Kernel::wave;
  k.sample_buf_ok = k.kernel != Kernel::none && k.kernel != Kernel::wave;
  return k;
}

// the rows of the image one render covers (rtclj_params.shard_*)
struct Shard { int index, count, rows; unsigned long long local_pixels; };
Shard shard_of(const rtclj_camera* cam, const rtclj_params* prm) {
  Shard s;
  s.count = prm->shard_count > 1 ? prm->shard_count : 1;
  s.index = s.count > 1 ? prm->shard_index : 0;
  s.rows = s.count > 1 ? prm->shard_rows : cam->height;
  s.local_pixels = (unsigned long long)local_rows_of(cam->height, s.index, s.count, s.rows) * (unsigned long long)cam->width;
  return s;
}

// One render launch: samples [sample_base, sample_base + samples) of every pixel of the shard, in work units of
// `spu` samples, then (finalize) finalize_kernel.
struct Pass {
  int sample_base = 0, samples = 0, spu = 0;
  double* sample_buf = nullptr;  // strict order: every sample's colour, added in sample order by finalize_kernel
  double* acc = nullptr;         // an accumulation's running sums (FParams::acc)
  bool seeded = false;           // strict accumulation on render_primary_kernel: the seeded variant
  int mean_n = 0;                // divisor of the pixel mean
  bool first = true;             // resets the counters and starts the timing: the first launch of a call
  bool finalize = false;
  bool listed = false;           // adaptive accumulation: listed kernels, finalize_adaptive_kernel
  bool decide = true;            // listed: the last launch of the pass applies the stopping rule and relists
  double* out_linear = nullptr;
  unsigned char* out_rgb8 = nullptr;
  // a camera sequence: the launch traces the units of frames[0 .. n_frames) (frame twins, FrameKParams), and the
  // images above hold n_frames full-size frames.  n_frames = 0: the single camera of launch_pass.
  const rtclj_camera* frames = nullptr;
  int n_frames = 0;
};

// the fold and stopping rule of an adaptive accumulation's pass, shard `sh` (finalize_adaptive_kernel)
AParams adaptive_params(const rtclj_ctx* c, const Shard& sh) {
  AParams A;
  std::memset(&A, 0, sizeof A);
  const auto& acc = c->accum;
  A.W = acc.cam.width; A.shard_index = sh.index; A.shard_count = sh.count; A.shard_rows = sh.rows;
  A.flags = acc.prm.flags; A.local_pixels = sh.local_pixels; A.sample_stride = sh.local_pixels;
  A.acc = c->acc.p; A.acc2 = c->acc2.p; A.samples = c->nsamp.p; A.live = c->live.p;
  A.strict = acc.strict; A.unit = acc.pass_unit; A.target = acc.prm.spp; A.min_samples = acc.min_samples;
  A.abs_tol = acc.abs_tol; A.rel_tol = acc.rel_tol;
  return A;
}

// rebuilds the list of live pixels and its count on the device (rtclj_adaptive.cuh)
int relist(rtclj_ctx* c, unsigned long long local_pixels, cudaStream_t stream) {
  CU(launch_relist(c->live.p, local_pixels, c->list_aux.p, c->list.p, stream));
  return RTCLJ_OK;
}

int launch_pass(rtclj_ctx* c, const rtclj_camera* cam, const rtclj_params* prm, const KernelChoice& ch, const Shard& sh,
                const Pass& ps, cudaStream_t stream) {
  const int grid = c->sm_count;
  const int nchunks = (ps.samples + ps.spu - 1) / ps.spu;
  const int nframes = ps.n_frames > 0 ? ps.n_frames : 1;
  const unsigned long long total_units = sh.local_pixels * (unsigned long long)nchunks * (unsigned long long)nframes;
  if (total_units > 0xffffffffull) {
    return fail(RTCLJ_E_INVALID, "%llu work units: raise samples_per_unit", total_units);
  }

  // a later launch of the same call resets the ticket queue only: the counters add up over the call
  CU(cudaMemsetAsync(c->counters.p, 0, (ps.first ? 8 : 1) * sizeof(unsigned long long), stream));
  if (total_units == 0) return RTCLJ_OK;

  if ((!ch.finishes || nchunks > 1) && !ps.sample_buf) CU(c->partial.reserve((size_t)total_units * 3));
  if (ps.first) CU(cudaEventRecord(c->ev0, stream));
  if (ch.kernel == Kernel::none) {
    CU(cudaMemsetAsync(c->partial.p, 0, (size_t)total_units * 3 * sizeof(double), stream));  // depth <= 0: black
  } else {
    KParams& P = c->kparams;  // 8.4 KB with the table: kept in the context, not on the stack of a JVM thread
    std::memset(&P, 0, offsetof(KParams, ctab));
    for (int a = 0; a < 3; ++a) {
      P.p00[a] = cam->pixel00[a]; P.du[a] = cam->pixel_du[a]; P.dv[a] = cam->pixel_dv[a];
      P.center[a] = cam->center[a]; P.ddu[a] = cam->defocus_u[a]; P.ddv[a] = cam->defocus_v[a];
      P.shift[a] = c->shift[a];
    }
    P.use_defocus = !(cam->defocus_angle <= 0.0);
    P.W = cam->width; P.H = cam->height; P.spp = ps.sample_base + ps.samples; P.max_depth = prm->max_depth;
    P.flags = prm->flags; P.k0 = (unsigned)prm->seed; P.k1 = (unsigned)(prm->seed >> 32);
    for (unsigned r = 0; r < 10; ++r) { P.rk[2 * r] = P.k0 + r * 0x9E3779B9u; P.rk[2 * r + 1] = P.k1 + r * 0xBB67AE85u; }
    if (ch.no_cull) P.flags |= RTCLJ_F_NO_CULL;
    P.n = c->n; P.nblocks = c->nhalf / 2; P.tail8 = c->nhalf & 1;
    P.nconst = (c->n + 2 * kCBP - 1) / (2 * kCBP);
    P.smem_blocks = smem_table_blocks(c->smem_optin);
    P.geom_bytes = (unsigned)std::min((size_t)c->nhalf * 256, (size_t)P.smem_blocks * 512);  // staged part
    P.shard_index = sh.index; P.shard_count = sh.count; P.shard_rows = sh.rows;
    P.nchunks = nchunks; P.spu = ps.spu; P.sample_base = ps.sample_base; P.total_units = total_units;
    P.geom32 = c->geom32.p; P.geomA = c->geomA.p; P.geom64 = c->geom64.p; P.mat = c->mat.p;
    P.partial = c->partial.p; P.acc = ps.acc; P.queue = c->counters.p; P.stats = c->counters.p + 1;
    P.sample_buf = ps.sample_buf; P.sample_stride = sh.local_pixels * (unsigned long long)nframes;
    P.list = ps.listed ? c->list.p : nullptr; P.list_count = ps.listed ? c->list_aux.p : nullptr;
    P.acc2 = ps.listed ? c->acc2.p : nullptr;
    const bool const_tab = ch.kernel != Kernel::render_smem, sample_buf = ps.sample_buf != nullptr;
    if (const_tab && !c->ctab_host.empty())
      std::memcpy(P.ctab, c->ctab_host.data(), std::min(sizeof P.ctab, c->ctab_host.size() * sizeof(float)));
    KernelFn fn = nullptr;
    FramesFn frames_fn = nullptr;
    bool any_defocus = false;  // a sequence: some frame has the defocus disk
    for (int f = 0; f < ps.n_frames; ++f) any_defocus = any_defocus || !(ps.frames[f].defocus_angle <= 0.0);
    unsigned blocks = (unsigned)grid, paths = 0;  // paths in flight per CTA: the rows of the attenuation stack
    int threads = 0;
    size_t sm = 0;
    bool stack = prm->max_depth > 1;  // the attenuating hits of a path, for either product order
    switch (ch.kernel) {
      case Kernel::primary: {
        std::memcpy(P.ctab, c->prim_geom, sizeof c->prim_geom);
        const unsigned long long want = (total_units + kPrimaryThreads - 1) / kPrimaryThreads;
        blocks = (unsigned)std::min<unsigned long long>(want, (unsigned long long)grid * (unsigned long long)(2048 / kPrimaryThreads));
        fn = kPrimaryFns[ps.listed][ps.seeded][P.use_defocus]; threads = kPrimaryThreads; stack = false;
        frames_fn = kPrimaryFramesFns[any_defocus];
        break;
      }
      case Kernel::wave:
        fn = kWaveFns[0]; threads = kWT; sm = WaveSmem::total; paths = kWS;
        P.out_linear = ps.out_linear; P.out_rgb8 = ps.out_rgb8;
        if (nchunks > 1 && (ps.out_linear || ps.out_rgb8)) {
          CU(c->arrive.reserve((size_t)sh.local_pixels));
          CU(cudaMemsetAsync(c->arrive.p, 0, (size_t)sh.local_pixels * sizeof(unsigned), stream));
          P.arrive = c->arrive.p;
        }
        break;
      case Kernel::split:
        fn = kSplitFns[sample_buf]; threads = kSplitThreads; sm = SplitSmem::total; paths = 2u * kSplitW;
        break;
      case Kernel::lane2:
        fn = kLane2Fns[ps.listed][sample_buf]; threads = kT2; sm = Lane2Smem::total; paths = 2u * kT2;
        frames_fn = kLane2FramesFns[sample_buf];
        break;
      default:  // render_kernel
        fn = kRenderFns[ps.listed][const_tab][sample_buf][ch.packed]; threads = threads_of(const_tab, ch.packed);
        sm = smem_needed(c->nhalf, const_tab, c->smem_optin, ch.packed); paths = (unsigned)threads;
        frames_fn = kRenderFramesFns[const_tab][sample_buf][ch.packed];
        stack = prm->flags & RTCLJ_F_REVERSE_PRODUCT;
    }
    P.stack_stride = (unsigned)grid * paths;
    if (stack) {
      CU(c->stack.reserve((size_t)prm->max_depth * P.stack_stride));
      P.stack = c->stack.p;
    }
#ifdef RTCLJ_TAIL_PROBE
    const size_t probe_words = (size_t)grid * (kT2 / 32) * 4 * 2;
    if (ch.kernel == Kernel::lane2) {
      CU(c->arrive.reserve(probe_words));
      CU(cudaMemsetAsync(c->arrive.p, 0, probe_words * sizeof(unsigned), stream));
      P.arrive = c->arrive.p;
    }
#endif
    if (ps.n_frames > 0) {
      if (!frames_fn) return fail(RTCLJ_E_INVALID, "this kernel renders no camera sequences");
      FrameKParams& F = c->fparams;
      F.P = P;
      F.frame_pixels = (unsigned)sh.local_pixels;
      F.frame_units = (unsigned)(sh.local_pixels * (unsigned long long)nchunks);
      for (int f = 0; f < ps.n_frames; ++f) {  // the fields launch_pass sets from a camera, in the same way
        const rtclj_camera& fc = ps.frames[f];
        FrameCam& fr = F.cam[f];
        for (int a = 0; a < 3; ++a) {
          fr.p00[a] = fc.pixel00[a]; fr.du[a] = fc.pixel_du[a]; fr.dv[a] = fc.pixel_dv[a];
          fr.center[a] = fc.center[a]; fr.ddu[a] = fc.defocus_u[a]; fr.ddv[a] = fc.defocus_v[a];
        }
        fr.use_defocus = !(fc.defocus_angle <= 0.0);
        fr.pad = 0;
      }
      frames_fn<<<blocks, threads, sm, stream>>>(F);
    } else {
      fn<<<blocks, threads, sm, stream>>>(P);
    }
#ifdef RTCLJ_TAIL_PROBE
    if (const char* path = std::getenv("RTCLJ_TAIL_PROBE_FILE"); path && ch.kernel == Kernel::lane2) {
      std::vector<unsigned> host(probe_words);
      CU(cudaStreamSynchronize(stream));
      CU(cudaMemcpy(host.data(), c->arrive.p, probe_words * sizeof(unsigned), cudaMemcpyDeviceToHost));
      if (FILE* f = std::fopen(path, "wb")) { std::fwrite(host.data(), sizeof(unsigned), probe_words, f); std::fclose(f); }
    }
#endif
    CU(cudaGetLastError());
  }
  CU(cudaEventRecord(c->ev1, stream));
  if (ps.finalize && ps.listed) {
    AParams A = adaptive_params(c, sh);
    A.sample_buf = ps.sample_buf; A.partial = c->partial.p; A.out_linear = ps.out_linear; A.out_rgb8 = ps.out_rgb8;
    A.spp = ps.samples; A.nchunks = nchunks; A.seeded = ps.seeded; A.mean_n = ps.mean_n; A.decide = ps.decide;
    const unsigned blocks = (unsigned)((sh.local_pixels + 255) / 256);
    finalize_adaptive_kernel<<<blocks, 256, 0, stream>>>(A);
    CU(cudaGetLastError());
    if (ps.decide) {
      int rc = relist(c, sh.local_pixels, stream);
      if (rc) return rc;
    }
  } else if (ps.finalize) {
    // one finalize_kernel per frame, on that frame's unit sums / sample colours and full-size images
    const size_t frame_values = (size_t)cam->width * (size_t)cam->height * 3u;
    for (int f = 0; f < nframes; ++f) {
      FParams F;
      F.sample_buf = ps.sample_buf ? ps.sample_buf + (size_t)f * sh.local_pixels * 4u : nullptr;
      F.sample_stride = sh.local_pixels * (unsigned long long)nframes;
      F.partial = c->partial.p + (size_t)f * sh.local_pixels * (size_t)nchunks * 3u;
      F.out_linear = ps.out_linear ? ps.out_linear + (size_t)f * frame_values : nullptr;
      F.out_rgb8 = ps.out_rgb8 ? ps.out_rgb8 + (size_t)f * frame_values : nullptr;
      F.W = cam->width; F.spp = ps.samples; F.nchunks = nchunks;
      F.shard_index = sh.index; F.shard_count = sh.count; F.shard_rows = sh.rows;
      F.flags = prm->flags; F.local_pixels = sh.local_pixels;
      F.acc = ps.acc; F.seeded = ps.seeded; F.mean_n = ps.mean_n;
      const unsigned blocks = (unsigned)((sh.local_pixels + 255) / 256);
      finalize_kernel<<<blocks, 256, 0, stream>>>(F);
      CU(cudaGetLastError());
    }
  }
  CU(cudaEventRecord(c->ev2, stream));
  c->render_pending = true;
  return RTCLJ_OK;
}

// The strict order of the general kernels goes through sample_buf (32 B per pixel and sample); an
// accumulation's pass that needs more is cut into sub-passes of at most this many bytes, each followed by its
// fold, and a camera sequence groups no more frames into one launch than this buffer -- or their unit sums -- holds.
// A one-shot strict render of 1920x1080 x 500 spp holds 33 GB; a strict accumulation or sequence never more than this.
constexpr size_t kAccumSampleBufBytes = (size_t)2 << 30;

// The strict order on long paths: one 500-sample unit lasts as long as its pixel's paths, the last ones run alone
// (measured: 622 vs 543 ms on one GPU, 162 vs 72 ms per GPU on eight).  Instead the samples are traced in small units
// and each sample's colour is STORED (32 B); finalize_kernel then adds them in sample order -- the same additions in
// the same order.  33 GB at 1920x1080 x 500 spp; HBM has 180 GB.  Returns the buffer of `need` doubles for a render
// that wants it (nullptr if it does not fit: one unit per pixel then); a render that does not gives a large one back.
double* strict_sample_buf(rtclj_ctx* c, bool wanted, size_t need) {
  if (wanted) {
    size_t free_b = 0, total_b = 0;
    // kept in the context between renders (allocating 33 GB per frame costs more than the frame)
    if (need <= c->sample_buf.cap ||
        (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && need * 8 < (free_b + c->sample_buf.cap * 8) / 2 &&
         c->sample_buf.reserve(need) == cudaSuccess))
      return c->sample_buf.p;
    cudaGetLastError();  // too large: fall back to one unit per pixel
  } else if (c->sample_buf.cap * 8 > ((size_t)1 << 30)) {
    c->sample_buf.release();  // (synchronises the device; only on a strict -> chunked change of mode)
  }
  return nullptr;
}

// The checks of a camera sequence, before any device is touched: frame f fails validate() under its own number
int check_frames(const rtclj_camera* cams, int32_t n_frames, const rtclj_params* prm) {
  if (n_frames <= 0) return fail(RTCLJ_E_INVALID, "n_frames must be positive, got %d", n_frames);
  if (!cams) return fail(RTCLJ_E_INVALID, "null camera array");
  if (!prm) return fail(RTCLJ_E_INVALID, "null params");
  if (prm->flags & (RTCLJ_F_WAVE_KERNEL | RTCLJ_F_SPLIT_KERNEL))
    return fail(RTCLJ_E_INVALID, "the wavefront and split kernels do not render camera sequences");
  for (int f = 0; f < n_frames; ++f) {
    if (validate(&cams[f], prm)) {
      char why[256];
      std::snprintf(why, sizeof why, "%s", rtclj_error_get());
      return fail(RTCLJ_E_INVALID, "frame %d: %s", f, why);
    }
    if (cams[f].width != cams[0].width || cams[f].height != cams[0].height)
      return fail(RTCLJ_E_INVALID, "frame %d is %dx%d, frame 0 %dx%d: a sequence has one image size", f, cams[f].width,
                  cams[f].height, cams[0].width, cams[0].height);
  }
  return RTCLJ_OK;
}

}  // namespace

extern "C" {

int rtclj_ctx_render(rtclj_ctx* c, const rtclj_camera* cam, const rtclj_params* prm, void* d_out_linear,
                     void* d_out_rgb8, void* stream_) {
  if (!c) return fail(RTCLJ_E_INVALID, "null ctx");
  if (!c->have_scene) return fail(RTCLJ_E_INVALID, "rtclj_ctx_set_scene has not been called");
  int rc = validate(cam, prm);
  if (rc) return rc;
  cudaStream_t stream = (cudaStream_t)stream_;
  CU(cudaSetDevice(c->device));

  const int W = cam->width, H = cam->height;
  const Shard sh = shard_of(cam, prm);
  const bool want_out = d_out_linear || d_out_rgb8;
  const KernelChoice ch = choose_kernel(c, prm, (double)sh.local_pixels * (double)prm->spp);

  // Summation unit.  Primary-ray renders (max-depth 1, normal shading) are bit-exact contracts and short
  // paths: they default to the reference's strict sequential sum (raytracing.clj:142-155,
  // raytracing_i.clj:146-163); other renders split a pixel into chunks for load balance.
  int spu = prm->samples_per_unit > 0 ? prm->samples_per_unit
                                      : (ch.primary_only ? prm->spp : auto_samples_per_unit(W, H, prm->spp));
  if (spu > prm->spp) spu = prm->spp;
  c->last_spu = spu;
  const bool strict_long = spu == prm->spp && !ch.primary_only && prm->spp >= 64 && ch.sample_buf_ok && want_out &&
                           sh.local_pixels > 0;
  double* sample_buf = strict_sample_buf(c, strict_long, (size_t)sh.local_pixels * (size_t)prm->spp * 4u);
  if (sample_buf) spu = auto_samples_per_unit(W, H, prm->spp);  // scheduling units; the arithmetic stays strict
  Pass ps;
  ps.samples = prm->spp; ps.spu = spu; ps.sample_buf = sample_buf; ps.mean_n = prm->spp;
  ps.finalize = !ch.finishes && want_out;
  ps.out_linear = (double*)d_out_linear; ps.out_rgb8 = (unsigned char*)d_out_rgb8;
  return launch_pass(c, cam, prm, ch, sh, ps, stream);
}

// A camera sequence (DESIGN.md section 4.12): the frames share launches -- one ticket queue, one tail -- in groups
// whose scratch (unit sums, or sample colours in strict order) stays within kAccumSampleBufBytes, whose units stay
// below 2^32 and whose cameras fit the kernel parameters (kMaxFrames).  The summation unit and the strict-order
// decision are the single frame's, so frame f is bit-identical to rtclj_ctx_render with cameras[f]; a frame that
// alone needs more scratch runs as a group of one under rtclj_ctx_render's rules.
int rtclj_ctx_render_frames(rtclj_ctx* c, const rtclj_camera* cams, int32_t n_frames, const rtclj_params* prm,
                            void* d_out_linear, void* d_out_rgb8, void* stream_) {
  if (!c) return fail(RTCLJ_E_INVALID, "null ctx");
  if (!c->have_scene) return fail(RTCLJ_E_INVALID, "rtclj_ctx_set_scene has not been called");
  int rc = check_frames(cams, n_frames, prm);
  if (rc) return rc;
  cudaStream_t stream = (cudaStream_t)stream_;
  CU(cudaSetDevice(c->device));

  const int W = cams[0].width, H = cams[0].height;
  const Shard sh = shard_of(&cams[0], prm);
  const bool want_out = d_out_linear || d_out_rgb8;
  // every kernel gives the same bits: the choice may see the whole batch
  const KernelChoice ch = choose_kernel(c, prm, (double)n_frames * (double)sh.local_pixels * (double)prm->spp);
  // the summation unit of ONE frame, as rtclj_ctx_render computes it
  int spu = prm->samples_per_unit > 0 ? prm->samples_per_unit
                                      : (ch.primary_only ? prm->spp : auto_samples_per_unit(W, H, prm->spp));
  if (spu > prm->spp) spu = prm->spp;
  c->last_spu = spu;
  const bool strict_long = spu == prm->spp && !ch.primary_only && prm->spp >= 64 && ch.sample_buf_ok && want_out &&
                           sh.local_pixels > 0;
  const int sched_spu = strict_long ? auto_samples_per_unit(W, H, prm->spp) : spu;
  const unsigned long long frame_units =
      sh.local_pixels * (unsigned long long)((prm->spp + sched_spu - 1) / sched_spu);
  const unsigned long long frame_bytes = strict_long ? sh.local_pixels * (unsigned long long)prm->spp * 32ull
                                                     : frame_units * 24ull;
  unsigned long long group = std::min<unsigned long long>((unsigned long long)n_frames, kMaxFrames);
  if (frame_bytes > 0) group = std::min(group, std::max(1ull, kAccumSampleBufBytes / frame_bytes));
  if (frame_units > 0) group = std::min(group, std::max(1ull, 0xffffffffull / frame_units));
  const size_t frame_values = (size_t)W * (size_t)H * 3u;
  for (int f0 = 0; f0 < n_frames; f0 += (int)group) {
    const int g = std::min((int)group, n_frames - f0);
    double* sample_buf = strict_sample_buf(c, strict_long, (size_t)g * (size_t)sh.local_pixels * (size_t)prm->spp * 4u);
    Pass ps;
    ps.samples = prm->spp; ps.spu = sample_buf ? sched_spu : spu; ps.sample_buf = sample_buf; ps.mean_n = prm->spp;
    ps.first = f0 == 0;
    ps.finalize = !ch.finishes && want_out;
    ps.out_linear = d_out_linear ? (double*)d_out_linear + (size_t)f0 * frame_values : nullptr;
    ps.out_rgb8 = d_out_rgb8 ? (unsigned char*)d_out_rgb8 + (size_t)f0 * frame_values : nullptr;
    ps.frames = cams + f0; ps.n_frames = g;
    rc = launch_pass(c, &cams[f0], prm, ch, sh, ps, stream);
    if (rc) return rc;
  }
  return RTCLJ_OK;
}

int rtclj_ctx_stats(rtclj_ctx* c, void* stream_, rtclj_stats* st) {
  if (!c || !st) return fail(RTCLJ_E_INVALID, "null ctx or stats");
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize((cudaStream_t)stream_));
  unsigned long long h[8];
  CU(cudaMemcpy(h, c->counters.p, sizeof h, cudaMemcpyDeviceToHost));
  std::memset(st, 0, sizeof *st);
  st->samples = h[1]; st->segments = h[2]; st->exact_tests = h[3]; st->list_overflows = h[4];
  st->prefilter_tests = h[5];
  float ms = 0.f;
  if (cudaEventElapsedTime(&ms, c->ev0, c->ev2) == cudaSuccess) st->device_ms = ms; else cudaGetLastError();
  if (cudaEventElapsedTime(&ms, c->ev0, c->ev1) == cudaSuccess) st->kernel_ms = ms; else cudaGetLastError();
  st->samples_per_unit = c->last_spu;
  st->n_devices = 1;
  c->render_pending = false;
  return RTCLJ_OK;
}

// ---------------------------------------------------------------- downloads into caller memory
// A shard owns tiles of `shard_rows` rows at a regular pitch (shard_count tiles apart); the device image
// has the full-size layout, so device and host offsets are the same.  Caller memory that CUDA knows as
// pinned (rtclj_host_alloc / rtclj_host_register / cudaHostAlloc) is written directly by asynchronous
// copies.  Pageable memory (numpy, malloc, a JVM Arena) goes through two pinned staging buffers of the
// context, pipelined: the device fills one while the host unpacks the other -- a device-to-pageable
// cudaMemcpyAsync would block the calling thread until the render in front of it has finished.
}  // extern "C"

namespace {

struct Piece { size_t off, pitch, width, height; };  // `height` runs of `width` bytes, `pitch` apart, from `off`

void plan_pieces(size_t H, size_t row_bytes, int shard_index, int shard_count, int shard_rows, size_t cap,
                 std::vector<Piece>& out) {
  if (shard_count <= 1) { shard_index = 0; shard_count = 1; shard_rows = (int)H; }
  const size_t sr = (size_t)shard_rows;
  const size_t ntiles = (H + sr - 1) / sr;
  if ((size_t)shard_index >= ntiles) return;
  const size_t mine = (ntiles - (size_t)shard_index + (size_t)shard_count - 1) / (size_t)shard_count;
  const size_t last = (size_t)shard_index + (mine - 1) * (size_t)shard_count;  // this shard's last tile
  const size_t last_rows = std::min(sr, H - last * sr);
  const size_t full = last_rows == sr ? mine : mine - 1;  // tiles of exactly shard_rows rows
  const size_t tile_bytes = sr * row_bytes, pitch = (size_t)shard_count * tile_bytes;
  const size_t first = (size_t)shard_index * tile_bytes;
  auto split = [&](size_t off, size_t bytes) {  // one contiguous run, in pieces of at most `cap` bytes
    for (size_t o = 0; o < bytes; o += cap) out.push_back(Piece{off + o, 0, std::min(cap, bytes - o), 1});
  };
  if (tile_bytes >= cap) {
    for (size_t t = 0; t < full; ++t) split(first + t * pitch, tile_bytes);
  } else {
    const size_t group = cap / tile_bytes;  // whole tiles per piece: one strided 2-D copy
    for (size_t t = 0; t < full; t += group) out.push_back(Piece{first + t * pitch, pitch, tile_bytes, std::min(group, full - t)});
  }
  if (full != mine) split(last * tile_bytes, last_rows * row_bytes);
}

bool is_pinned(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return at.type == cudaMemoryTypeHost;
}

constexpr size_t kStageBytes = 16u << 20;

int download_image(rtclj_ctx* c, const std::vector<Piece>& pieces, char* host, const char* dev, cudaStream_t stream) {
  if (pieces.empty()) return RTCLJ_OK;
  if (is_pinned(host)) {  // asynchronous all the way: the caller's stats call synchronises
    for (const Piece& p : pieces) {
      if (p.height == 1) CU(cudaMemcpyAsync(host + p.off, dev + p.off, p.width, cudaMemcpyDeviceToHost, stream));
      else CU(cudaMemcpy2DAsync(host + p.off, p.pitch, dev + p.off, p.pitch, p.width, p.height, cudaMemcpyDeviceToHost, stream));
    }
    return RTCLJ_OK;
  }
  if (!c->pin[0]) {
    CU(cudaHostAlloc(&c->pin[0], kStageBytes, cudaHostAllocDefault));
    CU(cudaHostAlloc(&c->pin[1], kStageBytes, cudaHostAllocDefault));
    c->pin_cap = kStageBytes;
  }
  auto unpack = [&](size_t i) {
    const Piece& p = pieces[i];
    const char* src = (const char*)c->pin[i & 1];
    for (size_t r = 0; r < p.height; ++r) std::memcpy(host + p.off + r * p.pitch, src + r * p.width, p.width);
  };
  for (size_t i = 0; i < pieces.size(); ++i) {
    const int b = (int)(i & 1);
    if (i >= 2) { CU(cudaEventSynchronize(c->pin_ev[b])); unpack(i - 2); }  // this buffer's previous piece
    const Piece& p = pieces[i];
    if (p.height == 1) CU(cudaMemcpyAsync(c->pin[b], dev + p.off, p.width, cudaMemcpyDeviceToHost, stream));
    else CU(cudaMemcpy2DAsync(c->pin[b], p.width, dev + p.off, p.pitch, p.width, p.height, cudaMemcpyDeviceToHost, stream));
    CU(cudaEventRecord(c->pin_ev[b], stream));
  }
  for (size_t i = pieces.size() >= 2 ? pieces.size() - 2 : 0; i < pieces.size(); ++i) {
    CU(cudaEventSynchronize(c->pin_ev[i & 1]));
    unpack(i);
  }
  return RTCLJ_OK;
}

// frame f of a camera sequence: the f-th full-size image of the device buffers and of the caller's
int download_rows(rtclj_ctx* c, const rtclj_camera* cam, int shard_index, int shard_count, int shard_rows,
                  double* out_linear, uint8_t* out_rgb8, cudaStream_t stream, int frame = 0) {
  const size_t W = (size_t)cam->width, H = (size_t)cam->height;
  const size_t frame_values = W * H * 3 * (size_t)frame;
  std::vector<Piece> pieces;
  if (out_linear) {
    plan_pieces(H, W * 3 * sizeof(double), shard_index, shard_count, shard_rows, kStageBytes, pieces);
    int rc = download_image(c, pieces, (char*)(out_linear + frame_values), (const char*)(c->out_linear.p + frame_values), stream);
    if (rc) return rc;
  }
  if (out_rgb8) {
    pieces.clear();
    plan_pieces(H, W * 3, shard_index, shard_count, shard_rows, kStageBytes, pieces);
    int rc = download_image(c, pieces, (char*)(out_rgb8 + frame_values), (const char*)(c->out_rgb8.p + frame_values), stream);
    if (rc) return rc;
  }
  return RTCLJ_OK;
}

// One cached context per device for the host-buffer entry points, each behind its OWN lock: calls on
// different devices overlap (rtclj_render_multi, or a host that gives each pool thread a GPU), calls on
// one device queue up.
std::mutex g_ctx_mu;
struct DeviceSlot { std::mutex mu; rtclj_ctx* ctx = nullptr; };
std::vector<std::unique_ptr<DeviceSlot>> g_slots;

// the cached context of `device`, created on first use; `lock` holds the device's slot when this returns
int cached_ctx(int device, std::unique_lock<std::mutex>& lock, rtclj_ctx** ctx) {
  int ndev = 0;
  int rc = rtclj_device_count(&ndev);
  if (rc) return rc;
  if (ndev == 0) return fail(RTCLJ_E_NO_DEVICE, "no CUDA device (this library has no CPU fallback)");
  if (device < 0 || device >= ndev) return fail(RTCLJ_E_INVALID, "device %d out of range [0,%d)", device, ndev);
  DeviceSlot* slot = nullptr;
  {
    std::lock_guard<std::mutex> lk(g_ctx_mu);
    if ((int)g_slots.size() < ndev) g_slots.resize((size_t)ndev);
    if (!g_slots[(size_t)device]) g_slots[(size_t)device].reset(new DeviceSlot());
    slot = g_slots[(size_t)device].get();
  }
  lock = std::unique_lock<std::mutex>(slot->mu);
  if (!slot->ctx) { rc = rtclj_ctx_create(device, &slot->ctx); if (rc) return rc; }
  *ctx = slot->ctx;
  return RTCLJ_OK;
}

// scene upload + render of one shard + download into the caller's images, on one device.  n_frames > 0: the camera
// sequence cam[0 .. n_frames) (rtclj_ctx_render_frames), the images hold n_frames frames
int render_shard_hostbuf(const rtclj_scene* scene, const rtclj_camera* cam, const rtclj_params* prm, double* out_linear,
                         uint8_t* out_rgb8, rtclj_stats* stats, int n_frames = 0) {
  const auto t0 = std::chrono::steady_clock::now();
  std::unique_lock<std::mutex> lock;
  rtclj_ctx* c = nullptr;
  int rc = cached_ctx(prm->device, lock, &c);
  if (rc) return rc;
  rc = rtclj_ctx_set_scene(c, scene);
  if (rc) return rc;
  const size_t nimg = (size_t)cam->width * (size_t)cam->height * 3 * (size_t)std::max(n_frames, 1);
  if (out_linear) CU(c->out_linear.reserve(nimg));
  if (out_rgb8) CU(c->out_rgb8.reserve(nimg));
  double* d_lin = out_linear ? c->out_linear.p : nullptr;
  unsigned char* d_rgb = out_rgb8 ? c->out_rgb8.p : nullptr;
  rc = n_frames > 0 ? rtclj_ctx_render_frames(c, cam, n_frames, prm, d_lin, d_rgb, c->own_stream)
                    : rtclj_ctx_render(c, cam, prm, d_lin, d_rgb, c->own_stream);
  if (rc) return rc;
  for (int f = 0; f < std::max(n_frames, 1); ++f) {
    rc = download_rows(c, cam, prm->shard_index, prm->shard_count, prm->shard_rows, out_linear, out_rgb8, c->own_stream, f);
    if (rc) return rc;
  }
  rtclj_stats s;
  rc = rtclj_ctx_stats(c, c->own_stream, &s);  // synchronises the stream: the direct copies have landed
  if (rc) return rc;
  s.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  if (stats) *stats = s;
  return RTCLJ_OK;
}

// the device list of a multi-GPU call: not empty, every ordinal valid and listed once
int check_devices(const int32_t* devices, int32_t n_devices) {
  if (n_devices <= 0 || !devices) return fail(RTCLJ_E_INVALID, "empty device list");
  int ndev = 0;
  int rc = rtclj_device_count(&ndev);
  if (rc) return rc;
  if (ndev == 0) return fail(RTCLJ_E_NO_DEVICE, "no CUDA device (this library has no CPU fallback)");
  for (int d = 0; d < n_devices; ++d) {
    if (devices[d] < 0 || devices[d] >= ndev) return fail(RTCLJ_E_INVALID, "device %d out of range [0,%d)", devices[d], ndev);
    for (int e = 0; e < d; ++e)
      if (devices[e] == devices[d]) return fail(RTCLJ_E_INVALID, "device %d listed twice", devices[d]);
  }
  return RTCLJ_OK;
}

// the counters of a multi-GPU call: the devices' counts add up, the times are the slowest device's
rtclj_stats sum_stats(const std::vector<rtclj_stats>& st) {
  rtclj_stats total;
  std::memset(&total, 0, sizeof total);
  for (const rtclj_stats& s : st) {
    total.samples += s.samples; total.segments += s.segments; total.exact_tests += s.exact_tests;
    total.list_overflows += s.list_overflows; total.prefilter_tests += s.prefilter_tests;
    total.device_ms = std::max(total.device_ms, s.device_ms);
    total.kernel_ms = std::max(total.kernel_ms, s.kernel_ms);
    total.samples_per_unit = s.samples_per_unit;
  }
  total.n_devices = (int32_t)st.size();
  return total;
}

// the rtclj_params of devices[d] in a call on n devices: its shard of the rows
rtclj_params shard_params(const rtclj_params* prm, const int32_t* devices, int d, int n) {
  rtclj_params q = *prm;
  q.device = devices[d];
  if (n > 1) {
    q.shard_index = d; q.shard_count = n;
    q.shard_rows = prm->shard_rows > 0 ? prm->shard_rows : 1;  // 1-row tiles balance best (DESIGN.md 6)
  } else {
    q.shard_index = 0; q.shard_count = 1; q.shard_rows = 0;
  }
  return q;
}

// nothing may throw across the C boundary (a JVM host would die): bad_alloc etc. become error codes
template <class F>
int guarded(F&& f) {
  try { return f(); }
  catch (const std::bad_alloc&) { return fail(RTCLJ_E_CUDA, "out of host memory"); }
  catch (const std::exception& e) { return fail(RTCLJ_E_CUDA, "unexpected exception: %s", e.what()); }
  catch (...) { return fail(RTCLJ_E_CUDA, "unexpected exception"); }
}

// fn(d) for d = 0 .. n-1 at once: a worker thread for each d > 0, d = 0 on the calling thread.  Returns the code
// of the lowest d that failed, with its message (which is thread-local: carried over)
template <class F>
int run_on_devices(int n, F&& fn) {
  std::vector<int> rcs((size_t)n, RTCLJ_OK);
  std::vector<std::string> msgs((size_t)n);
  auto work = [&](int d) {
    rcs[(size_t)d] = guarded([&]() { return fn(d); });
    if (rcs[(size_t)d]) msgs[(size_t)d] = rtclj_error_get();
  };
  std::vector<std::thread> pool;
  for (int d = 1; d < n; ++d) pool.emplace_back(work, d);
  work(0);
  for (std::thread& t : pool) t.join();
  for (int d = 0; d < n; ++d)
    if (rcs[(size_t)d]) { rtclj_error_set(msgs[(size_t)d].c_str()); return rcs[(size_t)d]; }
  return RTCLJ_OK;
}

// the checks of a pass of `samples` samples per pixel after `done`, towards `spp`, in pass units of `unit`
int check_pass(int done, int samples, int spp, int unit) {
  if (samples <= 0) return fail(RTCLJ_E_INVALID, "a pass needs a positive sample count, got %d", samples);
  if ((long long)done + samples > (long long)spp)
    return fail(RTCLJ_E_INVALID, "pass of %d samples after %d: beyond the target of %d", samples, done, spp);
  if (done + samples != spp && samples % unit != 0)
    return fail(RTCLJ_E_INVALID, "pass of %d samples: every pass but the last must be a multiple of pass_unit = %d",
                samples, unit);
  return RTCLJ_OK;
}

}  // namespace

extern "C" {

// The image rows interleaved over several GPUs, driven by this ONE process -- what a JVM host calls
// where the reference starts its pool (src/raytracing.clj:157-171).  One worker thread per device runs
// upload -> render -> download for its shard, so the devices render AND copy at the same time; the
// shards' rows are disjoint, the image needs no further gather.
int rtclj_render_multi(const rtclj_scene* scene, const rtclj_camera* cam, const rtclj_params* prm,
                       const int32_t* devices, int32_t n_devices, double* out_linear, uint8_t* out_rgb8,
                       rtclj_stats* stats) {
  return guarded([&]() -> int {
    const auto t0 = std::chrono::steady_clock::now();
    if (!scene) return fail(RTCLJ_E_INVALID, "null scene");
    int rc = validate(cam, prm);
    if (rc) return rc;
    rc = check_devices(devices, n_devices);
    if (rc) return rc;
    std::vector<rtclj_stats> st((size_t)n_devices);
    rc = run_on_devices(n_devices, [&](int d) {
      const rtclj_params q = shard_params(prm, devices, d, n_devices);
      return render_shard_hostbuf(scene, cam, &q, out_linear, out_rgb8, &st[(size_t)d]);
    });
    if (rc) return rc;
    rtclj_stats total = sum_stats(st);
    total.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats) *stats = total;
    return RTCLJ_OK;
  });
}

// A camera sequence on host buffers: rtclj_render_multi's rows and workers, each device renders its rows of every
// frame with rtclj_ctx_render_frames and downloads them frame by frame.
int rtclj_render_frames(const rtclj_scene* scene, const rtclj_camera* cams, int32_t n_frames, const rtclj_params* prm,
                        const int32_t* devices, int32_t n_devices, double* out_linear, uint8_t* out_rgb8,
                        rtclj_stats* stats) {
  return guarded([&]() -> int {
    const auto t0 = std::chrono::steady_clock::now();
    if (!scene) return fail(RTCLJ_E_INVALID, "null scene");
    int rc = check_frames(cams, n_frames, prm);
    if (rc) return rc;
    rc = check_devices(devices, n_devices);
    if (rc) return rc;
    std::vector<rtclj_stats> st((size_t)n_devices);
    rc = run_on_devices(n_devices, [&](int d) {
      const rtclj_params q = shard_params(prm, devices, d, n_devices);
      return render_shard_hostbuf(scene, cams, &q, out_linear, out_rgb8, &st[(size_t)d], n_frames);
    });
    if (rc) return rc;
    rtclj_stats total = sum_stats(st);
    total.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats) *stats = total;
    return RTCLJ_OK;
  });
}

int rtclj_render(const rtclj_scene* scene, const rtclj_camera* cam, const rtclj_params* prm, double* out_linear,
                 uint8_t* out_rgb8, rtclj_stats* stats) {
  return guarded([&]() -> int {
    if (!scene) return fail(RTCLJ_E_INVALID, "null scene");
    int rc = validate(cam, prm);
    if (rc) return rc;
    rc = render_shard_hostbuf(scene, cam, prm, out_linear, out_rgb8, stats);
    if (rc == RTCLJ_OK && stats) stats->n_devices = 1;
    return rc;
  });
}

// ---------------------------------------------------------------- accumulation over passes
// The compute-pixel loop (src/raytracing.clj:141-171) run in passes: a pass adds samples [d, d + n) of every
// pixel to the pixel's running sum, in the order a one-shot render adds them (DESIGN.md section 4.9).

}  // extern "C"

namespace {

// the pass unit of an accumulation: 1 in strict order, else the one-shot render's unit size
int accum_pass_unit(const rtclj_camera* cam, const rtclj_params* prm, bool* strict_out) {
  const bool strict = prm->samples_per_unit >= prm->spp || (prm->samples_per_unit <= 0 && primary_only(prm));
  if (strict_out) *strict_out = strict;
  return strict ? 1
                : (prm->samples_per_unit > 0 ? prm->samples_per_unit
                                             : auto_samples_per_unit(cam->width, cam->height, prm->spp));
}

// the arguments of an adaptive accumulation (checked before any device is touched): tolerance = {abs, rel}, both
// finite and >= 0; min_samples >= 2 pass units, so that the estimate has at least two units
int check_adaptive(const rtclj_camera* cam, const rtclj_params* prm, const double* tol, int32_t min_samples) {
  if (!tol) return fail(RTCLJ_E_INVALID, "null tolerance");
  if (!(std::isfinite(tol[0]) && std::isfinite(tol[1]) && tol[0] >= 0.0 && tol[1] >= 0.0))
    return fail(RTCLJ_E_INVALID, "tolerances must be finite and >= 0, got %g, %g", tol[0], tol[1]);
  int rc = validate(cam, prm);
  if (rc) return rc;
  const int unit = accum_pass_unit(cam, prm, nullptr);
  if ((long long)min_samples < 2ll * unit)
    return fail(RTCLJ_E_INVALID, "min_samples = %d: at least two pass units (%d)", min_samples, 2 * unit);
  return RTCLJ_OK;
}

// tol == nullptr: a plain accumulation
int accum_begin(rtclj_ctx* c, const rtclj_camera* cam, const rtclj_params* prm, const double* tol, int32_t min_samples,
                int32_t* pass_unit, cudaStream_t stream) {
  if (!c) return fail(RTCLJ_E_INVALID, "null ctx");
  if (!c->have_scene) return fail(RTCLJ_E_INVALID, "rtclj_ctx_set_scene has not been called");
  int rc = tol ? check_adaptive(cam, prm, tol, min_samples) : validate(cam, prm);
  if (rc) return rc;
  if (prm->flags & (RTCLJ_F_WAVE_KERNEL | RTCLJ_F_SPLIT_KERNEL))
    return fail(RTCLJ_E_INVALID, "the wavefront and split kernels do not accumulate over passes");
  // the kernels hold sample indices in 32-bit ints (render_lane2_kernel keeps k and k_end in shared memory
  // as 32-bit words) and compute k + samples_per_unit: keep that sum below 2^31
  if (prm->spp > (1 << 30)) return fail(RTCLJ_E_INVALID, "target of %d samples per pixel: at most 2^30", prm->spp);
  c->accum.active = false;
  CU(cudaSetDevice(c->device));
  bool strict = false;
  const int unit = accum_pass_unit(cam, prm, &strict);
  const Shard sh = shard_of(cam, prm);
  const size_t npix = (size_t)sh.local_pixels;
  CU(c->acc.reserve(std::max<size_t>(npix * 3, 1)));
  CU(cudaMemsetAsync(c->acc.p, 0, npix * 3 * sizeof(double), stream));
  if (tol) {
    // every pixel starts live, with no samples and S2 = 0; the list of all pixels is built by the compaction
    const size_t tiles = (npix + kListTile - 1) / kListTile;
    CU(c->acc2.reserve(std::max<size_t>(npix * 3, 1)));
    CU(c->nsamp.reserve(std::max<size_t>(npix, 1)));
    CU(c->live.reserve(std::max<size_t>(npix, 1)));
    CU(c->list.reserve(std::max<size_t>(npix, 1)));
    CU(c->list_aux.reserve(1 + tiles));
    CU(cudaMemsetAsync(c->acc2.p, 0, npix * 3 * sizeof(double), stream));
    CU(cudaMemsetAsync(c->nsamp.p, 0, npix * sizeof(int), stream));
    CU(cudaMemsetAsync(c->live.p, 1, npix, stream));
    CU(cudaMemsetAsync(c->list_aux.p, 0, sizeof(unsigned), stream));
    rc = relist(c, sh.local_pixels, stream);
    if (rc) return rc;
  }
  c->accum.strict = strict;
  c->accum.cam = *cam;
  c->accum.prm = *prm;
  c->accum.done = 0;
  c->accum.pass_unit = unit;
  c->accum.adaptive = tol != nullptr;
  c->accum.abs_tol = tol ? tol[0] : 0.0;
  c->accum.rel_tol = tol ? tol[1] : 0.0;
  c->accum.min_samples = tol ? min_samples : 0;
  c->accum.active = true;
  if (pass_unit) *pass_unit = unit;
  return RTCLJ_OK;
}

}  // namespace

extern "C" {

int rtclj_ctx_accum_begin(rtclj_ctx* c, const rtclj_camera* cam, const rtclj_params* prm, int32_t* pass_unit,
                          void* stream_) {
  return guarded([&]() -> int { return accum_begin(c, cam, prm, nullptr, 0, pass_unit, (cudaStream_t)stream_); });
}

int rtclj_ctx_accum_begin_adaptive(rtclj_ctx* c, const rtclj_camera* cam, const rtclj_params* prm,
                                   const double tolerance[2], int32_t min_samples, int32_t* pass_unit, void* stream_) {
  return guarded([&]() -> int {
    if (!c) return fail(RTCLJ_E_INVALID, "null ctx");
    if (!tolerance) return fail(RTCLJ_E_INVALID, "null tolerance");
    return accum_begin(c, cam, prm, tolerance, min_samples, pass_unit, (cudaStream_t)stream_);
  });
}

int rtclj_ctx_accum_step(rtclj_ctx* c, int32_t samples, void* d_out_linear, void* d_out_rgb8, int32_t* samples_done,
                         void* stream_) {
  return guarded([&]() -> int {
    if (!c) return fail(RTCLJ_E_INVALID, "null ctx");
    auto& A = c->accum;
    if (!A.active) return fail(RTCLJ_E_INVALID, "no accumulation: call rtclj_ctx_accum_begin (rtclj_ctx_set_scene ends one)");
    const rtclj_params* prm = &A.prm;
    const rtclj_camera* cam = &A.cam;
    int rc = check_pass(A.done, samples, prm->spp, A.pass_unit);
    if (rc) return rc;
    cudaStream_t stream = (cudaStream_t)stream_;
    CU(cudaSetDevice(c->device));
    const Shard sh = shard_of(cam, prm);
    const KernelChoice ch = choose_kernel(c, prm, (double)sh.local_pixels * (double)samples);
    const int d = A.done + samples;  // samples per pixel after this pass: the mean's divisor
    Pass ps;
    ps.sample_base = A.done; ps.samples = samples; ps.acc = c->acc.p; ps.mean_n = d; ps.finalize = true;
    ps.listed = A.adaptive;  // only the live pixels, each folded and tested (finalize_adaptive_kernel)
    ps.out_linear = (double*)d_out_linear; ps.out_rgb8 = (unsigned char*)d_out_rgb8;
    if (!A.strict || ch.kernel == Kernel::none) {
      // chunks of pass_unit samples, folded onto the running sums in chunk order (depth <= 0: one unit of black)
      ps.spu = ch.kernel != Kernel::none ? std::min(A.pass_unit, samples) : samples;
      rc = launch_pass(c, cam, prm, ch, sh, ps, stream);
    } else if (ch.kernel == Kernel::primary) {
      // one unit per pixel whose sums continue from the running sums: the reference's sequential sum in registers
      ps.spu = samples; ps.seeded = true;
      rc = launch_pass(c, cam, prm, ch, sh, ps, stream);
    } else {
      // every sample's colour through sample_buf, added in sample order by the fold: sub-passes of at most
      // kAccumSampleBufBytes, the fold is sequential per sample, so the cut changes no bit
      const size_t per_sample = (size_t)sh.local_pixels * 32u;
      const int per = per_sample ? (int)std::min<size_t>(kAccumSampleBufBytes / per_sample, (size_t)samples) : samples;
      if (per <= 0)
        return fail(RTCLJ_E_TOO_LARGE, "%llu pixels: one sample of each exceeds the %zu-byte strict buffer; use chunks "
                    "(samples_per_unit < spp)", sh.local_pixels, kAccumSampleBufBytes);
      CU(c->sample_buf.reserve(std::max<size_t>((size_t)per * per_sample / 8u, 1)));
      for (int b = 0; b < samples && rc == RTCLJ_OK; b += per) {
        Pass sub = ps;
        sub.sample_base = A.done + b;
        sub.samples = std::min(per, samples - b);
        sub.spu = auto_samples_per_unit(cam->width, cam->height, sub.samples);  // scheduling units only
        sub.sample_buf = c->sample_buf.p;
        sub.first = b == 0;
        sub.decide = b + per >= samples;
        if (b + per < samples) { sub.out_linear = nullptr; sub.out_rgb8 = nullptr; }  // fold only
        rc = launch_pass(c, cam, prm, ch, sh, sub, stream);
      }
    }
    if (rc) { A.active = false; return rc; }  // the running sums may hold part of the pass
    c->last_spu = A.strict ? d : A.pass_unit;
    A.done = d;
    if (samples_done) *samples_done = d;
    return RTCLJ_OK;
  });
}

int rtclj_ctx_accum_noise(rtclj_ctx* c, int32_t* d_samples, double* d_stderr, uint64_t* active_pixels, void* stream_) {
  return guarded([&]() -> int {
    if (!c) return fail(RTCLJ_E_INVALID, "null ctx");
    if (!c->accum.active || !c->accum.adaptive)
      return fail(RTCLJ_E_INVALID, "no adaptive accumulation: call rtclj_ctx_accum_begin_adaptive");
    cudaStream_t stream = (cudaStream_t)stream_;
    CU(cudaSetDevice(c->device));
    const Shard sh = shard_of(&c->accum.cam, &c->accum.prm);
    if ((d_samples || d_stderr) && sh.local_pixels > 0) {
      const unsigned blocks = (unsigned)((sh.local_pixels + 255) / 256);
      noise_export_kernel<<<blocks, 256, 0, stream>>>(adaptive_params(c, sh), d_samples, d_stderr);
      CU(cudaGetLastError());
    }
    if (active_pixels) {
      unsigned n = 0;
      CU(cudaMemcpyAsync(&n, c->list_aux.p, sizeof n, cudaMemcpyDeviceToHost, stream));
      CU(cudaStreamSynchronize(stream));
      *active_pixels = n;
    }
    return RTCLJ_OK;
  });
}

// A progressive render into host buffers, rows interleaved over several GPUs as in rtclj_render_multi.  Each
// device has a context of its own (not the cached one of rtclj_render, which other calls would give another
// scene and with it end the accumulation), accumulating its shard of the rows.
struct rtclj_progressive {
  std::vector<rtclj_ctx*> ctxs;
  std::vector<rtclj_params> prm;  // per device: its shard
  rtclj_camera cam;
  int spp = 0, pass_unit = 1, done = 0;
  bool adaptive = false;
  bool failed = false;  // a step failed on some device: the devices' running sums no longer agree
  ~rtclj_progressive() { for (rtclj_ctx* c : ctxs) rtclj_ctx_destroy(c); }
};

}  // extern "C"

namespace {

// tol == nullptr: a plain accumulation
int progressive_create(const rtclj_scene* scene, const rtclj_camera* cam, const rtclj_params* prm, const double* tol,
                       int32_t min_samples, const int32_t* devices, int32_t n_devices, int32_t* pass_unit,
                       rtclj_progressive** out) {
  return guarded([&]() -> int {
    if (!out) return fail(RTCLJ_E_INVALID, "null out");
    *out = nullptr;
    if (!scene) return fail(RTCLJ_E_INVALID, "null scene");
    int rc = validate(cam, prm);
    if (rc) return rc;
    if (tol) {
      rc = check_adaptive(cam, prm, tol, min_samples);
      if (rc) return rc;
    }
    rc = check_devices(devices, n_devices);
    if (rc) return rc;
    std::unique_ptr<rtclj_progressive> p(new rtclj_progressive());
    p->cam = *cam;
    p->spp = prm->spp;
    p->adaptive = tol != nullptr;
    for (int d = 0; d < n_devices; ++d) {
      const rtclj_params q = shard_params(prm, devices, d, n_devices);
      rtclj_ctx* c = nullptr;
      rc = rtclj_ctx_create(devices[d], &c);
      if (rc) return rc;
      p->ctxs.push_back(c);
      p->prm.push_back(q);
      rc = rtclj_ctx_set_scene(c, scene);
      if (rc) return rc;
      rc = accum_begin(c, cam, &q, tol, min_samples, &p->pass_unit, c->own_stream);
      if (rc) return rc;
    }
    if (pass_unit) *pass_unit = p->pass_unit;
    *out = p.release();
    return RTCLJ_OK;
  });
}

}  // namespace

extern "C" {

int rtclj_progressive_create(const rtclj_scene* scene, const rtclj_camera* cam, const rtclj_params* prm,
                             const int32_t* devices, int32_t n_devices, int32_t* pass_unit, rtclj_progressive** out) {
  return progressive_create(scene, cam, prm, nullptr, 0, devices, n_devices, pass_unit, out);
}

int rtclj_progressive_create_adaptive(const rtclj_scene* scene, const rtclj_camera* cam, const rtclj_params* prm,
                                      const double tolerance[2], int32_t min_samples, const int32_t* devices,
                                      int32_t n_devices, int32_t* pass_unit, rtclj_progressive** out) {
  if (out) *out = nullptr;
  if (!tolerance) return fail(RTCLJ_E_INVALID, "null tolerance");
  return progressive_create(scene, cam, prm, tolerance, min_samples, devices, n_devices, pass_unit, out);
}

int rtclj_progressive_step(rtclj_progressive* p, int32_t samples, double* out_linear, uint8_t* out_rgb8,
                           int32_t* samples_done, rtclj_stats* stats) {
  return guarded([&]() -> int {
    const auto t0 = std::chrono::steady_clock::now();
    if (!p) return fail(RTCLJ_E_INVALID, "null progressive handle");
    if (p->failed) return fail(RTCLJ_E_INVALID, "an earlier step failed: destroy this handle and create a new one");
    // rtclj_ctx_accum_step's checks, made before any device starts, so that the devices stay in step
    int rc = check_pass(p->done, samples, p->spp, p->pass_unit);
    if (rc) return rc;
    const size_t npix = (size_t)p->cam.width * (size_t)p->cam.height;
    std::vector<rtclj_stats> st(p->ctxs.size());
    rc = run_on_devices((int)p->ctxs.size(), [&](int d) -> int {  // pass -> this device's rows of the caller's images
      rtclj_ctx* c = p->ctxs[d];
      const rtclj_params& q = p->prm[d];
      CU(cudaSetDevice(c->device));
      if (out_linear) CU(c->out_linear.reserve(npix * 3));
      if (out_rgb8) CU(c->out_rgb8.reserve(npix * 3));
      int r = rtclj_ctx_accum_step(c, samples, out_linear ? c->out_linear.p : nullptr, out_rgb8 ? c->out_rgb8.p : nullptr,
                                   nullptr, c->own_stream);
      if (r) return r;
      r = download_rows(c, &p->cam, q.shard_index, q.shard_count, q.shard_rows, out_linear, out_rgb8, c->own_stream);
      if (r) return r;
      return rtclj_ctx_stats(c, c->own_stream, &st[(size_t)d]);  // synchronises the stream: the direct copies have landed
    });
    if (rc) { p->failed = true; return rc; }
    p->done += samples;
    if (samples_done) *samples_done = p->done;
    rtclj_stats total = sum_stats(st);
    total.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats) *stats = total;
    return RTCLJ_OK;
  });
}

int rtclj_progressive_noise(rtclj_progressive* p, int32_t* samples, double* stderr_, uint64_t* active_pixels) {
  return guarded([&]() -> int {
    if (!p) return fail(RTCLJ_E_INVALID, "null progressive handle");
    if (!p->adaptive) return fail(RTCLJ_E_INVALID, "not an adaptive progressive render");
    if (p->failed) return fail(RTCLJ_E_INVALID, "an earlier step failed: destroy this handle and create a new one");
    const size_t W = (size_t)p->cam.width, H = (size_t)p->cam.height;
    uint64_t total = 0;
    for (size_t d = 0; d < p->ctxs.size(); ++d) {  // (small images: one device after the other)
      rtclj_ctx* c = p->ctxs[d];
      const rtclj_params& q = p->prm[d];
      CU(cudaSetDevice(c->device));
      if (samples) CU(c->noise_samples.reserve(W * H));
      if (stderr_) CU(c->noise_stderr.reserve(W * H * 3));
      uint64_t n = 0;
      int rc = rtclj_ctx_accum_noise(c, samples ? c->noise_samples.p : nullptr, stderr_ ? c->noise_stderr.p : nullptr, &n,
                                     c->own_stream);
      if (rc) return rc;
      total += n;
      std::vector<Piece> pieces;
      if (samples) {
        plan_pieces(H, W * sizeof(int32_t), q.shard_index, q.shard_count, q.shard_rows, kStageBytes, pieces);
        rc = download_image(c, pieces, (char*)samples, (const char*)c->noise_samples.p, c->own_stream);
        if (rc) return rc;
      }
      if (stderr_) {
        pieces.clear();
        plan_pieces(H, W * 3 * sizeof(double), q.shard_index, q.shard_count, q.shard_rows, kStageBytes, pieces);
        rc = download_image(c, pieces, (char*)stderr_, (const char*)c->noise_stderr.p, c->own_stream);
        if (rc) return rc;
      }
      CU(cudaStreamSynchronize(c->own_stream));  // the direct copies into pinned memory have landed
    }
    if (active_pixels) *active_pixels = total;
    return RTCLJ_OK;
  });
}

int rtclj_progressive_destroy(rtclj_progressive* p) {
  return guarded([&]() -> int {
    delete p;  // (destroying the contexts waits for their streams)
    return RTCLJ_OK;
  });
}

}  // extern "C"

namespace {

// The render loop on several GPUs with the 8-bit image assembled on devices[0]: each device renders its shard and
// copies its rows into the root's out_rgb8 over NVLink.  Every device of the call is locked in `locks` until the
// caller lets go of them (the root's image is written by its peers); locks are taken in ordinal order, so two such
// calls cannot deadlock.  *root receives devices[0]'s context, *total the summed counters.
int render_to_root(const rtclj_scene* scene, const rtclj_camera* cam, const rtclj_params* prm, const int32_t* devices,
                   int32_t n_devices, std::vector<std::unique_lock<std::mutex>>& locks, rtclj_ctx** root_out,
                   rtclj_stats* total) {
  int rc = check_devices(devices, n_devices);
  if (rc) return rc;
  const size_t npix = (size_t)cam->width * (size_t)cam->height;
  std::vector<int> order(devices, devices + n_devices);
  std::sort(order.begin(), order.end());
  std::vector<rtclj_ctx*> ctxs((size_t)n_devices, nullptr);
  for (int dev : order) {
    rtclj_ctx* c = nullptr;
    locks.emplace_back();
    rc = cached_ctx(dev, locks.back(), &c);
    if (rc) return rc;
    for (int d = 0; d < n_devices; ++d) if (devices[d] == dev) ctxs[(size_t)d] = c;
  }
  rtclj_ctx* root = ctxs[0];
  CU(cudaSetDevice(root->device));
  CU(root->out_rgb8.reserve(npix * 3));
  std::vector<rtclj_stats> st((size_t)n_devices);
  rc = run_on_devices(n_devices, [&](int d) -> int {
    rtclj_ctx* c = ctxs[(size_t)d];
    const rtclj_params q = shard_params(prm, devices, d, n_devices);
    int r = rtclj_ctx_set_scene(c, scene);
    if (r) return r;
    if (c != root) CU(c->out_rgb8.reserve(npix * 3));
    r = rtclj_ctx_render(c, cam, &q, nullptr, c->out_rgb8.p, c->own_stream);
    if (r) return r;
    if (c != root) {  // this shard's rows -> the root's image, device to device
      int can = 0;
      if (cudaDeviceCanAccessPeer(&can, c->device, root->device) == cudaSuccess && can) {
        const cudaError_t e = cudaDeviceEnablePeerAccess(root->device, 0);
        if (e != cudaSuccess) cudaGetLastError();  // already enabled: fine; otherwise the copy is staged by the driver
      }
      std::vector<Piece> pieces;
      plan_pieces((size_t)cam->height, (size_t)cam->width * 3, q.shard_index, q.shard_count, q.shard_rows, (size_t)1 << 40, pieces);
      for (const Piece& pc : pieces) {
        if (pc.height == 1) CU(cudaMemcpyAsync(root->out_rgb8.p + pc.off, c->out_rgb8.p + pc.off, pc.width, cudaMemcpyDefault, c->own_stream));
        else CU(cudaMemcpy2DAsync(root->out_rgb8.p + pc.off, pc.pitch, c->out_rgb8.p + pc.off, pc.pitch, pc.width, pc.height, cudaMemcpyDefault, c->own_stream));
      }
    }
    return rtclj_ctx_stats(c, c->own_stream, &st[(size_t)d]);  // synchronises: render and copies are done
  });
  if (rc) return rc;
  *total = sum_stats(st);
  *root_out = root;
  CU(cudaSetDevice(root->device));
  return RTCLJ_OK;
}

// The filtered stream's length and the sizing call's answer (every segment stored) of a W x H PNG;
// RTCLJ_E_INVALID for sizes the encoder cannot take.
int png_sizes(int32_t width, int32_t height, size_t* nf, size_t* bound) {
  if (width <= 0 || height <= 0) return fail(RTCLJ_E_INVALID, "image size must be positive (%d x %d)", width, height);
  const size_t N = (size_t)height * ((size_t)width * 3 + 1);  // < 2^63 for any int32 size
  const size_t nseg = (N + kPngSeg - 1) / kPngSeg;
  if (nseg > 0x7ffffffeull) return fail(RTCLJ_E_INVALID, "a %d x %d PNG is too large for the device encoder", width, height);
  const size_t full = N / kPngSeg, rest = N - full * kPngSeg;
  *nf = N;
  *bound = kPngHead + kPngTail + full * (12 + kPngSeg + 10) + (rest ? 12 + rest + 5 * ((rest + 65534) / 65535) : 0);
  return RTCLJ_OK;
}

}  // namespace

extern "C" {

// Render on several GPUs and return the P3 TEXT -- the reference's loop plus its write-color! loop
// (src/raytracing.clj:141-175) as one call.  The 8-bit shards are assembled on devices[0] by peer copies
// over NVLink and the device P3 writer runs there; only the text crosses PCIe.  This is the one product for
// which a device-side gather beats the host gather (DESIGN.md section 6: 1.9 vs 13.4 ms at 3840x2160 on 8 GPUs).
int rtclj_render_multi_ppm(const rtclj_scene* scene, const rtclj_camera* cam, const rtclj_params* prm,
                           const int32_t* devices, int32_t n_devices, char* out, size_t capacity, size_t* len,
                           rtclj_stats* stats) {
  return guarded([&]() -> int {
    const auto t0 = std::chrono::steady_clock::now();
    if (!scene || !len) return fail(RTCLJ_E_INVALID, "null scene or len");
    int rc = validate(cam, prm);
    if (rc) return rc;
    const size_t npix = (size_t)cam->width * (size_t)cam->height;
    const size_t worst = 64 + npix * 12;  // "255 255 255\n" per pixel + header
    if (!out) { *len = worst; return RTCLJ_OK; }  // sizing call: an upper bound, nothing is rendered
    std::vector<std::unique_lock<std::mutex>> locks;
    rtclj_ctx* root = nullptr;
    rtclj_stats total;
    rc = render_to_root(scene, cam, prm, devices, n_devices, locks, &root, &total);
    if (rc) return rc;
    // the write-color! loop on the assembled image, then the text alone goes to the host
    CU(root->p3_text.reserve(worst));
    size_t need = 0;
    rc = rtclj_ctx_encode_ppm_p3(root, root->out_rgb8.p, cam->width, cam->height, reinterpret_cast<char*>(root->p3_text.p), worst, &need, root->own_stream);
    if (rc) return rc;
    *len = need;
    if (need > capacity) return fail(RTCLJ_E_BUFFER, "P3 text needs %zu bytes, capacity is %zu", need, capacity);
    CU(cudaMemcpyAsync(out, root->p3_text.p, need, cudaMemcpyDeviceToHost, root->own_stream));
    CU(cudaStreamSynchronize(root->own_stream));
    total.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats) *stats = total;
    return RTCLJ_OK;
  });
}

// The same render with the compressed PNG writer in place of the P3 writer: only the PNG crosses PCIe.
int rtclj_render_multi_png(const rtclj_scene* scene, const rtclj_camera* cam, const rtclj_params* prm,
                           const int32_t* devices, int32_t n_devices, uint8_t* out, size_t capacity, size_t* len,
                           rtclj_stats* stats) {
  return guarded([&]() -> int {
    const auto t0 = std::chrono::steady_clock::now();
    if (!scene || !len) return fail(RTCLJ_E_INVALID, "null scene or len");
    int rc = validate(cam, prm);
    if (rc) return rc;
    size_t nf = 0, bound = 0;
    rc = png_sizes(cam->width, cam->height, &nf, &bound);
    if (rc) return rc;
    if (!out) { *len = bound; return RTCLJ_OK; }  // sizing call: the stored bound, nothing is rendered
    std::vector<std::unique_lock<std::mutex>> locks;
    rtclj_ctx* root = nullptr;
    rtclj_stats total;
    rc = render_to_root(scene, cam, prm, devices, n_devices, locks, &root, &total);
    if (rc) return rc;
    CU(root->png_out.reserve(bound));
    size_t need = 0;
    rc = rtclj_ctx_encode_png(root, root->out_rgb8.p, cam->width, cam->height, root->png_out.p, bound, &need, root->own_stream);
    if (rc) return rc;
    *len = need;
    if (need > capacity) return fail(RTCLJ_E_BUFFER, "PNG needs %zu bytes, capacity is %zu", need, capacity);
    CU(cudaMemcpyAsync(out, root->png_out.p, need, cudaMemcpyDeviceToHost, root->own_stream));
    CU(cudaStreamSynchronize(root->own_stream));
    total.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats) *stats = total;
    return RTCLJ_OK;
  });
}

// The copies a shard's download consists of (host logic shared by rtclj_render / rtclj_render_multi),
// exposed so that the N > 1 arithmetic is testable without a GPU.
int rtclj_shard_plan(int32_t height, size_t row_bytes, int32_t shard_index, int32_t shard_count, int32_t shard_rows,
                     size_t max_piece_bytes, uint64_t* pieces, size_t capacity, size_t* n_pieces) {
  return guarded([&]() -> int {
    if (!n_pieces) return fail(RTCLJ_E_INVALID, "null n_pieces");
    if (height <= 0 || row_bytes == 0) return fail(RTCLJ_E_INVALID, "image size must be positive");
    if (shard_count > 1 && (shard_index < 0 || shard_index >= shard_count || shard_rows <= 0))
      return fail(RTCLJ_E_INVALID, "bad shard (%d of %d, %d rows)", shard_index, shard_count, shard_rows);
    std::vector<Piece> v;
    plan_pieces((size_t)height, row_bytes, shard_index, shard_count, shard_rows, max_piece_bytes ? max_piece_bytes : kStageBytes, v);
    *n_pieces = v.size();
    if (!pieces) return RTCLJ_OK;
    if (capacity < v.size()) return fail(RTCLJ_E_BUFFER, "%zu pieces, capacity %zu", v.size(), capacity);
    for (size_t i = 0; i < v.size(); ++i) {
      pieces[4 * i] = v[i].off; pieces[4 * i + 1] = v[i].pitch; pieces[4 * i + 2] = v[i].width; pieces[4 * i + 3] = v[i].height;
    }
    return RTCLJ_OK;
  });
}

// ---- pinned host memory for callers: images allocated (or registered) here are written by the GPUs
// directly, with no staging copy (Panama: MemorySegment.reinterpret over the returned address)
int rtclj_host_alloc(size_t bytes, void** out) {
  if (!out) return fail(RTCLJ_E_INVALID, "null out");
  *out = nullptr;
  int ndev = 0;
  int rc = rtclj_device_count(&ndev);
  if (rc) return rc;
  if (ndev == 0) return fail(RTCLJ_E_NO_DEVICE, "no CUDA device (this library has no CPU fallback)");
  CU(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable));
  return RTCLJ_OK;
}
int rtclj_host_free(void* p) {
  if (p) CU(cudaFreeHost(p));
  return RTCLJ_OK;
}
int rtclj_host_register(void* p, size_t bytes) {
  if (!p || !bytes) return fail(RTCLJ_E_INVALID, "null buffer");
  CU(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
  return RTCLJ_OK;
}
int rtclj_host_unregister(void* p) {
  if (p) CU(cudaHostUnregister(p));
  return RTCLJ_OK;
}

// ---- row f-1: the P3 writer (src/raytracing.clj:172-175) on the device
int rtclj_ctx_encode_ppm_p3(rtclj_ctx* c, const uint8_t* d_rgb8, int32_t width, int32_t height, char* d_out,
                            size_t capacity, size_t* len, void* stream_) {
  if (!c) return fail(RTCLJ_E_INVALID, "null ctx");
  if (width <= 0 || height <= 0 || !len || !d_rgb8) return fail(RTCLJ_E_INVALID, "bad image or null len");
  cudaStream_t stream = (cudaStream_t)stream_;
  CU(cudaSetDevice(c->device));
  const size_t npix = (size_t)width * (size_t)height;
  const size_t nb = (npix + kP3PixPerBlock - 1) / kP3PixPerBlock;
  if (nb > 0x7fffffffull) return fail(RTCLJ_E_TOO_LARGE, "image of %zu pixels is too large for the P3 writer", npix);
  P3Header hdr;
  hdr.n = std::snprintf(hdr.s, sizeof hdr.s, "P3\n%d %d\n255\n", width, height);
  const int aligned4 = (reinterpret_cast<uintptr_t>(d_rgb8) & 3u) == 0;
  // persistent grid: every CTA owns one contiguous run of tiles
  if (c->p3_ctas_per_sm == 0) {
    int occ = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, p3_encode_kernel, kP3Threads, 0));
    c->p3_ctas_per_sm = occ > 0 ? occ : 1;
  }
  const size_t want = (size_t)c->sm_count * (size_t)c->p3_ctas_per_sm;
  const size_t per_cta = (nb + want - 1) / want;
  const size_t grid = (nb + per_cta - 1) / per_cta;
  CU(c->p3_state.reserve(grid + 2));
  unsigned long long total = 0;
  const bool one_pass = d_out && capacity >= (size_t)hdr.n + npix * 12;  // the buffer holds the worst case
  c->p3_count_ms = c->p3_write_ms = 0.f;
  if (!one_pass) {  // the exact length first: sizing calls and tighter buffers
    CU(cudaMemsetAsync(c->p3_state.p, 0, (grid + 2) * sizeof(unsigned long long), stream));
    CU(cudaEventRecord(c->p3_ev0, stream));
    p3_encode_kernel<<<(unsigned)grid, kP3Threads, 0, stream>>>(d_rgb8, npix, aligned4, nb, per_cta, c->p3_state.p, nullptr, hdr, 1);
    CU(cudaGetLastError());
    CU(cudaEventRecord(c->p3_ev1, stream));
    CU(cudaMemcpyAsync(&total, c->p3_state.p + 1, sizeof total, cudaMemcpyDeviceToHost, stream));
    CU(cudaStreamSynchronize(stream));
    CU(cudaEventElapsedTime(&c->p3_count_ms, c->p3_ev0, c->p3_ev1));
    *len = (size_t)total;
    if (!d_out) return RTCLJ_OK;
    if ((size_t)total > capacity) return fail(RTCLJ_E_BUFFER, "P3 text needs %llu bytes, capacity is %zu", total, capacity);
  }
  CU(cudaMemsetAsync(c->p3_state.p, 0, (grid + 2) * sizeof(unsigned long long), stream));
  CU(cudaEventRecord(c->p3_ev0, stream));
  p3_encode_kernel<<<(unsigned)grid, kP3Threads, 0, stream>>>(d_rgb8, npix, aligned4, nb, per_cta, c->p3_state.p,
                                                            reinterpret_cast<unsigned char*>(d_out), hdr, 0);
  CU(cudaGetLastError());
  CU(cudaEventRecord(c->p3_ev1, stream));
  CU(cudaMemcpyAsync(&total, c->p3_state.p + 1, sizeof total, cudaMemcpyDeviceToHost, stream));
  CU(cudaStreamSynchronize(stream));
  CU(cudaEventElapsedTime(&c->p3_write_ms, c->p3_ev0, c->p3_ev1));
  *len = (size_t)total;
  return RTCLJ_OK;
}

int rtclj_ctx_encode_ms(rtclj_ctx* c, double* count_scan_ms, double* write_ms) {
  if (!c) return fail(RTCLJ_E_INVALID, "null ctx");
  if (count_scan_ms) *count_scan_ms = (double)c->p3_count_ms;
  if (write_ms) *write_ms = (double)c->p3_write_ms;
  return RTCLJ_OK;
}

int rtclj_encode_ppm_p3_gpu(int32_t device, const uint8_t* rgb8, int32_t width, int32_t height, char* out,
                            size_t capacity, size_t* len) {
  if (width <= 0 || height <= 0 || !len || !rgb8) return fail(RTCLJ_E_INVALID, "bad image or null len");
  std::unique_lock<std::mutex> lock;
  rtclj_ctx* c = nullptr;
  int rc = cached_ctx(device, lock, &c);
  if (rc) return rc;
  CU(cudaSetDevice(c->device));
  const size_t npix = (size_t)width * (size_t)height;
  CU(c->p3_in.reserve(npix * 3));
  CU(cudaMemcpyAsync(c->p3_in.p, rgb8, npix * 3, cudaMemcpyHostToDevice, c->own_stream));
  size_t need = 0;
  if (!out) return rtclj_ctx_encode_ppm_p3(c, c->p3_in.p, width, height, nullptr, 0, len, c->own_stream);
  const size_t worst = 64 + npix * 12;  // "255 255 255\n" per pixel
  CU(c->p3_text.reserve(worst));
  rc = rtclj_ctx_encode_ppm_p3(c, c->p3_in.p, width, height, reinterpret_cast<char*>(c->p3_text.p),
                               std::min(worst, capacity), &need, c->own_stream);
  *len = need;
  if (rc) return rc;
  CU(cudaMemcpyAsync(out, c->p3_text.p, need, cudaMemcpyDeviceToHost, c->own_stream));
  CU(cudaStreamSynchronize(c->own_stream));
  return RTCLJ_OK;
}

// ---- the compressed PNG writer on the device (DESIGN.md section 4.11; the format: include/rtclj_b200.h)
int rtclj_ctx_encode_png(rtclj_ctx* c, const uint8_t* d_rgb8, int32_t width, int32_t height, uint8_t* d_out,
                         size_t capacity, size_t* len, void* stream_) {
  return guarded([&]() -> int {
    if (!c || !len) return fail(RTCLJ_E_INVALID, "null ctx or len");
    size_t N = 0, bound = 0;
    int rc = png_sizes(width, height, &N, &bound);
    if (rc) return rc;
    if (!d_out) { *len = bound; return RTCLJ_OK; }
    if (!d_rgb8) return fail(RTCLJ_E_INVALID, "null image");
    cudaStream_t stream = (cudaStream_t)stream_;
    CU(cudaSetDevice(c->device));
    if (!c->png_attr) {
      CU(cudaFuncSetAttribute(png_deflate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PngDeflateSmem)));
      CU(cudaFuncSetAttribute(png_place_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(PngPlaceSmem)));
      c->png_attr = true;
    }
    static const PngCrcShifts shifts = png_crc_shifts();
    const size_t nseg = (N + kPngSeg - 1) / kPngSeg;
    CU(c->png_f.reserve(nseg * kPngSeg));
    CU(c->png_stage.reserve(nseg * kPngSlot));
    CU(c->png_rec.reserve(nseg));
    CU(c->png_state.reserve(1));
    png_filter_kernel<<<(unsigned)height, kPngFilterThreads, 0, stream>>>(d_rgb8, (size_t)width * 3, c->png_f.p);
    CU(cudaGetLastError());
    png_deflate_kernel<<<(unsigned)nseg, kPngThreads, sizeof(PngDeflateSmem), stream>>>(c->png_f.p, N, c->png_stage.p, c->png_rec.p);
    CU(cudaGetLastError());
    unsigned long long total = 0;
    if (capacity < bound) {  // the exact length first: the buffer may be too small for it
      png_place_kernel<<<(unsigned)nseg + 1, kPngThreads, sizeof(PngPlaceSmem), stream>>>(
          c->png_f.p, N, c->png_stage.p, c->png_rec.p, (unsigned)nseg, (unsigned)width, (unsigned)height, nullptr, c->png_state.p, 1, shifts);
      CU(cudaGetLastError());
      CU(cudaMemcpyAsync(&total, c->png_state.p, sizeof total, cudaMemcpyDeviceToHost, stream));
      CU(cudaStreamSynchronize(stream));
      *len = (size_t)total;
      if ((size_t)total > capacity) return fail(RTCLJ_E_BUFFER, "PNG needs %llu bytes, capacity is %zu", total, capacity);
    }
    png_place_kernel<<<(unsigned)nseg + 1, kPngThreads, sizeof(PngPlaceSmem), stream>>>(
        c->png_f.p, N, c->png_stage.p, c->png_rec.p, (unsigned)nseg, (unsigned)width, (unsigned)height, d_out, c->png_state.p, 0, shifts);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(&total, c->png_state.p, sizeof total, cudaMemcpyDeviceToHost, stream));
    CU(cudaStreamSynchronize(stream));
    *len = (size_t)total;
    return RTCLJ_OK;
  });
}

int rtclj_encode_png_gpu(int32_t device, const uint8_t* rgb8, int32_t width, int32_t height, uint8_t* out,
                         size_t capacity, size_t* len) {
  return guarded([&]() -> int {
    if (!len) return fail(RTCLJ_E_INVALID, "null len");
    size_t N = 0, bound = 0;
    int rc = png_sizes(width, height, &N, &bound);
    if (rc) return rc;
    if (!out) { *len = bound; return RTCLJ_OK; }
    if (!rgb8) return fail(RTCLJ_E_INVALID, "null image");
    std::unique_lock<std::mutex> lock;
    rtclj_ctx* c = nullptr;
    rc = cached_ctx(device, lock, &c);
    if (rc) return rc;
    CU(cudaSetDevice(c->device));
    const size_t bytes = (size_t)width * (size_t)height * 3;
    CU(c->png_in.reserve(bytes));
    CU(c->png_out.reserve(bound));
    CU(cudaMemcpyAsync(c->png_in.p, rgb8, bytes, cudaMemcpyHostToDevice, c->own_stream));
    size_t need = 0;
    rc = rtclj_ctx_encode_png(c, c->png_in.p, width, height, c->png_out.p, bound, &need, c->own_stream);
    if (rc) return rc;
    *len = need;
    if (need > capacity) return fail(RTCLJ_E_BUFFER, "PNG needs %zu bytes, capacity is %zu", need, capacity);
    CU(cudaMemcpyAsync(out, c->png_out.p, need, cudaMemcpyDeviceToHost, c->own_stream));
    CU(cudaStreamSynchronize(c->own_stream));
    return RTCLJ_OK;
  });
}

int rtclj_calibrate_peaks(int32_t device, double* ffma, double* ffma2, double* dfma, int32_t* sm_count) {
  int ndev = 0;
  int rc = rtclj_device_count(&ndev);
  if (rc) return rc;
  if (device < 0 || device >= ndev) return fail(RTCLJ_E_INVALID, "device %d out of range", device);
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  const int sms = prop.multiProcessorCount;
  if (sm_count) *sm_count = sms;
  const int blocks = sms * 4, threads = 512, iters = 1 << 14;
  struct Scratch {  // released on every path out of this function
    float* out = nullptr; cudaEvent_t e0 = nullptr, e1 = nullptr;
    ~Scratch() { if (e0) cudaEventDestroy(e0); if (e1) cudaEventDestroy(e1); if (out) cudaFree(out); }
  } sc;
  CU(cudaMalloc(&sc.out, sizeof(float) * (size_t)blocks * threads));
  CU(cudaEventCreate(&sc.e0));
  CU(cudaEventCreate(&sc.e1));
  float* out = sc.out;
  cudaEvent_t e0 = sc.e0, e1 = sc.e1;
  double res[3] = {0, 0, 0};
  for (int mode = 0; mode < 3; ++mode) {
    double best = 0;
    for (int rep = 0; rep < 4; ++rep) {
      CU(cudaEventRecord(e0));
      if (mode == 0) peak_kernel<0><<<blocks, threads>>>(out, iters, 1.0f);
      else if (mode == 1) peak_kernel<1><<<blocks, threads>>>(out, iters, 1.0f);
      else peak_kernel<2><<<blocks, threads>>>(out, iters / 2, 1.0f);
      CU(cudaEventRecord(e1));
      CU(cudaEventSynchronize(e1));
      float ms = 0;
      CU(cudaEventElapsedTime(&ms, e0, e1));
      const double fmas = (double)blocks * threads * 8.0 * (mode == 2 ? iters / 2 : iters) * (mode == 1 ? 2.0 : 1.0);
      const double tf = 2.0 * fmas / (ms * 1e-3) / 1e12;
      if (rep > 0 && tf > best) best = tf;
    }
    res[mode] = best;
  }
  if (ffma) *ffma = res[0];
  if (ffma2) *ffma2 = res[1];
  if (dfma) *dfma = res[2];
  return RTCLJ_OK;
}

}  // extern "C"
