/*
 * rtclj_b200.h -- C ABI of librtclj_b200.so, the B200 (sm_100a) backend for the
 * per-pixel render loop of keychera/raytracing-clj.
 *
 * The reference has NO plugin / FFI interface (SURVEY.md 8b): its hot path is an
 * anonymous closure and a loop inside `-main`.  Each entry point below therefore
 * names the reference code it stands in for:
 *
 *   rtclj_render            src/raytracing.clj:141-171  (compute-pixel + the 2-thread
 *                           row-chunk pool, up to `colors`), and
 *                           src/realm/raytracing.clj:325-346 (the j/i/spp loop filling
 *                           realm[0 .. 3*W*H)), and
 *                           src/experimental/raytracing_i.clj:146-163
 *   rtclj_render_multi      the same loop, image rows interleaved over several GPUs
 *   rtclj_render_multi_ppm  the same loop followed by the write-color! loop (raytracing.clj:172-175):
 *                           several GPUs in, the text of scene.ppm out
 *   rtclj_ctx_*             the same loop with device-resident buffers (scene upload
 *                           once, many renders; what bench.py times as `value`)
 *   rtclj_ctx_render_frames, rtclj_render_frames
 *                           the same loop for a sequence of cameras (one scene), every frame in shared launches
 *   rtclj_ctx_accum_*, rtclj_progressive_*
 *                           the same loop run in passes of samples (progressive rendering),
 *                           bit-identical to a one-shot render after every pass
 *   rtclj_quantise_rgb8     write-color! / linear->gamma / clamp,
 *                           src/raytracing.clj:19-26 ; realm/raytracing.clj:246-249,356-357
 *   rtclj_encode_ppm_p3     the P3 writer, src/raytracing.clj:172-175 ;
 *                           realm/raytracing.clj:350-358 (host)
 *   rtclj_ctx_encode_ppm_p3, rtclj_encode_ppm_p3_gpu
 *                           the same writer as device kernels (device / host buffers)
 *   rtclj_encode_png, rtclj_decode_ppm_p3
 *                           ppm->png, src/raytracing.clj:176 (src/ppm2png.clj:35-87): writer, reader
 *   rtclj_ctx_encode_png, rtclj_encode_png_gpu
 *                           a compressed PNG of the same image, written by device kernels (device / host buffers)
 *   rtclj_render_multi_png  the render loop and ppm->png as one call: several GPUs in, a compressed PNG out
 *   rtclj_camera_main/_realm/_i
 *                           the camera let-blocks, src/raytracing.clj:105-139 ;
 *                           realm/raytracing.clj:264-280,306-322 ;
 *                           experimental/raytracing_i.clj:82-90,127-144
 *   rtclj_scene_random_field  the RTIOW random-sphere field (not in the reference;
 *                           BASELINE.json configs 3 and 5, SURVEY.md Appendix D)
 *
 * Conventions: plain C, POD structs with fixed-width fields (Panama MemoryLayout /
 * JNA Structure friendly); the caller owns every buffer; the library copies what it
 * needs and keeps no caller pointer after a call returns; no callbacks; every
 * function returns 0 on success or an RTCLJ_E_* code and sets a thread-local message
 * readable with rtclj_last_error(); nothing throws across the boundary.  Every entry
 * point selects its CUDA device itself, so JVM pool threads may call it directly.
 * There is NO CPU fallback: without a CUDA device the render calls fail with
 * RTCLJ_E_NO_DEVICE.
 */
#ifndef RTCLJ_B200_H
#define RTCLJ_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTCLJ_ABI_VERSION 1

/* material ids: material/lambertian, material/metal, material/dielectric
 * (src/material.clj:13,21,34; realm/raytracing.clj:138,147,160) */
enum { RTCLJ_LAMBERTIAN = 0, RTCLJ_METAL = 1, RTCLJ_DIELECTRIC = 2 };

/* error codes */
enum {
  RTCLJ_OK = 0,
  RTCLJ_E_INVALID = 1,   /* bad argument (null pointer, non-positive size, ...) */
  RTCLJ_E_NO_DEVICE = 2, /* no usable CUDA device: there is no CPU fallback      */
  RTCLJ_E_CUDA = 3,      /* a CUDA call failed; see rtclj_last_error()           */
  RTCLJ_E_TOO_LARGE = 4, /* more than 65 532 spheres                              */
  RTCLJ_E_BUFFER = 5     /* output buffer too small                              */
};

/* variant switches -- the differences between the reference's programs
 * (SURVEY.md Appendix A.2) */
enum {
  RTCLJ_F_NEAR_ZERO_GUARD = 1u, /* lambertian falls back to the normal, material.clj:17     */
  RTCLJ_F_SCHLICK = 2u,         /* Schlick reflectance + its uniform, material.clj:30-32,42 */
  RTCLJ_F_REVERSE_PRODUCT = 4u, /* attenuation product innermost-first, raytracing.clj:52-53;
                                   off = forward product, realm/raytracing.clj:206,225,236  */
  RTCLJ_F_MEAN_DIVIDE = 8u,     /* pixel = sum / spp, raytracing.clj:155;
                                   off = sum * (1/spp), realm/raytracing.clj:25,344         */
  RTCLJ_F_NORMAL_SHADING = 16u, /* hit -> 0.5*(N+1), no bounces, raytracing_i.clj:59-73     */
  RTCLJ_F_QUANT_LINEAR = 32u,   /* 8-bit = int(255.999*c), no gamma, raytracing_i.clj:170   */
  RTCLJ_F_NO_CULL = 1u << 16,   /* skip the fp32 cull, test every sphere in fp64 (same image; the library
                                   chooses this by itself for scenes of <= 2 spheres, <= 6 when only primary
                                   rays are traced, where it is faster) */
  RTCLJ_F_SMEM_TABLE = 1u << 17, /* testing: use the shared-memory-table kernel even for a small scene */
  /* Scenes of <= 512 spheres have four kernels that produce the same image; these select one
   * explicitly (A/B timing, tests).  Without them the library uses the fastest one measured for the
   * regime (DESIGN.md sections 4 and 7): two paths per lane for >= 64 spheres and >= 4e7 samples per
   * shard, one path per lane otherwise (its own instantiation below 64 spheres), and for primary-ray
   * renders (RTCLJ_F_NORMAL_SHADING or max_depth 1) of <= 6 spheres a kernel without the path
   * machinery.  RTCLJ_F_LANE_KERNEL also keeps such a render on the general kernel. */
  RTCLJ_F_LANE_KERNEL = 1u << 18,  /* one path per lane (round 1)                                   */
  RTCLJ_F_WAVE_KERNEL = 1u << 19,  /* wavefront kernel: path state in shared memory, per-phase queues */
  RTCLJ_F_LANE2_KERNEL = 1u << 20, /* two paths per lane, culled together                            */
  RTCLJ_F_SPLIT_KERNEL = 1u << 21  /* dedicated cull warps (four rays per lane) + path warps          */
};
#define RTCLJ_FLAGS_MAIN                                                               \
  (RTCLJ_F_NEAR_ZERO_GUARD | RTCLJ_F_SCHLICK | RTCLJ_F_REVERSE_PRODUCT | RTCLJ_F_MEAN_DIVIDE)
#define RTCLJ_FLAGS_REALM 0u
#define RTCLJ_FLAGS_I (RTCLJ_F_NORMAL_SHADING | RTCLJ_F_QUANT_LINEAR)

/* The hittable list as a structure of arrays, in LIST ORDER (the first body wins an
 * exact tie, raytracing.clj:33-43).  Replaces `to-render` (raytracing.clj:102) and the
 * Entity[] (realm/raytracing.clj:285-301).
 * Accepted values: everything the reference's constructors accept (negative or zero radius,
 * fuzz > 1, any ior, albedo outside [0,1]) as long as it is finite and |coordinate|, |radius| < 1e18;
 * NaN / infinity / larger magnitudes return RTCLJ_E_INVALID (the reference's scan degenerates on a NaN
 * root, and the fp32 cull squares coordinates).  Spheres beyond 1e15 are simply never culled. */
typedef struct rtclj_scene {
  int32_t n;
  int32_t _pad;
  const double *center_xyz; /* [3n] hittable/sphere center                       */
  const double *radius;     /* [n]  hittable/sphere radius                       */
  const int32_t *material;  /* [n]  RTCLJ_LAMBERTIAN | RTCLJ_METAL | RTCLJ_DIELECTRIC */
  const double *albedo_rgb; /* [3n] lambertian / metal albedo (ignored otherwise) */
  const double *fuzz;       /* [n]  metal fuzz                                    */
  const double *ior;        /* [n]  dielectric refraction index                   */
} rtclj_scene;

/* The vectors the reference derives before its loop (raytracing.clj:126-139;
 * realm/raytracing.clj:306-322).  Row 0 is the top of the image.
 * Every value must be finite; only `center` and the defocus vectors are range-limited
 * (|center| + |defocus_u| + |defocus_v| < 1e18 per axis).  The directions pixel00 + du*x + dv*y - origin
 * are not: d = 0 or |d|^2 beyond the fp64 range give NaN roots, which are handled as the reference
 * handles them (DESIGN.md 4.1). */
typedef struct rtclj_camera {
  double pixel00[3];    /* pixel-00-loc   */
  double pixel_du[3];   /* pixel-du       */
  double pixel_dv[3];   /* pixel-dv       */
  double center[3];     /* camera-center  */
  double defocus_u[3];  /* defocus-disk-u */
  double defocus_v[3];  /* defocus-disk-v */
  double defocus_angle; /* <= 0: rays start at `center` (raytracing.clj:147)     */
  int32_t width;        /* image-width    */
  int32_t height;       /* image-height   */
} rtclj_camera;

typedef struct rtclj_params {
  int32_t spp;       /* samples-per-px */
  int32_t max_depth; /* max-depth      */
  uint64_t seed;     /* Philox key; the stream is keyed by (pixel, sample, bounce) */
  uint32_t flags;    /* RTCLJ_F_*      */
  /* Samples summed sequentially per work unit.  >= spp: one sequential sum per pixel, exactly the
   * reference's order (raytracing.clj:142-155, raytracing_i.clj:146-163).  Smaller units split a
   * pixel into chunks whose sums are added in index order: only the association of <= spp
   * additions changes (<= 1e-13 relative), and load balance improves.  <= 0: the library chooses,
   * from the image size alone (reported in rtclj_stats.samples_per_unit): the strict sequential sum
   * when max_depth == 1 or RTCLJ_F_NORMAL_SHADING is set (primary-ray renders, whose contract is
   * bit-exactness), chunks otherwise. */
  int32_t samples_per_unit;
  /* Row sharding for one-process-per-GPU hosts: rows are cut into tiles of
   * `shard_rows` rows and tile t belongs to shard t % shard_count.  A sharded render
   * writes ONLY its own rows of the (full-size) output buffers.  shard_count <= 1:
   * the whole image. */
  int32_t shard_index;
  int32_t shard_count;
  int32_t shard_rows;
  int32_t device; /* CUDA device ordinal for rtclj_render */
  int32_t _pad;
} rtclj_params;

typedef struct rtclj_stats {
  uint64_t samples;         /* camera rays started                                  */
  uint64_t segments;        /* ray segments = closest-hit searches (the "rays" of
                               BASELINE.json's metric), counted on the device      */
  uint64_t exact_tests;     /* fp64 ray-sphere tests run on cull survivors          */
  uint64_t list_overflows;  /* segments whose survivor list overflowed (full fp64 scan) */
  uint64_t prefilter_tests; /* cull survivors examined by the fp32 root prefilter          */
  double device_ms;         /* CUDA-event time of render + finalize kernels         */
  double kernel_ms;         /* CUDA-event time of the render kernel alone           */
  double total_ms;          /* wall time of the call, including copies              */
  int32_t samples_per_unit; /* the unit size actually used                          */
  int32_t n_devices;
} rtclj_stats;

typedef struct rtclj_ctx rtclj_ctx; /* one per (host thread, device) */

int rtclj_abi_version(void);
const char *rtclj_last_error(void);
int rtclj_device_count(int *count);

/* Host buffers in, host buffers out.  out_linear: W*H*3 doubles (row-major, x fastest,
 * RGB interleaved -- the order write-color! consumes, raytracing.clj:170-175), or NULL.
 * out_rgb8: W*H*3 bytes quantised like write-color!, or NULL.  stats may be NULL. */
int rtclj_render(const rtclj_scene *scene, const rtclj_camera *camera,
                 const rtclj_params *params, double *out_linear, uint8_t *out_rgb8,
                 rtclj_stats *stats);

/* The same image, rows interleaved over `n_devices` GPUs driven by this ONE process -- the call a JVM
 * host makes where the reference starts its pool (src/raytracing.clj:157-171).  One worker thread per
 * device uploads, renders and downloads its shard, so the devices overlap; rows are cut into tiles of
 * params->shard_rows rows (<= 0: 1) and tile t goes to devices[t % n_devices].  params->shard_index,
 * shard_count and device are ignored.  The image is identical for any device list. */
int rtclj_render_multi(const rtclj_scene *scene, const rtclj_camera *camera,
                       const rtclj_params *params, const int32_t *devices, int32_t n_devices,
                       double *out_linear, uint8_t *out_rgb8, rtclj_stats *stats);

/* The render loop AND the write-color! loop (src/raytracing.clj:141-175) as one call: renders on
 * `n_devices` GPUs (n_devices = 1 is fine), assembles the 8-bit shards on devices[0] by device-to-device
 * copies, runs the device P3 writer there and returns the text of the PPM file -- the bytes
 * rtclj_encode_ppm_p3 would produce from rtclj_render's rgb8 image; only the text crosses PCIe.
 * out == NULL: *len receives a sufficient capacity (an upper bound; nothing is rendered). */
int rtclj_render_multi_ppm(const rtclj_scene *scene, const rtclj_camera *camera,
                           const rtclj_params *params, const int32_t *devices, int32_t n_devices,
                           char *out, size_t capacity, size_t *len, rtclj_stats *stats);

/* The copies a sharded download consists of -- the host-side arithmetic behind rtclj_render (shard_*)
 * and rtclj_render_multi, callable without a GPU.  Piece i = pieces[4i .. 4i+3] = {byte offset (the same
 * in the device image and in the caller's image), pitch, width, height}: `height` runs of `width` bytes,
 * `pitch` bytes apart.  max_piece_bytes = 0: the library's staging size.  pieces == NULL: count only. */
int rtclj_shard_plan(int32_t height, size_t row_bytes, int32_t shard_index, int32_t shard_count,
                     int32_t shard_rows, size_t max_piece_bytes, uint64_t *pieces, size_t capacity,
                     size_t *n_pieces);

/* Pinned host memory.  Output images that live in memory CUDA knows as pinned are written by the GPUs
 * directly and asynchronously; pageable images (malloc, numpy, a JVM Arena) are filled through pinned
 * staging buffers inside the library (one extra host copy).  rtclj_host_alloc returns pinned memory
 * (Panama: MemorySegment.ofAddress(p).reinterpret(bytes)); rtclj_host_register pins memory the caller
 * already owns (page-aligned ranges register fastest) until rtclj_host_unregister. */
int rtclj_host_alloc(size_t bytes, void **out);
int rtclj_host_free(void *p);
int rtclj_host_register(void *p, size_t bytes);
int rtclj_host_unregister(void *p);

/* Device-resident path. */
int rtclj_ctx_create(int32_t device, rtclj_ctx **out);
void rtclj_ctx_destroy(rtclj_ctx *ctx);
int rtclj_ctx_set_scene(rtclj_ctx *ctx, const rtclj_scene *scene);
/* Enqueues the render on `stream` (a cudaStream_t, NULL = the default stream) and
 * returns without synchronising.  d_out_linear / d_out_rgb8 are DEVICE pointers to
 * full-size images (either may be NULL).  One context serves one stream at a time: its
 * work buffers belong to the render in flight (rtclj_ctx_set_scene waits for it).  Different
 * contexts -- also on one device, with different scenes -- may render concurrently: a launch
 * carries its cull table with it (kernel parameters), the library holds no per-device state. */
int rtclj_ctx_render(rtclj_ctx *ctx, const rtclj_camera *camera, const rtclj_params *params,
                     void *d_out_linear, void *d_out_rgb8, void *stream);
/* Synchronises `stream` and reads the counters of the last rtclj_ctx_render (or accumulation pass, or sequence). */
int rtclj_ctx_stats(rtclj_ctx *ctx, void *stream, rtclj_stats *stats);

/* ---- Camera sequences: n_frames frames of one scene (a turntable, a fly-through, a focus pull) in shared launches --
 * one ticket queue and one kernel tail per launch instead of one per frame (DESIGN.md section 4.12).
 *   - A sequence is one scene, one rtclj_params and n_frames >= 1 cameras of equal width x height; defocus angles may
 *     differ between frames, with and without the disk in one sequence.
 *   - Frame f's images (linear and 8-bit) are bit-identical to rtclj_ctx_render with cameras[f] and the same params,
 *     for every kernel choice, device list, shard_* setting and frame count.  The seed is shared by all frames (per-frame
 *     seeds: one call per frame).
 *   - The output buffers hold n_frames consecutive full-size images, frame stride W*H*3 values; a sharded call writes
 *     only its own rows of each frame.  Either buffer may be NULL.
 *   - Every camera passes the checks of rtclj_ctx_render before anything runs; otherwise RTCLJ_E_INVALID with a message
 *     naming the frame, and nothing is written.  RTCLJ_E_INVALID as well: n_frames <= 0, a null camera array, sizes that
 *     differ between frames, RTCLJ_F_WAVE_KERNEL or RTCLJ_F_SPLIT_KERNEL.  max_depth <= 0 renders black frames.
 *   - Stats (rtclj_ctx_stats after rtclj_ctx_render_frames, or the stats of rtclj_render_frames) cover the whole call:
 *     counters summed over the frames; samples_per_unit is the one every frame used.
 *   - A launch takes at most 128 frames (their cameras travel as kernel parameters), at most 2 GiB of scratch (unit
 *     sums, or per-sample colours in strict order) and fewer than 2^32 work units; longer sequences take several
 *     launches, and a frame that alone needs more scratch renders exactly as rtclj_ctx_render renders it. */
/* Device-resident, like rtclj_ctx_render: enqueues on `stream` without synchronising, honours shard_*; one context
 * serves one stream at a time.  d_out_linear / d_out_rgb8 are DEVICE pointers to n_frames full-size images. */
int rtclj_ctx_render_frames(rtclj_ctx *ctx, const rtclj_camera *cameras, int32_t n_frames,
                            const rtclj_params *params, void *d_out_linear, void *d_out_rgb8, void *stream);
/* Host buffers, like rtclj_render_multi: rows interleaved over `n_devices` GPUs (tiles of params->shard_rows rows,
 * <= 0: 1), one worker per device renders its rows of every frame; out_linear / out_rgb8 hold n_frames images. */
int rtclj_render_frames(const rtclj_scene *scene, const rtclj_camera *cameras, int32_t n_frames,
                        const rtclj_params *params, const int32_t *devices, int32_t n_devices,
                        double *out_linear, uint8_t *out_rgb8, rtclj_stats *stats);

/* ---- Progressive rendering: the compute-pixel loop (src/raytracing.clj:141-171) run in passes, so that
 * an image can be shown while it refines, stopped early or extended without tracing its samples again.
 *
 * An accumulation is fixed at its start by a scene, a camera and params; params->spp is the TARGET
 * sample count.  A pass of n samples adds samples [d, d + n) of every pixel to the pixel's running
 * sum, d being the samples done before it, and writes the images of the mean over d + n samples.
 *   - pass_unit, reported by the call that begins the accumulation: 1 in strict order
 *     (samples_per_unit >= spp, or <= 0 for a primary-ray render: the library's default there), else
 *     the unit size (samples_per_unit, or the library's choice when <= 0).  Every pass but the one that
 *     reaches spp must be a multiple of pass_unit; a pass that is not, or that would go beyond spp,
 *     returns RTCLJ_E_INVALID.
 *   - After passes totalling d samples the images (linear and 8-bit) are bit-identical to
 *     rtclj_ctx_render with the same camera and params but spp = d and samples_per_unit = pass_unit
 *     (strict order: samples_per_unit = d).  At d = spp that is the one-shot render of the
 *     accumulation's own params.  The images do not depend on the pass sizes, on the number of GPUs
 *     or on the device list.
 *   - RTCLJ_F_WAVE_KERNEL and RTCLJ_F_SPLIT_KERNEL are refused (RTCLJ_E_INVALID); spp is at most 2^30.
 *     max_depth <= 0 accumulates black.
 * Strict order holds at most 2 GiB of per-sample colours per context, whatever the image size. */

/* Device-resident, on the caller's stream (a cudaStream_t, NULL = the default stream); one accumulation
 * per context.  begin zeroes the running sums (24 B per pixel of the shard) and returns the pass unit;
 * step enqueues one pass and returns the samples per pixel done after it.  d_out_linear / d_out_rgb8 are
 * DEVICE pointers to full-size images, either may be NULL (the pass is still added).  rtclj_ctx_set_scene
 * ends the accumulation (step returns RTCLJ_E_INVALID until the next begin), and so does a failed
 * pass; rtclj_ctx_render between two steps leaves it intact.  rtclj_ctx_stats reports the last pass. */
int rtclj_ctx_accum_begin(rtclj_ctx *ctx, const rtclj_camera *camera, const rtclj_params *params,
                          int32_t *pass_unit, void *stream);
int rtclj_ctx_accum_step(rtclj_ctx *ctx, int32_t samples, void *d_out_linear, void *d_out_rgb8,
                         int32_t *samples_done, void *stream);

/* Host buffers, image rows interleaved over `n_devices` GPUs as in rtclj_render_multi (tiles of
 * params->shard_rows rows, <= 0: 1) -- what a JVM host calls to show an image while it refines.  The
 * handle owns a context per device and uploads the scene at create.  Each step runs one pass on every
 * device and writes the whole image into out_linear / out_rgb8 (either may be NULL); stats may be NULL.
 * One thread at a time per handle.  A step that fails on any device ends the accumulation. */
typedef struct rtclj_progressive rtclj_progressive; /* opaque */
int rtclj_progressive_create(const rtclj_scene *scene, const rtclj_camera *camera,
                             const rtclj_params *params, const int32_t *devices, int32_t n_devices,
                             int32_t *pass_unit, rtclj_progressive **out);
int rtclj_progressive_step(rtclj_progressive *p, int32_t samples, double *out_linear,
                           uint8_t *out_rgb8, int32_t *samples_done, rtclj_stats *stats);
int rtclj_progressive_destroy(rtclj_progressive *p); /* NULL is fine */

/* ---- Adaptive sampling: an accumulation whose passes trace only the pixels that are still noisy
 * (DESIGN.md section 4.10).  Same pass rules, refusals and target as above, plus a tolerance {abs, rel}
 * (finite, >= 0) and min_samples (>= 2 * pass_unit), else RTCLJ_E_INVALID.
 *   - Every pixel starts active.  A pass of n samples after d traces samples [d, d + n) of the pixels active
 *     when it starts; at its end each traced pixel p is tested and, once stopped, keeps its sample count n_p
 *     for good.
 *   - After every step the images of EVERY pixel are bit-identical to rtclj_ctx_render with spp = n_p and
 *     samples_per_unit = pass_unit (strict order: = n_p); each step rewrites the whole image.
 *   - The rule.  A unit is pass_unit samples (one chunk sum; strict order: one sample's colour).  Per pixel and
 *     channel S1 = the running sum and S2 = the sum of the squared unit sums in unit order; m = ceil(n_p / u)
 *     -- the short last chunk at the target counts as a unit like the others.  stderr = sqrt(fmax(((S2 -
 *     S1*S1/m) / (m (m - 1))) / (u u), 0)).  The pixel stays active iff n_p < spp and (n_p < min_samples or
 *     stderr > abs + rel * |mean| in some channel, mean = its linear value, or S1*S1 or S2 is not finite in
 *     some channel: moments that overflowed make the variance inf - inf, which the clamp would read as 0, so
 *     such a pixel counts as noisy).  The exported noise estimate is the clamped value.
 *   - A pixel's decision depends on its own sums only: for one sequence of pass sizes, images, sample-count
 *     map and noise are the same on every device list, shard_rows and kernel.  A different sequence of pass
 *     sizes may stop pixels at other counts.
 *   - With min_samples >= spp no pixel stops early: the plain accumulation, bit for bit.
 * Memory: 33 bytes per pixel of the shard on top of the accumulation's 24. */
int rtclj_ctx_accum_begin_adaptive(rtclj_ctx *ctx, const rtclj_camera *camera, const rtclj_params *params,
                                   const double tolerance[2] /* abs, rel */, int32_t min_samples,
                                   int32_t *pass_unit, void *stream);
/* after a step of an adaptive accumulation: d_samples (int32 W*H) / d_stderr (double W*H*3) are DEVICE
 * pointers to full-size images, either may be NULL (the shard's rows are written); active_pixels != NULL
 * synchronises `stream` and returns the shard's pixels still active.  RTCLJ_E_INVALID for a non-adaptive
 * accumulation. */
int rtclj_ctx_accum_noise(rtclj_ctx *ctx, int32_t *d_samples, double *d_stderr, uint64_t *active_pixels, void *stream);
/* host buffers, as rtclj_progressive_create / rtclj_progressive_step; noise writes the whole sample-count map
 * (int32 W*H) and noise estimate (double W*H*3), either may be NULL, and the pixels still active on all devices. */
int rtclj_progressive_create_adaptive(const rtclj_scene *scene, const rtclj_camera *camera,
                                      const rtclj_params *params, const double tolerance[2], int32_t min_samples,
                                      const int32_t *devices, int32_t n_devices, int32_t *pass_unit,
                                      rtclj_progressive **out);
int rtclj_progressive_noise(rtclj_progressive *p, int32_t *samples, double *noise, uint64_t *active_pixels);

/* Measures this GPU's arithmetic peaks with pure-FMA kernels (no memory traffic): scalar
 * FFMA, packed FFMA2 and fp64 DFMA, in TFLOP/s (2 flops per FMA), plus the SM count.
 * bench.py reports the roofline against these next to the nominal figure. */
int rtclj_calibrate_peaks(int32_t device, double *ffma_tflops, double *ffma2_tflops,
                          double *dfma_tflops, int32_t *sm_count);

/* ---- the rows SURVEY.md 8(f) ranks next: the steps either side of the loop ---- */

/* write-color!: 3 linear doubles -> 3 ints in 0..255 per pixel (host). */
int rtclj_quantise_rgb8(const double *linear, size_t n_values, uint32_t flags, uint8_t *out);

/* "P3\nW H\n255\n" + one "r g b\n" line per pixel.  Call with out == NULL to get a sufficient
 * capacity (an upper bound) in *len; the full call sets *len to the bytes written.  Images of 2^18
 * pixels and more are written by several short-lived host threads (half of the cores, at most 16). */
int rtclj_encode_ppm_p3(const uint8_t *rgb8, int32_t width, int32_t height, char *out,
                        size_t capacity, size_t *len);

/* The same writer as kernels on the device (row f-1 of SURVEY.md section 8: at 3840x2160 the text is
 * 89 MB and a host writer costs more than the render of a primary-ray image).  d_rgb8 and d_out are
 * DEVICE pointers; the bytes produced are identical to rtclj_encode_ppm_p3's.  d_out == NULL is a
 * sizing call that returns the exact length.  Synchronises `stream` before returning (the length
 * comes back from the device).  rtclj_ctx_encode_ms reports the device time of the last call's
 * two phases (line lengths + scan; text write). */
int rtclj_ctx_encode_ppm_p3(rtclj_ctx *ctx, const uint8_t *d_rgb8, int32_t width, int32_t height,
                            char *d_out, size_t capacity, size_t *len, void *stream);
int rtclj_ctx_encode_ms(rtclj_ctx *ctx, double *count_scan_ms, double *write_ms);
/* Host buffers in and out, the encoding on `device` (copies inside the call). */
int rtclj_encode_ppm_p3_gpu(int32_t device, const uint8_t *rgb8, int32_t width, int32_t height,
                            char *out, size_t capacity, size_t *len);

/* An 8-bit RGB PNG of the same image (what ppm->png produces from the P3 file,
 * src/raytracing.clj:176 / src/ppm2png.clj:35-87 -- re-implemented from the PNG specification, the
 * reference file carries a GPL header and nothing of it is used).  Stored (uncompressed) deflate
 * blocks.  Call with out == NULL to get the required capacity in *len. */
int rtclj_encode_png(const uint8_t *rgb8, int32_t width, int32_t height, uint8_t *out, size_t capacity,
                     size_t *len);

/* A compressed PNG of the same image, encoded on the device.  The bytes are exactly those of this definition
 * (tests/png_model.py reproduces them; DESIGN.md section 4.11):
 *   1. Chunks: the signature; IHDR as rtclj_encode_png's (8-bit truecolour, no interlace); an IDAT holding only the
 *      zlib header 78 01; one IDAT per segment; an IDAT holding only the big-endian Adler-32 of the whole filtered
 *      stream; IEND.  Each chunk's CRC-32 covers its type and data.
 *   2. Filtering: each row is filtered with each of the five PNG filters (bpp 3; outside the image a = b = c = 0).
 *      The cost is the sum of |byte as int8| over the filtered row, filter 0 included; the lowest cost wins, a tie
 *      goes to the lower type.  The filtered stream F is H * (1 + 3W) bytes.
 *   3. Segments: F is cut at multiples of 65 536 bytes (the last segment may be shorter); segments are encoded
 *      independently, no match reaches back past a segment's first byte.
 *   4. Tokens: a maximal run of L equal bytes starting at s within a segment is a literal at s, then
 *      (L - 1) / 258 matches (258, distance 1), then the remainder q = (L - 1) % 258 as one match of length q if
 *      q >= 3, else as q literals (what zlib's greedy deflate_rle emits).
 *   5. Each segment is one dynamic block (BTYPE 2) of all its tokens plus end-of-block:
 *      - literal/length code lengths by package-merge limited to 15 bits; items ordered by (frequency, symbol)
 *        ascending, at equal weight leaves before packages (the end-of-block symbol and the segment's first literal
 *        are always present);
 *      - distance code: codes 0 and 1, length 1 each (HDIST = 2); only code 0 (distance 1) is emitted;
 *      - HLIT = highest used literal/length symbol + 1, at least 257;
 *      - the HLIT + HDIST lengths as one sequence: a zero run of 11..138 is symbol 18, of 3..10 symbol 17, longest
 *        first, greedily; a non-zero length is written once, then symbol 16 covers each further run of 3..6
 *        repeats of it; everything else is a literal length;
 *      - code-length code by package-merge limited to 7 bits, same ordering; if only one symbol is used, the lowest
 *        other symbol gets length 1 as well;
 *      - HCLEN trimmed on the order 16 17 18 0 8 7 9 6 10 5 11 4 12 3 13 2 14 1 15, at least 4 entries;
 *      - canonical codes (RFC 1951 3.2.2), packed LSB-first.
 *   6. Stored fallback: if the dynamic encoding, flush included, is not shorter in bytes than stored blocks of at
 *      most 65 535 bytes, the segment is written stored (incompressible noise).
 *   7. A dynamic segment but the last is followed by an empty stored block (sync flush: 000, padding to the byte,
 *      00 00 FF FF); a stored segment ends on a byte boundary; the last segment's last block has BFINAL = 1 and is
 *      padded to the byte.
 * out == NULL (d_out == NULL) is the sizing call: *len receives a sufficient capacity, the size with every segment
 * stored, and nothing runs on the GPU.  A capacity below the exact length returns RTCLJ_E_BUFFER with *len set to
 * the exact length.  Non-positive sizes, null pointers and images whose F would exceed 2^31 - 2 segments return
 * RTCLJ_E_INVALID.  rtclj_ctx_encode_png reads the DEVICE image d_rgb8 and writes DEVICE memory d_out; it keeps F
 * (the image's bytes plus one per row) and one 64 KiB staging slot per segment in the context, and synchronises
 * `stream` (the length comes back from the device). */
int rtclj_ctx_encode_png(rtclj_ctx *ctx, const uint8_t *d_rgb8, int32_t width, int32_t height, uint8_t *d_out,
                         size_t capacity, size_t *len, void *stream);
/* Host buffers in and out, the encoding on `device` (copies inside the call). */
int rtclj_encode_png_gpu(int32_t device, const uint8_t *rgb8, int32_t width, int32_t height, uint8_t *out,
                         size_t capacity, size_t *len);
/* rtclj_render_multi_ppm with this PNG writer in place of the P3 writer: renders on `n_devices` GPUs, assembles the
 * 8-bit rows on devices[0] and encodes them there; only the PNG crosses PCIe.  The bytes are those of
 * rtclj_encode_png_gpu on rtclj_render's rgb8 image. */
int rtclj_render_multi_png(const rtclj_scene *scene, const rtclj_camera *camera, const rtclj_params *params,
                           const int32_t *devices, int32_t n_devices, uint8_t *out, size_t capacity, size_t *len,
                           rtclj_stats *stats);

/* The reader half of ppm->png (src/ppm2png.clj:35-87 reads "P3", "W H", a maximum <= 255 and one
 * "r g b" line per pixel; this parser accepts any whitespace between the tokens).  Call with
 * out_rgb8 == NULL to get the dimensions; RTCLJ_E_INVALID for a malformed file (bad magic, bad
 * dimensions, maximum outside 0..255, a component outside 0..max, too few or too many values),
 * RTCLJ_E_BUFFER if capacity < 3*W*H.  Bodies of 4 MB and more are parsed by several short-lived host
 * threads (at most 16); results and errors are those of the one-thread parser. */
int rtclj_decode_ppm_p3(const char *text, size_t len, int32_t *width, int32_t *height,
                        uint8_t *out_rgb8, size_t capacity);

/* Clojure's Ratio -> double (Ratio.doubleValue rounds through 16 decimal digits). */
double rtclj_ratio_to_double(int64_t num, int64_t den);
int rtclj_camera_main(int32_t width, int32_t height, double vfov, const double look_from[3],
                      const double look_at[3], const double vup[3], double defocus_angle,
                      double focus_dist, rtclj_camera *out);
int rtclj_camera_realm(int32_t width, int32_t height, double vfov, const double look_from[3],
                       const double look_at[3], const double vup[3], rtclj_camera *out);
int rtclj_camera_i(int32_t width, int32_t height, rtclj_camera *out);

/* Fills caller arrays (capacity `cap` spheres) with the random-sphere field over the
 * integer grid [lo,hi)^2; *n_out receives the sphere count (call with cap = 0 to size). */
int rtclj_scene_random_field(uint64_t seed, int32_t lo, int32_t hi, int32_t cap, double *center_xyz,
                             double *radius, int32_t *material, double *albedo_rgb, double *fuzz,
                             double *ior, int32_t *n_out);

#ifdef __cplusplus
}
#endif
#endif
