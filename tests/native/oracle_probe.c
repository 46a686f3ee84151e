/* rto_probe_render: the CPU oracle's render (oracle/rt_oracle.c, compiled into this file, which leaves it as it is)
 * with a probe on every closest-hit scan of trace_sample.  Test infrastructure: it shows which paths a scene
 * reaches in the REFERENCE's arithmetic, so that a GPU test case cannot silently stop covering the path it is for
 * (tests/test_gpu_degenerate_rays.py).
 *
 * The probe sits in the t_max argument of trace_sample's one call of hit_anything, the only INFINITY in
 * rt_oracle.c: the macro below evaluates probe_scan(origin, dir) and then gives INFINITY.  rto_probe_render checks
 * that the probe saw exactly one scan per segment, so it fails if the hook ever moves.
 *
 * counts[0] scans; [1] scans of a direction the kernels treat as degenerate (fp32 |d|^2 outside (1e-30, 1e30),
 * the fp32 arithmetic of make_view); [2] scans whose closest root is NaN (an accepted NaN root); [3] segments. */
#include <math.h>
#include <stdint.h>

static uint64_t probe_counts[3];
static void probe_scan(double ox, double oy, double oz, double dx, double dy, double dz);
#undef INFINITY
#define INFINITY (probe_scan(origin.x, origin.y, origin.z, dir.x, dir.y, dir.z), HUGE_VAL)
#include "../../oracle/rt_oracle.c"
#undef INFINITY
#define INFINITY HUGE_VAL

static const rto_scene *probe_scene;

static void probe_scan(double ox, double oy, double oz, double dx, double dy, double dz) {
  probe_counts[0]++;
  const float fx = (float)dx, fy = (float)dy, fz = (float)dz;
  const float l2 = fx * fx + fy * fy + fz * fz;
  if (!(l2 > 1e-30f && l2 < 1e30f)) probe_counts[1]++;
  hit_rec rec;
  if (hit_anything(probe_scene, v3_make(ox, oy, oz), v3_make(dx, dy, dz), 1e-3, HUGE_VAL, &rec) && rec.t != rec.t)
    probe_counts[2]++;
}

int rto_probe_render(const rto_scene *scene, const rto_camera *cam, const rto_params *prm, uint64_t counts[4]) {
  rto_stats st;
  probe_scene = scene;
  memset(probe_counts, 0, sizeof probe_counts);
  /* one thread: the counters are plain statics */
  if (rto_render(scene, cam, prm, 1, 0, cam->height, NULL, NULL, &st) != 0) return 1;
  if (probe_counts[0] != st.segments) return 2;
  counts[0] = probe_counts[0]; counts[1] = probe_counts[1]; counts[2] = probe_counts[2]; counts[3] = st.segments;
  return 0;
}
