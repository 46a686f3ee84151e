/* rto_sample_colors: the colour of every sample [0, spp) of each pixel of rows [row_begin, row_end), from the CPU
 * oracle's own trace_sample (oracle/rt_oracle.c is compiled into this file, which leaves it as it is and reaches its
 * internal function).  out: [rows][W][spp][3] doubles.  Test infrastructure: it gives the adaptive-sampling tests
 * the unit sums from an implementation other than the kernels (tests/test_gpu_adaptive.py). */
#include "../../oracle/rt_oracle.c"

int rto_sample_colors(const rto_scene *scene, const rto_camera *cam, const rto_params *prm, int row_begin,
                      int row_end, double *out) {
  if (!scene || !cam || !prm || !out || scene->n < 0 || cam->width <= 0 || prm->spp <= 0 || row_begin < 0 ||
      row_end > cam->height)
    return 1;
  tracer tr;
  memset(&tr, 0, sizeof tr);
  tr.scene = scene; tr.cam = cam; tr.prm = prm;
  tr.k0 = (uint32_t)prm->seed; tr.k1 = (uint32_t)(prm->seed >> 32);
  tr.att_stack = (int32_t *)malloc(sizeof(int32_t) * (size_t)(prm->max_depth > 0 ? prm->max_depth : 1));
  const int W = cam->width;
  for (int j = row_begin; j < row_end; ++j)
    for (int i = 0; i < W; ++i) {
      const uint32_t pixel = (uint32_t)j * (uint32_t)W + (uint32_t)i;
      double *o = out + ((size_t)(j - row_begin) * (size_t)W + (size_t)i) * (size_t)prm->spp * 3u;
      for (int k = 0; k < prm->spp; ++k) {
        const v3 c = trace_sample(&tr, pixel, i, j, (uint32_t)k);
        o[3 * k] = c.x; o[3 * k + 1] = c.y; o[3 * k + 2] = c.z;
      }
    }
  free(tr.att_stack);
  return 0;
}
