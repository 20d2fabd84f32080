/* oracle_rt_samples.c -- Draw with the caller's own sample offsets per pixel.
 *
 * TEST INFRASTRUCTURE ONLY, like oracle_rt.c: checks the library's render_raytrace_samples; never linked into or
 * loaded by the product library.
 *
 * It includes oracle_rt_rays.c whole (and through it oracle_rt.c), as oracle_rt_direct_light.c does, and restates
 * oracle_rt_render's pixel loop with an offset table in place of the 3x3 grid; closest_intersection and
 * direct_light are called unchanged.  tests/samples_helpers.py compiles it with oracle/Makefile's flags
 * (-ffp-contract=off, no -march).
 */
#include "oracle_rt_rays.c"

/* Draw (raytracer/Source/skeleton.cpp:104-169), rows [row0, row1), with sample k of every pixel the ray along
 * (dir.x + offsets[2k], dir.y + offsets[2k+1], focal), k < n_samples, in that order; the pixel is
 * pix / (float)n_samples if any sample hit.  dist/index are those of sample depth_sample.  Outputs are full-frame
 * arrays (only the band's rows are written); any may be NULL.  counts[0] += primary rays, counts[1] += shadow
 * rays.  With offsets 0.5 * (i, j), i = -1..1 outer, j = -1..1 inner, and depth_sample = 4 this is
 * oracle_rt_render. */
int oracle_rt_samples(int W, int H, float focal, const float *cam, const float *R, const float *lights7,
                      int n_lights, const void *tris_, int n_tris, const void *sph_, int n_sph, const float *offsets,
                      int n_samples, int depth_sample, int row0, int row1, float *rgb_out, float *dist_out,
                      int32_t *index_out, uint32_t *argb_out, uint64_t *counts) {
  const o_tri *tris = (const o_tri *)tris_;
  const o_sph *sph = (const o_sph *)sph_;
  uint64_t n_primary = 0, n_shadow = 0;
  for (int v = row0; v < row1; ++v) {
    for (int u = 0; u < W; ++u) {
      /* dir = R * vec4(u - W/2, v - H/2, f, 1): glm mat4*vec4 pairwise sums
       * (glm/glm/detail/type_mat4x4.inl:640-652) */
      float x = (float)(u - W / 2), y = (float)(v - H / 2);
      float dir[4];
      for (int r = 0; r < 4; ++r)
        dir[r] = (R[0 + r] * x + R[4 + r] * y) + (R[8 + r] * focal + R[12 + r] * 1.0f);
      float pix[3] = {0.f, 0.f, 0.f};
      int valid = 0;
      for (int k = 0; k < n_samples; ++k) {
        float nd[3] = {dir[0] + offsets[2 * k], dir[1] + offsets[2 * k + 1], focal};
        o_isect is;
        ++n_primary;
        int hit = closest_intersection(cam, nd, tris, n_tris, sph, n_sph, &is);
        if (k == depth_sample) {
          size_t p = (size_t)v * W + u;
          if (dist_out) dist_out[p] = hit ? is.distance : INFINITY;
          if (index_out) index_out[p] = hit ? (is.tri != -1 ? is.tri : -1 - is.sph) : INT32_MIN;
        }
        if (hit) {
          valid = 1;
          const float *oc = is.tri != -1 ? tris[is.tri].color : sph[is.sph].color;
          for (int l = 0; l < n_lights; ++l) {
            float p3[3];
            direct_light(&is, tris, n_tris, sph, n_sph, lights7 + 7 * l, p3, &n_shadow);
            pix[0] += p3[0]; pix[1] += p3[1]; pix[2] += p3[2];
          }
          pix[0] = pix[0] + oc[0] * 0.5f;
          pix[1] = pix[1] + oc[1] * 0.5f;
          pix[2] = pix[2] + oc[2] * 0.5f;
        }
      }
      float outc[3] = {0.f, 0.f, 0.f};
      const float n = (float)n_samples;
      if (valid) { outc[0] = pix[0] / n; outc[1] = pix[1] / n; outc[2] = pix[2] / n; }
      size_t p = (size_t)v * W + u;
      if (rgb_out) { rgb_out[3 * p] = outc[0]; rgb_out[3 * p + 1] = outc[1]; rgb_out[3 * p + 2] = outc[2]; }
      if (argb_out) argb_out[p] = put_pixel(outc);
    }
  }
  if (counts) { counts[0] += n_primary; counts[1] += n_shadow; }
  return 0;
}
