/* oracle_rt_direct_light.c -- DirectLight for caller-supplied hits.
 *
 * TEST INFRASTRUCTURE ONLY, like oracle_rt.c: checks the library's rt_direct_light; never linked into or loaded by
 * the product library.
 *
 * It includes oracle_rt_rays.c whole (and through it oracle_rt.c), so one library holds the ray-query entries and
 * the entry below, which calls oracle_rt.c's direct_light, arithmetic unchanged.  tests/direct_light_helpers.py
 * compiles it with oracle/Makefile's flags (-ffp-contract=off, no -march).
 */
#include "oracle_rt_rays.c"

/* DirectLight (skeleton.cpp:366-415) for caller-supplied hits (28-byte Intersection each) and lights (pos[4],
 * colour[3] each): power[(i * n_lights + l) * 3 + c], one call of direct_light per (entry, light).  The entry rule of
 * the reference's `if (triangleIndex != -1)`: triangle_index != -1 names that triangle, which must lie in
 * [0, n_tris); otherwise sphere_index must lie in [0, n_sph).  Any other entry gives 0 and traces nothing.
 * *n_shadow (if non-null) receives the shadow rays traced. */
int oracle_rt_direct_light(const void *hits_, int n_hits, const void *tris_, int n_tris, const void *sph_, int n_sph,
                           const float *lights7, int n_lights, float *power, uint64_t *n_shadow) {
  const o_isect *hits = (const o_isect *)hits_;
  uint64_t shadow = 0;
  for (int i = 0; i < n_hits; ++i) {
    const o_isect *is = &hits[i];
    const int named = is->tri != -1 ? (is->tri >= 0 && is->tri < n_tris) : (is->sph >= 0 && is->sph < n_sph);
    for (int l = 0; l < n_lights; ++l) {
      float *p = power + ((size_t)i * n_lights + l) * 3;
      if (named) direct_light(is, (const o_tri *)tris_, n_tris, (const o_sph *)sph_, n_sph, lights7 + 7 * l, p, &shadow);
      else p[0] = p[1] = p[2] = 0.0f;
    }
  }
  if (n_shadow) *n_shadow = shadow;
  return 0;
}
