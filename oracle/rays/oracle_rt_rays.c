/* oracle_rt_rays.c -- ClosestIntersection and DirectLight's shadow test for caller-supplied rays.
 *
 * TEST INFRASTRUCTURE ONLY, like oracle_rt.c: checks the library's ray queries (rt_closest_hits,
 * rt_occluded); never linked into or loaded by the product library.
 *
 * It includes oracle_rt.c whole, so the two entries below call that file's closest_intersection,
 * arithmetic unchanged, and builds into a library of its own (tests/rays_helpers.py compiles it with
 * oracle/Makefile's flags: -ffp-contract=off, no -march).
 */
#include "../oracle_rt.c"
/* ClosestIntersection for caller-supplied rays (raytracer/Source/skeleton.cpp:263-363): rays8 holds start[4],
 * dir[4] per ray; out receives the Intersection (skeleton.cpp:40-45, 28 bytes).  On a miss (distance not below
 * FLT_MAX) position is 0 and both indices -1; distance is what the reference leaves. */
int oracle_rt_closest(const float *rays8, int n_rays, const void *tris_, int n_tris, const void *sph_, int n_sph,
                      void *out_) {
  o_isect *out = (o_isect *)out_;
  for (int i = 0; i < n_rays; ++i) {
    o_isect is;
    memset(&is, 0, sizeof is);
    is.tri = -1; is.sph = -1;
    if (!closest_intersection(rays8 + 8 * i, rays8 + 8 * i + 4, (const o_tri *)tris_, n_tris, (const o_sph *)sph_,
                              n_sph, &is)) {
      is.pos[0] = is.pos[1] = is.pos[2] = is.pos[3] = 0.0f;
      is.tri = -1; is.sph = -1;
    }
    out[i] = is;
  }
  return 0;
}

/* DirectLight's shadow test (skeleton.cpp:394-397) for caller-supplied rays and limits:
 * out[i] = ClosestIntersection(...) && distance < max_distance[i]. */
int oracle_rt_occluded(const float *rays8, const float *max_distance, int n_rays, const void *tris_, int n_tris,
                       const void *sph_, int n_sph, uint8_t *out) {
  for (int i = 0; i < n_rays; ++i) {
    o_isect is;
    const int hit = closest_intersection(rays8 + 8 * i, rays8 + 8 * i + 4, (const o_tri *)tris_, n_tris,
                                         (const o_sph *)sph_, n_sph, &is);
    out[i] = (hit && is.distance < max_distance[i]) ? 1 : 0;
  }
  return 0;
}
