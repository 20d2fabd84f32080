// Kernel parameters and per-pixel epilogue shared by the two raytracer kernels.
#pragma once
#include "common.cuh"
#include "rt_exact.cuh"

struct RtKParams {
  float cam[4];
  float focal;
  float R[16];
  int W, H, row0, row1;
  int il_n, il_r;            // 16-row block b of the range is rendered by the launch with b % il_n == il_r
  int blocks_y;              // 16-row blocks in [row0, row1) (all of them, not only this launch's)
  int n_lights;
  float lights[B200_MAX_LIGHTS][7];
  const float4 *geom;        // 3 x float4 per triangle: v0, e1, e2
  const rt_triangle *src;    // as uploaded; normal / colour are gathered from here
  const rt_sphere *sph;
  int n_tris, n_sph;
  // filtered kernel only
  const float4 *planes;      // see rt_filtered.cuh
  const float *dt_cam;       // per triangle: det(camera - v0, e1, e2)
  const float *self_D;       // per (light, triangle): see RtPrepParams
  int tris_per_tile;
  // direction grids (rt_grid.cuh), GRID kernels only
  const unsigned *cell_off;  // first entry of each cell's list
  const unsigned *cell_cnt;  // entries in it
  const float4 *cell_rec;    // plane records, list by list
  const int *cell_idx;       // triangle index of each entry
  // GRID kernels, frames that follow a frame of the same shape: blocks run in the order of `plan` (1-D launch) and
  // the blocks that were expensive last time are split into eight launches of four pixels per warp (see rt_plan_kernel)
  const unsigned *plan;      // entry: block x | block row of this launch << 12 | column of the 8 x 4 patches << 24 | split << 27
  const unsigned *plan_n;    // entries (blocks beyond it leave at once)
  unsigned *block_cost;      // this frame's cost per block (cycles >> 8 of its slowest warp; x 8 when split), for the next frame's plan
  int gx;                    // 16-pixel blocks per row of blocks
  // outputs: full-frame addressing (pixel (x, y) at y*W + x); any may be null
  float *rgb;
  float *depth;
  int32_t *index;
  uint32_t *argb;
  unsigned long long *counters;  // [0] shadow rays, [1] exact evaluations (filtered kernel)
};

// Colour and shading normal of the surface that was hit (skeleton.cpp:148-149,
// 377-387; Sphere::getNormal TestModelH.h:68-75).
__device__ __forceinline__ void rt_surface(const RtKParams &p, int idx, float px, float py, float pz,
                                           float *col, float &nx, float &ny, float &nz) {
  if (idx >= 0) {
    const rt_triangle *t = p.src + idx;
    col[0] = __ldg(&t->color[0]); col[1] = __ldg(&t->color[1]); col[2] = __ldg(&t->color[2]);
    nx = __ldg(&t->normal[0]); ny = __ldg(&t->normal[1]); nz = __ldg(&t->normal[2]);
  } else {
    const rt_sphere *s = p.sph + (-1 - idx);
    col[0] = s->color[0]; col[1] = s->color[1]; col[2] = s->color[2];
    const float ax = xsub(px, s->centre[0]), ay = xsub(py, s->centre[1]), az = xsub(pz, s->centre[2]);
    const float inv = xdiv(1.0f, xsqrt(xdot3(ax, ay, az, ax, ay, az)));
    nx = xmul(ax, inv); ny = xmul(ay, inv); nz = xmul(az, inv);
  }
}

// averageLight = pixelColour / 9 or black (skeleton.cpp:160-166), then the
// optional PutPixelSDL quantisation.
__device__ __forceinline__ void rt_store_pixel(const RtKParams &p, size_t pid, bool valid, const float *pix) {
  float o[3] = {0.f, 0.f, 0.f};
  if (valid) { o[0] = xdiv_const<9>(pix[0]); o[1] = xdiv_const<9>(pix[1]); o[2] = xdiv_const<9>(pix[2]); }
  if (p.rgb) { p.rgb[3 * pid] = o[0]; p.rgb[3 * pid + 1] = o[1]; p.rgb[3 * pid + 2] = o[2]; }
  if (p.argb) p.argb[pid] = put_pixel_argb(o[0], o[1], o[2]);
}

__device__ __forceinline__ void rt_count(unsigned long long *counter, unsigned long long n) {
  // warp-level sum, then one atomic per warp
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
  if ((threadIdx.x & 31) == 0 && n) atomicAdd(counter, n);
}

__device__ __forceinline__ void rt_count_shadow(const RtKParams &p, unsigned long long n) {
  rt_count(p.counters + 0, n);
}

// ClosestIntersection (skeleton.cpp:263-363) by brute force: the reference arithmetic on every triangle, then every
// sphere (rt_bruteforce_kernel, rt_rays_bruteforce_kernel).
__device__ __forceinline__ RtHit rt_closest_bruteforce(const RtKParams &p, float sx, float sy, float sz,
                                                       float dx, float dy, float dz) {
  RtHit best;
  best.t = 0.f; best.dist = FLT_MAX; best.idx = 0;
  const float len = xsqrt(xdot3(dx, dy, dz, dx, dy, dz));  // glm::length(dir3), :307
  for (int i = 0; i < p.n_tris; ++i) {
    const float4 g0 = __ldg(p.geom + 3 * i), g1 = __ldg(p.geom + 3 * i + 1), g2 = __ldg(p.geom + 3 * i + 2);
    rt_exact_triangle(sx, sy, sz, dx, dy, dz, len, g0, g1, g2, i, best);
  }
  rt_exact_spheres(p.sph, p.n_sph, sx, sy, sz, dx, dy, dz, best);
  return best;
}
