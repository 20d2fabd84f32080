// rt_filtered_kernel: see rt_filtered.cuh for the method.  The long, rarely
// executed reference-arithmetic pieces are __noinline__ so that the hot filter
// loops stay small enough for the instruction cache.
#pragma once

// Reference arithmetic for one (primary ray, triangle) pair; `inside` = the
// filter proved `check` (:328) true, so u and v need not be formed.
__device__ __noinline__ RtHit rt_ex_primary(const float4 *__restrict__ geom, const float *__restrict__ dt_cam,
                                            float cx, float cy, float cz, int tri, int inside, float dx, float dy,
                                            float dz, float len, RtHit best) {
  const float4 g0 = __ldg(geom + 3 * tri), g1 = __ldg(geom + 3 * tri + 1), g2 = __ldg(geom + 3 * tri + 2);
  const float e1x = g0.w, e1y = g1.x, e1z = g1.y, e2x = g1.z, e2y = g1.w, e2z = g2.x;
  const float D = xdet3(-dx, -dy, -dz, e1x, e1y, e1z, e2x, e2y, e2z);
  const float t = xdiv(__ldg(dt_cam + tri), D);   // numerator: the same for every primary ray (rt_prep_planes_kernel)
  const float distance = xmul(t, len);
  if (distance < 0.0f) return best;
  // The reference walks the triangles in ascending order and replaces on a strict `<`
  // (:313): the closest hit, lowest index on ties.  Written order-independently, because
  // the direction-grid lists (rt_grid.cuh) are unordered.
  if (distance > best.dist || distance > FLT_MAX) return best;
  if (distance == best.dist && (best.dist == FLT_MAX || tri > best.idx)) return best;
  if (!inside) {
    const float sx = xsub(cx, g0.x), sy = xsub(cy, g0.y), sz = xsub(cz, g0.z);
    const float u = xdiv(xdet3(-dx, -dy, -dz, sx, sy, sz, e2x, e2y, e2z), D);
    const float v = xdiv(xdet3(-dx, -dy, -dz, e1x, e1y, e1z, sx, sy, sz), D);
    if (!((u >= 0) && (v >= 0) && (xadd(u, v) <= 1))) return best;
  }
  best.t = t; best.dist = distance; best.idx = tri;
  return best;
}

// Reference arithmetic for one (shadow ray, triangle) pair: does this triangle
// make DirectLight return black (skeleton.cpp:394-397)?  Any accepted hit with
// distance < r_magnitude does, because ClosestIntersection keeps the minimum.
__device__ __noinline__ int rt_ex_shadow(const float4 *__restrict__ geom, const rt_triangle *__restrict__ src,
                                         const rt_sphere *__restrict__ sph, int tri, int hit_idx, float px,
                                         float py, float pz, float Lx, float Ly, float Lz) {
  float col[3], nx, ny, nz;
  rt_surface2(src, sph, hit_idx, px, py, pz, col, nx, ny, nz);
  const float rx = xsub(Lx, px), ry = xsub(Ly, py), rz = xsub(Lz, pz);                          // :370
  const float ox = xadd(px, xmul(nx, 0.00001f)), oy = xadd(py, xmul(ny, 0.00001f)),
              oz = xadd(pz, xmul(nz, 0.00001f));                                                 // :394
  const float4 g0 = __ldg(geom + 3 * tri), g1 = __ldg(geom + 3 * tri + 1), g2 = __ldg(geom + 3 * tri + 2);
  const float e1x = g0.w, e1y = g1.x, e1z = g1.y, e2x = g1.z, e2y = g1.w, e2z = g2.x;
  const float sx = xsub(ox, g0.x), sy = xsub(oy, g0.y), sz = xsub(oz, g0.z);
  const float D = xdet3(-rx, -ry, -rz, e1x, e1y, e1z, e2x, e2y, e2z);
  const float Dt = xdet3(sx, sy, sz, e1x, e1y, e1z, e2x, e2y, e2z);
  const float rr = xdot3(rx, ry, rz, rx, ry, rz);
  // The usual outcome for the triangle the ray starts on: t = Dt / D is negative, so
  // `distance < 0` (:311) rejects it.  The sign of an IEEE quotient is the sign of
  // its operands and neither t nor t * len can underflow to -0 under the guards
  // below, so the division, the length and the double-precision r_magnitude are
  // not needed to know that.
  if (((Dt < 0.0f) != (D < 0.0f)) && fabsf(Dt) > 1e-20f * fabsf(D) && fabsf(D) < 1e30f && rr > 1e-30f && rr < 1e30f)
    return 0;
  const float len = xsqrt(rr);
  const float r_mag = rt_exact_rmag(rx, ry, rz);
  const float t = xdiv(Dt, D);
  const float distance = xmul(t, len);
  if (distance < 0.0f) return 0;
  if (!(distance < r_mag) || distance > FLT_MAX) return 0;
  const float u = xdiv(xdet3(-rx, -ry, -rz, sx, sy, sz, e2x, e2y, e2z), D);
  const float v = xdiv(xdet3(-rx, -ry, -rz, e1x, e1y, e1z, sx, sy, sz), D);
  return ((u >= 0) && (v >= 0) && (xadd(u, v) <= 1)) ? 1 : 0;
}

// Conservative sphere pre-test: the reference reports no root when
// discriminant = b*b - 4*a*c < 0 (TestModelH.h:27-28).  disc = 4 q with
// q = (d.L)^2 - (d.d)(L.L - r^2); reject when q is negative beyond the rounding
// error of either evaluation (|error| < 2e-6 (d.d)(L.L + r^2), tolerance 1e-4).
__device__ __forceinline__ bool rt_sphere_may_hit(const rt_sphere &s, float sx, float sy, float sz, float dx,
                                                  float dy, float dz) {
  const float Lx = sx - s.centre[0], Ly = sy - s.centre[1], Lz = sz - s.centre[2];
  const float dL = fmaf(dx, Lx, fmaf(dy, Ly, dz * Lz));
  const float dd = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
  const float LL = fmaf(Lx, Lx, fmaf(Ly, Ly, Lz * Lz));
  const float q = fmaf(dL, dL, -dd * (LL - s.radius_squared));
  const float tol = 1e-4f * fmaf(dL, dL, dd * (LL + s.radius_squared));
  return !(q < -tol);
}

struct RtSphT { int hit; float t; };
__device__ __noinline__ RtSphT rt_ex_sphere(const rt_sphere *__restrict__ s, float sx, float sy, float sz, float dx,
                                            float dy, float dz) {
  RtSphT r;
  r.t = 0.f;
  r.hit = rt_exact_sphere(*s, sx, sy, sz, dx, dy, dz, r.t) ? 1 : 0;
  return r;
}

// DirectLight for one hit once the triangles' verdict (`occluded`) is known:
// sphere occluders, then the Lambert term (skeleton.cpp:366-415).  Also returns
// the surface colour for the indirect term (:156).
struct RtShade { float pw[3]; float col[3]; };
__device__ __noinline__ RtShade rt_ex_shade(const rt_triangle *__restrict__ src, const rt_sphere *__restrict__ sph,
                                            int n_sph, int hit_idx, float px, float py, float pz, float Lx,
                                            float Ly, float Lz, float lr, float lg, float lb, int occluded,
                                            int want_light) {
  RtShade o;
  float nx, ny, nz;
  rt_surface2(src, sph, hit_idx, px, py, pz, o.col, nx, ny, nz);
  o.pw[0] = o.pw[1] = o.pw[2] = 0.f;
  if (!want_light || occluded) return o;
  const float rx = xsub(Lx, px), ry = xsub(Ly, py), rz = xsub(Lz, pz);
  const float r_mag = rt_exact_rmag(rx, ry, rz);
  if (n_sph > 0) {
    const float ox = xadd(px, xmul(nx, 0.00001f)), oy = xadd(py, xmul(ny, 0.00001f)),
                oz = xadd(pz, xmul(nz, 0.00001f));
    for (int s = 0; s < n_sph; ++s) {
      if (!rt_sphere_may_hit(sph[s], ox, oy, oz, rx, ry, rz)) continue;
      float t;
      if (rt_exact_sphere(sph[s], ox, oy, oz, rx, ry, rz, t) && t < r_mag) return o;   // :348 + :395
    }
  }
  const float lcol[3] = {lr, lg, lb};
  rt_exact_lambert(rx, ry, rz, r_mag, nx, ny, nz, o.col, lcol, o.pw);
  return o;
}

// Hit point of sample k = 3 kx + ky, start + t * dir (skeleton.cpp:326): the sample's direction is
// (dir0 + 0.5 (kx - 1), dir1 + 0.5 (ky - 1), f) (:134-137), formed from the middle sample's
// (dx1, dy1) -- the same float as from dir0 / dir1, -0 included -- for a k known only at run time.
__device__ __forceinline__ void rt_hit_point(float cx, float cy, float cz, float dx1, float dy1, float dz, float t,
                                             int k, float &px, float &py, float &pz) {
  const int kx = k / 3, ky = k - 3 * kx;
  const float dx = xadd(dx1, xmul(0.5f, (float)(kx - 1))), dy = xadd(dy1, xmul(0.5f, (float)(ky - 1)));
  px = xadd(cx, xmul(t, dx)); py = xadd(cy, xmul(t, dy)); pz = xadd(cz, xmul(t, dz));
}

// Walks the lists a pixel block has to stream, tile by tile: the whole scene, or
// (GRID) the lists of the direction cells in cells[0 .. nc).  Uniform over the block.
struct RtCursor {
  const float4 *rec;
  const int *idx;
  int cnt, pos;
  const int *cells;
  int ci, nc;
};

__device__ __forceinline__ RtCursor rt_cursor_scene(const float4 *planes, int n_tris) {
  RtCursor c;
  c.rec = planes; c.idx = nullptr; c.cnt = n_tris; c.pos = 0; c.cells = nullptr; c.ci = 0; c.nc = 0;
  return c;
}
__device__ __forceinline__ RtCursor rt_cursor_cells(const int *cells, int nc) {
  RtCursor c;
  c.rec = nullptr; c.idx = nullptr; c.cnt = 0; c.pos = 0; c.cells = cells; c.ci = 0; c.nc = nc;
  return c;
}

template <bool GRID, int TILE>
__device__ __forceinline__ bool rt_cursor_next(const RtKParams &p, RtCursor &c, RtItem &it) {
  while (c.pos >= c.cnt) {
    if (!GRID || c.ci >= c.nc) return false;
    const int cell = c.cells[c.ci++];
    const unsigned off = __ldg(p.cell_off + cell);
    c.cnt = (int)__ldg(p.cell_cnt + cell);
    c.rec = p.cell_rec + (size_t)off * RT_REC_F4;
    c.idx = p.cell_idx + off;
    c.pos = 0;
  }
  it.rec = c.rec + (size_t)c.pos * RT_REC_F4;
  it.idx = c.idx ? c.idx + c.pos : nullptr;
  it.base = c.pos;
  it.cnt = min(TILE, c.cnt - c.pos);
  c.pos += TILE;
  return true;
}

// Shadow phase, GRID: the cube-map cell (around the light) that g = hit - light falls
// into: face * RT_GRID_FACE + j * RT_GRID_G + i, or -1 for a vector that has no direction.
// The division's rounding moves a direction by far less than the 2 % of a cell by
// which rt_grid_test_light widens every cell.
__device__ __forceinline__ int rt_grid_cell_of(float gx, float gy, float gz) {
  const float ax = fabsf(gx), ay = fabsf(gy), az = fabsf(gz);
  const int a = (ax >= ay && ax >= az) ? 0 : (ay >= az ? 1 : 2);
  const float ga = a == 0 ? gx : (a == 1 ? gy : gz);
  const float gb = a == 0 ? gy : (a == 1 ? gz : gx);
  const float gc = a == 0 ? gz : (a == 1 ? gx : gy);
  const float m = fabsf(ga);
  if (!(m > 1e-30f && m < 1e30f)) return -1;
  const float G = (float)RT_GRID_G;
  const int i = min(max((int)floorf((gb / m + 1.0f) * 0.5f * G), 0), RT_GRID_G - 1);
  const int j = min(max((int)floorf((gc / m + 1.0f) * 0.5f * G), 0), RT_GRID_G - 1);
  return (2 * a + (ga < 0.0f ? 1 : 0)) * RT_GRID_FACE + j * RT_GRID_G + i;
}

// Adds `cell` to the block's set (open addressing in shared memory; the list keeps
// the distinct cells).  *n_cells may run past RT_GRID_MAX_CELLS: the caller checks.
__device__ __forceinline__ void rt_grid_mark(int cell, int *table, int *cells, int *n_cells) {
  unsigned hsh = ((unsigned)cell * 2654435761u) >> (32 - RT_GRID_TABLE_LOG2);
  for (int probe = 0; probe < (1 << RT_GRID_TABLE_LOG2); ++probe) {
    const int old = atomicCAS(table + hsh, -1, cell);
    if (old == cell) return;
    if (old == -1) {
      const int pos = atomicAdd(n_cells, 1);
      if (pos < RT_GRID_MAX_CELLS) cells[pos] = cell;
      return;
    }
    hsh = (hsh + 1) & ((1u << RT_GRID_TABLE_LOG2) - 1);
  }
  atomicAdd(n_cells, RT_GRID_MAX_CELLS + 1);   // table full: stream the scene
}

// Resident blocks per SM: with the per-sample hit state in shared memory the scene-streaming
// kernel fits 80 registers and runs three blocks (24 warps) per SM, which hides the latency of
// its dependent exact arithmetic better than two blocks at 128 registers (measured: 1.21 vs 1.36 ms
// on the Cornell box at 4K); the grid kernels need 80 KB of shared memory per block: two.
#ifndef RT_MIN_BLOCKS
#define RT_MIN_BLOCKS 3
#endif
// Pixel of this thread in a batched launch: block (x, y) of whole frame blockIdx.z, warps as in rt_filtered_body.
// The indices are read afresh (volatile): merged with the kernel's own u and v, they were kept in a spill slot.
__device__ __forceinline__ size_t rt_views_pid(const RtKParams &p) {
  unsigned t, bx, by, bz;
  asm volatile("mov.u32 %0, %%tid.x;" : "=r"(t));
  asm volatile("mov.u32 %0, %%ctaid.x;" : "=r"(bx));
  asm volatile("mov.u32 %0, %%ctaid.y;" : "=r"(by));
  asm volatile("mov.u32 %0, %%ctaid.z;" : "=r"(bz));
  const int lane = t & 31, warp = t >> 5;
  const int u = bx * 16 + (warp & 1) * 8 + (lane & 7), v = by * 16 + (warp >> 1) * 4 + (lane >> 3);
  return ((size_t)bz * p.H + v) * p.W + u;
}

// VIEWS (scene streaming only): blockIdx.z is the view of a batched launch; its camera comes from vp, its camera
// records and dt_cam from its own slices, its pixels go to frame blockIdx.z of the outputs.
// SAMPLES: the pixel's samples are the caller's table sp (render_raytrace_samples) instead of the 3x3 grid.  They
// run in groups of up to nine in the nine slots of the hit state -- a primary walk and the shadow phase per group --
// and the pixel's running sum carries over from group to group in sample order.  Every bound of the primary-ray
// filters is built for a bundle of +-0.5 around the pixel's direction; rounding is monotone, so RN(dir + o) for
// |o| <= 0.5 lies between RN(dir - 0.5) and RN(dir + 0.5) and those bounds hold unchanged (DESIGN §3.5).
template <bool MULTI, bool GRID, bool VIEWS, bool SAMPLES = false>
__device__ __forceinline__ void rt_filtered_body(const RtKParams &p, const RtViewsParams *vp,
                                                 const RtSamplesParams *sp = nullptr) {
  // Scene streaming (GRID = false): the block shares one double-buffered ring of RT_TILE-record
  // tiles, refilled under __syncthreads.  Cell lists (GRID = true): every WARP has its own ring of
  // RT_WTILE-record tiles, its own cell set and no block barrier at all -- the lists are short,
  // and a warp on a dense or silhouette patch no longer holds the other seven back.
  static_assert(!(GRID && VIEWS), "batched views run the scene-streaming kernel");
  static_assert(!(SAMPLES && VIEWS), "batched views take Draw's nine samples");
  constexpr int TILE = GRID ? RT_WTILE : RT_TILE;
  constexpr int NRING = GRID ? RT_THREADS / 32 : 1;
  extern __shared__ __align__(128) float4 tile_smem[];  // NRING x 2 x TILE x 3 float4 (+ GRID: NRING x 2 x TILE int)
  __shared__ __align__(8) uint64_t bars_all[2 * NRING];
  __shared__ int s_cells_all[GRID ? NRING * RT_GRID_MAX_CELLS : 1];
  __shared__ int s_table_all[GRID ? NRING * (1 << RT_GRID_TABLE_LOG2) : 1];
  __shared__ int s_ncells_all[NRING];
  // grid kernels: the L0 survivors a warp has already worked on in this light phase (a triangle
  // is in the list of every cell it overlaps; a warp that walks several cells meets it again)
  __shared__ int s_seen_all[GRID ? NRING * RT_SEEN : 1];

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // which 16 x 16 pixel block: the launch's own coordinates, or (GRID, planned frames) what the plan says
  int bx = (int)blockIdx.x, by = (int)blockIdx.y, sub = -1;
  if (GRID && p.plan) {
    if (blockIdx.x >= *p.plan_n) return;
    const unsigned e = __ldg(p.plan + blockIdx.x);
    bx = (int)(e & 0xfffu); by = (int)((e >> 12) & 0xfffu);
    if ((e >> 27) & 1u) sub = (int)((e >> 24) & 7u);   // a split block: this launch takes one pixel column of every patch
  }
  // (kept in shared memory: two registers held over the whole kernel made it spill)
  __shared__ unsigned s_cost_t0[GRID ? NRING : 1];
  __shared__ int s_cost_at[GRID ? NRING : 1];
  __shared__ int s_split;
  if (GRID && lane == 0) {
    s_cost_t0[warp] = (unsigned)clock();     // 32 bits wrap after two seconds; a warp runs milliseconds
    s_cost_at[warp] = ((p.row0 >> 4) + by * p.il_n + p.il_r) * p.gx + bx;   // by the block's place in the whole frame
    if (warp == 0) s_split = sub >= 0;       // (read after the block barrier below)
  }
  // warp = 8x4 pixel patch; 8 warps tile a 16x16 block as 2 columns x 4 rows
  const int u = bx * 16 + (warp & 1) * 8 + (lane & 7);
  const int block_y = by * p.il_n + p.il_r;     // 16-row block of the range (interleaved launches)
  const int v = p.row0 + block_y * 16 + (warp >> 1) * 4 + (lane >> 3);
  const bool live = (u < p.W) && (v < p.row1) && (sub < 0 || (lane & 7) == sub);
  const int view = VIEWS ? (int)blockIdx.z : 0;
  // VIEWS: frame `view` of the outputs.  Formed again where the pixel is stored (held over the kernel, the
  // 64-bit offset made it spill more)
  const size_t pid = VIEWS ? 0 : (size_t)v * p.W + u;
#define PID (VIEWS ? rt_views_pid(p) : pid)
  const size_t origin_stride = (size_t)((p.n_tris + RT_TILE - 1) / RT_TILE) * RT_TILE * RT_REC_F4;
  const float *cam = VIEWS ? vp->view[view].cam : p.cam;
  const float *R = VIEWS ? vp->view[view].R : p.R;
  const float focal = VIEWS ? vp->view[view].focal : p.focal;
  const float4 *cam_planes = VIEWS ? p.planes + (size_t)view * origin_stride : p.planes;
  const int first_light = VIEWS ? vp->n_views : 1;    // origin of light 0's records

  if (threadIdx.x == 0) {
    for (int i = 0; i < 2 * NRING; ++i) mbar_init(&bars_all[i], 1);
    mbar_fence_init();
  }
  __syncthreads();
  const int ring_id = GRID ? warp : 0;
  uint64_t *bars = bars_all + 2 * ring_id;
  int *s_cells = s_cells_all + (GRID ? ring_id * RT_GRID_MAX_CELLS : 0);
  int *s_table = s_table_all + (GRID ? ring_id * (1 << RT_GRID_TABLE_LOG2) : 0);
  int &s_ncells = s_ncells_all[ring_id];
  int *s_seen = s_seen_all + (GRID ? ring_id * RT_SEEN : 0);
  const bool issuer = GRID ? lane == 0 : threadIdx.x == 0;     // who issues the ring's TMA copies
  auto ring_sync = [] { if (GRID) __syncwarp(); else __syncthreads(); };
  RtRing ring = rt_ring<TILE>(tile_smem + (size_t)ring_id * 2 * TILE * RT_REC_F4,
                              reinterpret_cast<int *>(tile_smem + (size_t)NRING * 2 * TILE * RT_REC_F4) + ring_id * 2 * TILE,
                              bars);

  // dir = R * vec4(u - W/2, v - H/2, f, 1)   (skeleton.cpp:126-128)
  const float x = (float)(u - p.W / 2), y = (float)(v - p.H / 2);
  const float dir0 = xadd(xadd(xmul(R[0], x), xmul(R[4], y)), xadd(xmul(R[8], focal), xmul(R[12], 1.0f)));
  const float dir1 = xadd(xadd(xmul(R[1], x), xmul(R[5], y)), xadd(xmul(R[9], focal), xmul(R[13], 1.0f)));
  const float dz = focal;
  const float cx = cam[0], cy = cam[1], cz = cam[2];
  // the nine sample directions (:134-137): three x offsets, three y offsets
  const float dxs[3] = {xadd(dir0, xmul(0.5f, -1.0f)), xadd(dir0, xmul(0.5f, 0.0f)), xadd(dir0, xmul(0.5f, 1.0f))};
  const float dys[3] = {xadd(dir1, xmul(0.5f, -1.0f)), xadd(dir1, xmul(0.5f, 0.0f)), xadd(dir1, xmul(0.5f, 1.0f))};
  // SAMPLES: slot k of the current group is sample smp0 + k of the caller's table, for k < ng
  int smp0 = 0, ng = 9;
#define RT_SDX(k) (SAMPLES ? xadd(dir0, sp->off[2 * (smp0 + (k))]) : dxs[(k) / 3])
#define RT_SDY(k) (SAMPLES ? xadd(dir1, sp->off[2 * (smp0 + (k)) + 1]) : dys[(k) % 3])
  unsigned n_exact = 0;
#ifdef RT_PROFILE_COUNTERS
  unsigned prof_cnt[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
#define RT_PC(i) (++prof_cnt[i])
#else
#define RT_PC(i)
#endif
#ifdef RT_PROFILE_CLOCK   // diagnostic build: where the long-running warps are and why (profiles/rt_block_cycles.py)
  const long long prof_t0 = clock64();
  unsigned prof_recs = 0, prof_cells = 0, prof_l1 = 0, prof_l2 = 0, prof_ex0 = 0;
#endif

  // The closest hit of each of the nine samples lives in shared memory (thread-private slices,
  // conflict-free: word k of thread t at [k][t]) instead of 27 registers.
  float *s_ht = reinterpret_cast<float *>(tile_smem + (size_t)NRING * 2 * TILE * RT_REC_F4) + (GRID ? NRING * 2 * TILE : 0);
  float *s_hd = s_ht + 9 * RT_THREADS;
  int *s_hi = reinterpret_cast<int *>(s_hd + 9 * RT_THREADS);
  float *s_len = s_hd + 18 * RT_THREADS;
#define HT(k) s_ht[(k) * RT_THREADS + threadIdx.x]
#define HD(k) s_hd[(k) * RT_THREADS + threadIdx.x]
#define HI(k) s_hi[(k) * RT_THREADS + threadIdx.x]
  // The scene-streaming kernel (80 registers) also keeps the nine direction lengths and the pixel's running colour
  // sum there: in registers, most of its spill traffic was that sum, stored and reloaded around every shading call.
  // The grid kernels (128 registers, no such spills) keep them in registers: 12 KB more shared memory per block
  // measured 1.2 % slower on the 100 800-triangle box (B200, 1000 W power limit).
  float len_r[GRID ? 9 : 1], pix_r[GRID ? 3 : 1];
#define LEN(k) (GRID ? len_r[GRID ? (k) : 0] : s_len[(k) * RT_THREADS + threadIdx.x])
#define PIX(c) (GRID ? pix_r[GRID ? (c) : 0] : s_len[(9 + (c)) * RT_THREADS + threadIdx.x])
  // SAMPLES: hit samples of the earlier groups (shadow-ray count), and whether any sample of the pixel hit
  unsigned n_hit = 0;
  bool any_hit = false;
  const int n_groups = SAMPLES ? (sp->n + 8) / 9 : 1;
  for (int grp = 0; grp < n_groups; ++grp) {   // (one pass without SAMPLES; the body keeps its indentation)
  if (SAMPLES) {
    smp0 = 9 * grp;
    ng = min(9, sp->n - smp0);
    if (grp > 0) ring_sync();   // the last light phase of the previous group is done with the ring and the cell set
  }
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    HT(k) = 0.f; HD(k) = FLT_MAX; HI(k) = 0;
    if (SAMPLES && k >= ng) continue;
    LEN(k) = xsqrt(xdot3(RT_SDX(k), RT_SDY(k), dz, RT_SDX(k), RT_SDY(k), dz));
  }

  // ============================ primary rays ============================
  {
    // bounding box of the warp's direction bundle in the (dx, dy) plane
    const float lo0 = warp_min(live ? dir0 : INFINITY), hi0 = warp_max(live ? dir0 : -INFINITY);
    const float lo1 = warp_min(live ? dir1 : INFINITY), hi1 = warp_max(live ? dir1 : -INFINITY);
    const bool warp_live = hi0 >= lo0;
    const float wc0 = 0.5f * (lo0 + hi0), wc1 = 0.5f * (lo1 + hi1);
    const float wh0 = (0.5f * (hi0 - lo0) + 0.5f) * 1.0001f + 1e-3f;
    const float wh1 = (0.5f * (hi1 - lo1) + 0.5f) * 1.0001f + 1e-3f;

    RtCursor cursor = rt_cursor_scene(cam_planes, p.n_tris);   // origin 0 (VIEWS: origin `view`)
    if (GRID) {
      if (issuer) s_cells[0] = block_y * (GRID ? p.gx : (int)gridDim.x) + bx;   // this block's own cell
      ring_sync();
      cursor = rt_cursor_cells(s_cells, warp_live ? 1 : 0);
    }
    RtItem item;
    bool have = rt_cursor_next<GRID, TILE>(p, cursor, item);
    if (issuer && have) rt_ring_issue<TILE>(ring, item);
    while (have) {
      const int buf = ring.issued & 1;
      ++ring.issued;
      ring_sync();   // everyone is done with the other buffer (it held the previous tile): refill it
      RtItem next_item;
      const bool have_next = rt_cursor_next<GRID, TILE>(p, cursor, next_item);
      if (issuer && have_next) rt_ring_issue<TILE>(ring, next_item);
      mbar_wait(&bars[buf], (ring.phase_bits >> buf) & 1u);
      ring.phase_bits ^= 1u << buf;
      const float4 *T = ring.buf[0] + (size_t)buf * TILE * RT_REC_F4;
      const int *Tidx = ring.smem_idx + buf * TILE;
      const bool listed = GRID && item.idx != nullptr;
      const int base = item.base;
      const int cnt = warp_live ? item.cnt : 0;
#ifdef RT_PROFILE_COUNTERS
      if (issuer) atomicAdd(p.counters + 12, (unsigned long long)item.cnt);
#endif
      item = next_item;
      have = have_next;
      for (int r0 = 0; r0 < cnt; r0 += 32) {
        // ---- L0: one triangle per lane vs the warp's bundle box ----
        bool pass = false;
        if (r0 + lane < cnt) {
          const float4 q0 = T[(r0 + lane) * 3], q1 = T[(r0 + lane) * 3 + 1], q2 = T[(r0 + lane) * 3 + 2];
          // E already covers the rounding of the centre evaluation (|wc| <= dmax);
          // the half-width terms are sums of non-negative products, inflated above
          pass = rt_box_may_hit_cam<GRID>(q0, q1, q2, wc0, wc1, wh0, wh1);
        }
        unsigned mask = __ballot_sync(0xffffffffu, pass);
        // ---- L1: every lane tests its pixel (centre, margin widened by the +-0.5 jitter)
        //      against every survivor and remembers the ones it needs ----
        unsigned mine = 0;
        while (mask) {
          const int j = __ffs(mask) - 1;
          mask &= mask - 1;
          const float4 q0 = T[(r0 + j) * 3], q1 = T[(r0 + j) * 3 + 1], q2 = T[(r0 + j) * 3 + 2];
          const float cu = fmaf(q0.x, dir0, fmaf(q0.y, dir1, q0.z));
          const float cv = fmaf(q0.w, dir0, fmaf(q1.x, dir1, q1.y));
          const float cw = fmaf(q1.z, dir0, fmaf(q1.w, dir1, q2.x));
          if (live) RT_PC(0);
          if (live && !(fminf(fminf(cu, cv), cw) < -q2.w)) mine |= 1u << j;
        }
        // ---- L2 / EX: each lane walks ITS OWN candidates, in ascending order; lanes are on
        //      different triangles here, so small triangles do not serialise the warp ----
        while (mine) {
          const int j = __ffs(mine) - 1;
          mine &= mine - 1;
          const int tri = listed ? Tidx[r0 + j] : base + r0 + j;
          const float4 q0 = T[(r0 + j) * 3], q1 = T[(r0 + j) * 3 + 1], q2 = T[(r0 + j) * 3 + 2];
          RT_PC(1);
          const float E = q2.y, dt_lo = q2.z;
          // ---- L2 / EX: per ray ----
#pragma unroll
          for (int k = 0; k < 9; ++k) {
            if (SAMPLES && k >= ng) continue;
            const float dx = RT_SDX(k), dy = RT_SDY(k);
            const float mU = fmaf(q0.x, dx, fmaf(q0.y, dy, q0.z));
            const float mV = fmaf(q0.w, dx, fmaf(q1.x, dy, q1.y));
            const float mW = fmaf(q1.z, dx, fmaf(q1.w, dy, q2.x));
            const float m3 = fminf(fminf(mU, mV), mW);
            if (m3 >= -E) {
              RT_PC(2);
              const float mN = mU + mV + mW;
              // reference distance >= dt_lo*len/(mN+E): cannot beat the current closest
              RtHit b;
              b.dist = HD(k);
              const bool farther = (mN > E) && (dt_lo * LEN(k) > b.dist * (mN + E));
              if (!farther) {
                ++n_exact;
                b.t = HT(k); b.idx = HI(k);
                const RtHit nb = rt_ex_primary(p.geom, VIEWS ? p.dt_cam + (size_t)blockIdx.z * p.n_tris : p.dt_cam, cx, cy, cz, tri, m3 >= E ? 1 : 0, dx, dy, dz, LEN(k), b);
                if (nb.idx != b.idx || nb.dist != b.dist) { HT(k) = nb.t; HD(k) = nb.dist; HI(k) = nb.idx; }
              }
            }
          }
        }
      }
    }
  }

  // spheres (skeleton.cpp:341-355)
  if (live) {
    for (int s = 0; s < p.n_sph; ++s) {     // per ray the spheres still come in ascending order
      // Bundle pre-test: an upper bound of q + tolerance (see rt_sphere_may_hit) over the pixel's
      // nine directions d = (dxs[1] +- 0.5, dys[1] +- 0.5, f).  Negative: no sample can report a root.
      {
        const float Lx = cx - __ldg(&p.sph[s].centre[0]), Ly = cy - __ldg(&p.sph[s].centre[1]),
                    Lz = cz - __ldg(&p.sph[s].centre[2]);
        const float r2 = __ldg(&p.sph[s].radius_squared);
        const float LL = fmaf(Lx, Lx, fmaf(Ly, Ly, Lz * Lz)), c = LL - r2;
        if (c > 0.0f) {                        // camera outside the sphere
          const float hw = 0.5002f;            // half-width of the bundle, with the rounding of the +-0.5 offsets
          const float dL = fabsf(fmaf(dxs[1], Lx, fmaf(dys[1], Ly, dz * Lz))) + hw * (fabsf(Lx) + fabsf(Ly));
          const float a_max = dL * dL * 1.00001f;
          const float ax0 = fmaxf(fabsf(dxs[1]) - hw, 0.0f), ay0 = fmaxf(fabsf(dys[1]) - hw, 0.0f);
          const float ax1 = fabsf(dxs[1]) + hw, ay1 = fabsf(dys[1]) + hw;
          const float dd_min = fmaf(ax0, ax0, fmaf(ay0, ay0, dz * dz)) * 0.99999f;
          const float dd_max = fmaf(ax1, ax1, fmaf(ay1, ay1, dz * dz)) * 1.00001f;
          if (a_max - dd_min * c < -1.001e-4f * (a_max + dd_max * (LL + r2))) continue;
        }
      }
#pragma unroll
      for (int k = 0; k < 9; ++k) {
        if (SAMPLES && k >= ng) continue;
        const float dx = RT_SDX(k), dy = RT_SDY(k);
        if (!rt_sphere_may_hit(p.sph[s], cx, cy, cz, dx, dy, dz)) continue;
        const RtSphT h = rt_ex_sphere(p.sph + s, cx, cy, cz, dx, dy, dz);
        if (h.hit && h.t < HD(k)) { HT(k) = h.t; HD(k) = h.t; HI(k) = -1 - s; }
      }
    }
  }
  unsigned active = 0;
  // HT(k): ray parameter of each hit; position = start + t * dir (:326 / :345)
#pragma unroll
  for (int k = 0; k < 9; ++k)
    if (live && HD(k) < FLT_MAX) active |= 1u << k;
  if (SAMPLES) {
    const int kd = sp->depth_sample - smp0;   // the depth sample's slot, if it is in this group
    if (live && kd >= 0 && kd < ng) {
      const bool hit = (active >> kd) & 1u;
      if (p.depth) p.depth[PID] = hit ? HD(kd) : INFINITY;
      if (p.index) p.index[PID] = hit ? HI(kd) : INT32_MIN;
    }
    n_hit += __popc(active);
    any_hit = any_hit || active != 0;
  } else if (live) {
    const bool hit4 = (active >> 4) & 1u;
    if (p.depth) p.depth[PID] = hit4 ? HD(4) : INFINITY;
    if (p.index) p.index[PID] = hit4 ? HI(4) : INT32_MIN;
  }

#ifdef RT_PROFILE_CLOCK
  prof_ex0 = n_exact;
#endif
  // ============================ shadow rays ============================
  constexpr int NL = MULTI ? B200_MAX_LIGHTS : 1;
  float dl[MULTI ? NL * 27 : 1];
  if (!SAMPLES || grp == 0) {
#pragma unroll
    for (int c = 0; c < 3; ++c) PIX(c) = 0.f;
  }
  const unsigned warp_active = __ballot_sync(0xffffffffu, active != 0);
  for (int l = 0; l < p.n_lights; ++l) {
    const float Lx = p.lights[l][0], Ly = p.lights[l][1], Lz = p.lights[l][2];
    unsigned occluded = 0;
    // g = hit - light per ray; boxes of the pixel's and the warp's bundles
    float glo[3] = {INFINITY, INFINITY, INFINITY}, ghi[3] = {-INFINITY, -INFINITY, -INFINITY};
#pragma unroll(GRID ? 1 : 9)   // grid kernels: smaller code (their warps run out of step and miss in the instruction cache)
    for (int k = 0; k < 9; ++k) {
      if ((active >> k) & 1u) {
        const float gx = -xsub(Lx, xadd(cx, xmul(HT(k), RT_SDX(k))));
        const float gy = -xsub(Ly, xadd(cy, xmul(HT(k), RT_SDY(k))));
        const float gz = -xsub(Lz, xadd(cz, xmul(HT(k), dz)));
        glo[0] = fminf(glo[0], gx); ghi[0] = fmaxf(ghi[0], gx);
        glo[1] = fminf(glo[1], gy); ghi[1] = fmaxf(ghi[1], gy);
        glo[2] = fminf(glo[2], gz); ghi[2] = fmaxf(ghi[2], gz);
      }
    }
    float pc[3], ph[3], wc[3], wh[3];
    float pnorm = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      pc[c] = 0.5f * (glo[c] + ghi[c]);
      ph[c] = 0.5f * (ghi[c] - glo[c]) * 1.0001f + 1e-7f * fmaxf(fabsf(glo[c]), fabsf(ghi[c]));
      pnorm = fmaxf(pnorm, fmaxf(fabsf(glo[c]), fabsf(ghi[c])));
      const float wl = warp_min(glo[c]), wu = warp_max(ghi[c]);
      wc[c] = 0.5f * (wl + wu);
      wh[c] = 0.5f * (wu - wl) * 1.0001f + 1e-7f * fmaxf(fabsf(wl), fabsf(wu));
    }
    if (!active) { pnorm = 0.f; pc[0] = pc[1] = pc[2] = 0.f; ph[0] = ph[1] = ph[2] = 0.f; }
    float wnorm = warp_max(pnorm) * 1.0001f;
    pnorm *= 1.0001f;
    // GRID (large scenes): a patch that straddles a silhouette has hits on two surfaces and
    // one box around both sweeps everything in between.  Split the bundle across the middle
    // of the box's longest axis and keep a tight box around each half.
    float wc2[3] = {0.f, 0.f, 0.f}, wh2[3] = {0.f, 0.f, 0.f}, wnorm2 = 0.f;
    bool two = false;
    // (a compact bundle -- extent below 3 % of its distance from the light -- is left alone)
    if (GRID && warp_active && fmaxf(wh[0], fmaxf(wh[1], wh[2])) > 0.03f * wnorm) {
      const int ax = (wh[0] >= wh[1] && wh[0] >= wh[2]) ? 0 : (wh[1] >= wh[2] ? 1 : 2);
      const float mid = ax == 0 ? wc[0] : (ax == 1 ? wc[1] : wc[2]);
      float alo[3] = {INFINITY, INFINITY, INFINITY}, ahi[3] = {-INFINITY, -INFINITY, -INFINITY};
      float blo[3] = {INFINITY, INFINITY, INFINITY}, bhi[3] = {-INFINITY, -INFINITY, -INFINITY};
#pragma unroll(GRID ? 1 : 9)   // grid kernels: smaller code (their warps run out of step and miss in the instruction cache)
      for (int k = 0; k < 9; ++k) {
        if ((active >> k) & 1u) {
          const float g[3] = {-xsub(Lx, xadd(cx, xmul(HT(k), RT_SDX(k)))), -xsub(Ly, xadd(cy, xmul(HT(k), RT_SDY(k)))),
                              -xsub(Lz, xadd(cz, xmul(HT(k), dz)))};
          const bool in_a = (ax == 0 ? g[0] : (ax == 1 ? g[1] : g[2])) < mid;
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            if (in_a) { alo[c] = fminf(alo[c], g[c]); ahi[c] = fmaxf(ahi[c], g[c]); }
            else { blo[c] = fminf(blo[c], g[c]); bhi[c] = fmaxf(bhi[c], g[c]); }
          }
        }
      }
      float na = 0.f, nb = 0.f;
      bool has_a = true, has_b = true;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float al = warp_min(alo[c]), au = warp_max(ahi[c]), bl = warp_min(blo[c]), bu = warp_max(bhi[c]);
        has_a = has_a && au >= al; has_b = has_b && bu >= bl;
        alo[c] = al; ahi[c] = au; blo[c] = bl; bhi[c] = bu;
      }
      if (has_a && has_b) {
        two = true;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          wc[c] = 0.5f * (alo[c] + ahi[c]);
          wh[c] = 0.5f * (ahi[c] - alo[c]) * 1.0001f + 1e-7f * fmaxf(fabsf(alo[c]), fabsf(ahi[c]));
          na = fmaxf(na, fmaxf(fabsf(alo[c]), fabsf(ahi[c])));
          wc2[c] = 0.5f * (blo[c] + bhi[c]);
          wh2[c] = 0.5f * (bhi[c] - blo[c]) * 1.0001f + 1e-7f * fmaxf(fabsf(blo[c]), fabsf(bhi[c]));
          nb = fmaxf(nb, fmaxf(fabsf(blo[c]), fabsf(bhi[c])));
        }
        wnorm = na * 1.0001f;
        wnorm2 = nb * 1.0001f;
      }
    }

    const float4 *src = p.planes + (size_t)(first_light + l) * origin_stride;
    // the buffer about to be refilled last held the tile before the previous
    // phase's final one; every thread left it at that phase's last barrier
    ring_sync();
    RtCursor cursor = rt_cursor_scene(src, p.n_tris);
    bool dedupe = false;
    if (GRID) {
      // the cube-map cells around this light that the block's shadow rays fall into
      for (int i = lane; i < (1 << RT_GRID_TABLE_LOG2); i += 32) s_table[i] = -1;
      for (int i = lane; i < RT_SEEN; i += 32) s_seen[i] = -1;
      if (lane == 0) s_ncells = 0;
      __syncwarp();
      const int cell_base = (GRID ? p.gx : (int)gridDim.x) * p.blocks_y + l * 6 * RT_GRID_FACE;
      int last = -2;
      float lb0 = 0.f, lb1 = 0.f, lc0 = 0.f, lc1 = 0.f;   // the last cell's bounds on its face plane
#pragma unroll(GRID ? 1 : 9)   // grid kernels: smaller code (their warps run out of step and miss in the instruction cache)
      for (int k = 0; k < 9; ++k) {
        if (!((active >> k) & 1u)) continue;
        const float gx = -xsub(Lx, xadd(cx, xmul(HT(k), RT_SDX(k))));
        const float gy = -xsub(Ly, xadd(cy, xmul(HT(k), RT_SDY(k))));
        const float gz = -xsub(Lz, xadd(cz, xmul(HT(k), dz)));
        if (last >= 0) {
          // Usually the same cell as the previous sample: four products instead of two divisions.
          // (A direction within rounding of a cell border may be counted to either side: every
          // list is built for its cell widened by 2 %.)
          const int face = last / RT_GRID_FACE, a = face >> 1;
          const float ga = a == 0 ? gx : (a == 1 ? gy : gz), gb = a == 0 ? gy : (a == 1 ? gz : gx),
                      gc = a == 0 ? gz : (a == 1 ? gx : gy);
          const float m = fabsf(ga);
          if ((ga < 0.0f) == ((face & 1) != 0) && m > 1e-30f && m < 1e30f && gb >= lb0 * m && gb < lb1 * m &&
              gc >= lc0 * m && gc < lc1 * m)
            continue;
        }
        const int cell = rt_grid_cell_of(gx, gy, gz);
        if (cell == last) continue;
        last = cell;
        if (cell >= 0) {
          const float cw = 2.0f / (float)RT_GRID_G;
          const int ci = cell % RT_GRID_G, cj = (cell / RT_GRID_G) % RT_GRID_G;
          lb0 = -1.0f + cw * (float)ci; lb1 = lb0 + cw;
          lc0 = -1.0f + cw * (float)cj; lc1 = lc0 + cw;
        }
        if (cell < 0) atomicAdd(&s_ncells, RT_GRID_MAX_CELLS + 1);   // no direction: stream the scene
        else rt_grid_mark(cell_base + cell, s_table, s_cells, &s_ncells);
      }
      __syncwarp();
      if (s_ncells <= RT_GRID_MAX_CELLS) cursor = rt_cursor_cells(s_cells, s_ncells);
      else if (!warp_active) cursor = rt_cursor_cells(s_cells, 0);
      dedupe = s_ncells > 1 && s_ncells <= RT_GRID_MAX_CELLS;
#ifdef RT_PROFILE_CLOCK
      prof_cells += (unsigned)s_ncells;
#endif
#ifdef RT_PROFILE_COUNTERS
      if (lane == 0) {
        if (s_ncells > RT_GRID_MAX_CELLS) atomicAdd(p.counters + 10, 1ull);
        else atomicAdd(p.counters + 11, (unsigned long long)s_ncells);
      }
#endif
    }
    RtItem item;
    bool have = rt_cursor_next<GRID, TILE>(p, cursor, item);
    if (issuer && have) rt_ring_issue<TILE>(ring, item);
    while (have) {
      const int buf = ring.issued & 1;
      ++ring.issued;
      ring_sync();
      RtItem next_item;
      const bool have_next = rt_cursor_next<GRID, TILE>(p, cursor, next_item);
      if (issuer && have_next) rt_ring_issue<TILE>(ring, next_item);
      mbar_wait(&bars[buf], (ring.phase_bits >> buf) & 1u);
      ring.phase_bits ^= 1u << buf;
      const float4 *T = ring.buf[0] + (size_t)buf * TILE * RT_REC_F4;
      const int *Tidx = ring.smem_idx + buf * TILE;
      const bool listed = GRID && item.idx != nullptr;
      const int base = item.base;
      const int cnt = warp_active ? item.cnt : 0;
#ifdef RT_PROFILE_COUNTERS
      if (issuer) atomicAdd(p.counters + 13, (unsigned long long)item.cnt);
#endif
#ifdef RT_PROFILE_CLOCK
      prof_recs += (unsigned)cnt;
#endif
      item = next_item;
      have = have_next;
      for (int r0 = 0; r0 < cnt; r0 += 32) {
        // ---- L0: one triangle per lane vs the warp's shadow-bundle box ----
        bool pass = false;
        if (r0 + lane < cnt) {
          const float4 q0 = T[(r0 + lane) * 3], q1 = T[(r0 + lane) * 3 + 1], q2 = T[(r0 + lane) * 3 + 2];
          const float Eg = q2.y * wnorm;
          const float nx = q0.x + q0.w + q1.z, ny = q0.y + q1.x + q1.w, nz = q0.z + q1.y + q2.x;
          const float mN = fmaf(nx, wc[0], fmaf(ny, wc[1], nz * wc[2])) +
                           fmaf(fabsf(nx), wh[0], fmaf(fabsf(ny), wh[1], fabsf(nz) * wh[2]));
          pass = rt_box_may_hit_light<GRID>(q0, q1, q2, wc, wh, Eg) && !(mN + 1.1f * Eg < q2.z);
          if (GRID && two && !pass) {
            const float Eg2 = q2.y * wnorm2;
            const float mN2 = fmaf(nx, wc2[0], fmaf(ny, wc2[1], nz * wc2[2])) +
                              fmaf(fabsf(nx), wh2[0], fmaf(fabsf(ny), wh2[1], fabsf(nz) * wh2[2]));
            pass = rt_box_may_hit_light<GRID>(q0, q1, q2, wc2, wh2, Eg2) && !(mN2 + 1.1f * Eg2 < q2.z);
          }
          if (GRID && pass && listed && dedupe) {
            // met in an earlier cell of this phase?  (open addressing; a full table only means
            // that the triangle is worked on again, which changes nothing)
            const int tri = Tidx[r0 + lane];
            unsigned hsh = ((unsigned)tri * 2654435761u) >> (32 - RT_SEEN_LOG2);
            for (int probe = 0; probe < 8; ++probe) {
              const int old = atomicCAS(s_seen + hsh, -1, tri);
              if (old == tri) { pass = false; break; }
              if (old == -1) break;
              hsh = (hsh + 1) & (RT_SEEN - 1);
            }
          }
        }
        unsigned mask = __ballot_sync(0xffffffffu, pass);
        // ---- L1: the pixel's own bundle box against every survivor ----
        unsigned mine = 0;
        while (mask) {
          const int j = __ffs(mask) - 1;
          mask &= mask - 1;
          const float4 q0 = T[(r0 + j) * 3], q1 = T[(r0 + j) * 3 + 1], q2 = T[(r0 + j) * 3 + 2];
          const float Eg = q2.y * pnorm;
          const float cu = fmaf(q0.x, pc[0], fmaf(q0.y, pc[1], q0.z * pc[2]));
          const float cv = fmaf(q0.w, pc[0], fmaf(q1.x, pc[1], q1.y * pc[2]));
          const float cw = fmaf(q1.z, pc[0], fmaf(q1.w, pc[1], q2.x * pc[2]));
          const float hu = fmaf(fabsf(q0.x), ph[0], fmaf(fabsf(q0.y), ph[1], fabsf(q0.z) * ph[2]));
          const float hv = fmaf(fabsf(q0.w), ph[0], fmaf(fabsf(q1.x), ph[1], fabsf(q1.y) * ph[2]));
          const float hw = fmaf(fabsf(q1.z), ph[0], fmaf(fabsf(q1.w), ph[1], fabsf(q2.x) * ph[2]));
          const float m3 = fminf(fminf(cu + hu, cv + hv), cw + hw);
          const float mN = (cu + cv + cw) + (hu + hv + hw);
          if (active) RT_PC(3);
          if ((active & ~occluded) && !((m3 < -Eg) || (mN + Eg < q2.z))) mine |= 1u << j;
#ifdef RT_PROFILE_CLOCK
          ++prof_l1;
#endif
        }
#ifdef RT_PROFILE_CLOCK
        prof_l2 += (unsigned)__popc(mine);
#endif
        // ---- L2 / EX: each lane walks its own candidates ----
        while (mine) {
          const int j = __ffs(mine) - 1;
          mine &= mine - 1;
          const unsigned todo = active & ~occluded;
          if (!todo) break;
          const int tri = listed ? Tidx[r0 + j] : base + r0 + j;
          const float4 q0 = T[(r0 + j) * 3], q1 = T[(r0 + j) * 3 + 1], q2 = T[(r0 + j) * 3 + 2];
          const float Eg = q2.y * pnorm;
          RT_PC(4);
          if (GRID) {
            // ---- L2 / EX: per shadow ray.  The grid kernels keep the reference's call inside the unrolled loop and
            //      no self-pair test: with the test below they measured 1.2-2.7 % slower on the 100 800-triangle box
            //      (B200, 1000 W power limit; their warps run out of step and the loop's code size costs more) ----
#pragma unroll
            for (int k = 0; k < 9; ++k) {
              if (!((todo >> k) & 1u) || ((occluded >> k) & 1u)) continue;
              const float px = xadd(cx, xmul(HT(k), RT_SDX(k))), py = xadd(cy, xmul(HT(k), RT_SDY(k))),
                          pz = xadd(cz, xmul(HT(k), dz));
              const float gx = -xsub(Lx, px), gy = -xsub(Ly, py), gz = -xsub(Lz, pz);
              const float mU = fmaf(q0.x, gx, fmaf(q0.y, gy, q0.z * gz));
              const float mV = fmaf(q0.w, gx, fmaf(q1.x, gy, q1.y * gz));
              const float mW = fmaf(q1.z, gx, fmaf(q1.w, gy, q2.x * gz));
              const float m3 = fminf(fminf(mU, mV), mW);
              const float mN = mU + mV + mW;
              RT_PC(5);
              if (m3 < -Eg || mN + Eg < q2.z) continue;          // definite miss / behind the start
              RT_PC(6);
              if (m3 >= Eg && mN - Eg >= q2.w && q2.z >= 1e-4f * mN) {
                occluded |= 1u << k;                              // definite occluder
                continue;
              }
              ++n_exact;
#ifdef RT_PROFILE_COUNTERS
              RT_PC(7);
              if (tri == HI(k)) RT_PC(8);
#endif
              if (rt_ex_shadow(p.geom, p.src, p.sph, tri, HI(k), px, py, pz, Lx, Ly, Lz)) occluded |= 1u << k;
            }
            continue;
          }
          // ---- L2: per shadow ray; what it cannot decide is left in `amb` ----
          unsigned amb = 0;
#pragma unroll
          for (int k = 0; k < 9; ++k) {
            if (!((todo >> k) & 1u) || ((occluded >> k) & 1u)) continue;
            const float px = xadd(cx, xmul(HT(k), RT_SDX(k))), py = xadd(cy, xmul(HT(k), RT_SDY(k))),
                        pz = xadd(cz, xmul(HT(k), dz));
            const float gx = -xsub(Lx, px), gy = -xsub(Ly, py), gz = -xsub(Lz, pz);
            const float mU = fmaf(q0.x, gx, fmaf(q0.y, gy, q0.z * gz));
            const float mV = fmaf(q0.w, gx, fmaf(q1.x, gy, q1.y * gz));
            const float mW = fmaf(q1.z, gx, fmaf(q1.w, gy, q2.x * gz));
            const float m3 = fminf(fminf(mU, mV), mW);
            const float mN = mU + mV + mW;
            RT_PC(5);
            if (m3 < -Eg || mN + Eg < q2.z) continue;          // definite miss / behind the start
            RT_PC(6);
            if (m3 >= Eg && mN - Eg >= q2.w && q2.z >= 1e-4f * mN) {
              occluded |= 1u << k;                              // definite occluder
              continue;
            }
            amb |= 1u << k;
          }
          // ---- the rays that start on this triangle: where rt_prep_planes_kernel knows the sign of the
          //      reference's D (self_D), Dt formed as rt_ex_shadow forms it decides the pair the way its early
          //      return does (|self_D| >= |D|): t < 0.  A loop without calls: the triangle's data stay in registers ----
          if (amb) {
            const float sD = p.self_D ? __ldg(p.self_D + (size_t)l * p.n_tris + tri) : 0.0f;
            const float4 g0 = __ldg(p.geom + 3 * tri), g1 = __ldg(p.geom + 3 * tri + 1);
            const float e2z = __ldg(&p.geom[3 * tri + 2].x);
            const float *n = p.src[tri].normal;
            const float n0 = __ldg(n), n1 = __ldg(n + 1), n2 = __ldg(n + 2);
            for (unsigned m = amb; m; m &= m - 1) {   // (sD tested inside: every load is issued at once)
              const int k = __ffs(m) - 1;
              if (sD == 0.0f || HI(k) != tri) continue;
              float px, py, pz;
              if (SAMPLES) { px = xadd(cx, xmul(HT(k), RT_SDX(k))); py = xadd(cy, xmul(HT(k), RT_SDY(k))); pz = xadd(cz, xmul(HT(k), dz)); }
              else rt_hit_point(cx, cy, cz, dxs[1], dys[1], dz, HT(k), k, px, py, pz);
              const float ox = xadd(px, xmul(n0, 0.00001f)), oy = xadd(py, xmul(n1, 0.00001f)),
                          oz = xadd(pz, xmul(n2, 0.00001f));                                    // :394
              const float Dt = xdet3(xsub(ox, g0.x), xsub(oy, g0.y), xsub(oz, g0.z), g0.w, g1.x, g1.y, g1.z, g1.w, e2z);
              if (((Dt < 0.0f) != (sD < 0.0f)) && fabsf(Dt) > 1e-20f * fabsf(sD)) amb &= ~(1u << k);
            }
          }
          // ---- EX: the reference arithmetic, one copy of the code outside the unrolled loop (instruction cache) ----
          while (amb) {
            const int k = __ffs(amb) - 1;
            amb &= amb - 1;
            float px, py, pz;
            if (SAMPLES) { px = xadd(cx, xmul(HT(k), RT_SDX(k))); py = xadd(cy, xmul(HT(k), RT_SDY(k))); pz = xadd(cz, xmul(HT(k), dz)); }
            else rt_hit_point(cx, cy, cz, dxs[1], dys[1], dz, HT(k), k, px, py, pz);
            ++n_exact;
#ifdef RT_PROFILE_COUNTERS
            RT_PC(7);
            if (tri == HI(k)) RT_PC(8);
#endif
            if (rt_ex_shadow(p.geom, p.src, p.sph, tri, HI(k), px, py, pz, Lx, Ly, Lz)) occluded |= 1u << k;
          }
        }
      }
    }

    // sphere occluders + the lighting tail of DirectLight, then (single light)
    // the pixelColour accumulation in the reference's order (:151-156)
#pragma unroll(GRID ? 1 : 9)   // grid kernels: smaller code (their warps run out of step and miss in the instruction cache)
    for (int k = 0; k < 9; ++k) {
      if (!((active >> k) & 1u)) continue;
      const float px = xadd(cx, xmul(HT(k), RT_SDX(k))), py = xadd(cy, xmul(HT(k), RT_SDY(k))),
                  pz = xadd(cz, xmul(HT(k), dz));
      const RtShade s = rt_ex_shade(p.src, p.sph, p.n_sph, HI(k), px, py, pz, Lx, Ly, Lz, p.lights[l][4],
                                    p.lights[l][5], p.lights[l][6], (occluded >> k) & 1u, 1);
      if (MULTI) {
        dl[(l * 9 + k) * 3 + 0] = s.pw[0]; dl[(l * 9 + k) * 3 + 1] = s.pw[1]; dl[(l * 9 + k) * 3 + 2] = s.pw[2];
      } else {
        PIX(0) = xadd(PIX(0), s.pw[0]); PIX(1) = xadd(PIX(1), s.pw[1]); PIX(2) = xadd(PIX(2), s.pw[2]);
        PIX(0) = xadd(PIX(0), xmul(s.col[0], 0.5f));
        PIX(1) = xadd(PIX(1), xmul(s.col[1], 0.5f));
        PIX(2) = xadd(PIX(2), xmul(s.col[2], 0.5f));
      }
    }
  }

  if (live) {
    if (MULTI || p.n_lights == 0) {
#pragma unroll
      for (int k = 0; k < 9; ++k) {
        if (!((active >> k) & 1u)) continue;
        if (MULTI)
          for (int l = 0; l < p.n_lights; ++l) {
            PIX(0) = xadd(PIX(0), dl[(l * 9 + k) * 3 + 0]);
            PIX(1) = xadd(PIX(1), dl[(l * 9 + k) * 3 + 1]);
            PIX(2) = xadd(PIX(2), dl[(l * 9 + k) * 3 + 2]);
          }
        const float px = xadd(cx, xmul(HT(k), RT_SDX(k))), py = xadd(cy, xmul(HT(k), RT_SDY(k))),
                    pz = xadd(cz, xmul(HT(k), dz));
        const RtShade s = rt_ex_shade(p.src, p.sph, 0, HI(k), px, py, pz, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0, 0);
        PIX(0) = xadd(PIX(0), xmul(s.col[0], 0.5f));
        PIX(1) = xadd(PIX(1), xmul(s.col[1], 0.5f));
        PIX(2) = xadd(PIX(2), xmul(s.col[2], 0.5f));
      }
    }
    if (!SAMPLES) {
      const float pix[3] = {PIX(0), PIX(1), PIX(2)};
      rt_store_pixel(p, PID, active != 0, pix);
    }
  }
  if (!SAMPLES) rt_count(p.counters + 0, (unsigned long long)__popc(active) * p.n_lights);
  }   // groups of samples
  if (SAMPLES) {
    if (live) {
      const float pix[3] = {PIX(0), PIX(1), PIX(2)};
      rt_store_pixel_n(p, PID, any_hit, pix, sp->n);
    }
    rt_count(p.counters + 0, (unsigned long long)n_hit * p.n_lights);
  }
  rt_count(p.counters + 1, (unsigned long long)n_exact);
  if (GRID && p.block_cost && lane == 0)   // what the next frame's plan is made from
    atomicMax(p.block_cost + s_cost_at[warp], (((unsigned)clock() - s_cost_t0[warp]) >> 8) * (s_split ? 8u : 1u));
#ifdef RT_PROFILE_COUNTERS
  if (live) for (int i = 0; i < 6; ++i) atomicAdd(p.counters + 2 + i, (unsigned long long)prof_cnt[i + (i >= 2 ? 1 : 0)]);
  if (live) { atomicAdd(p.counters + 8, (unsigned long long)prof_cnt[8]); atomicAdd(p.counters + 14, (unsigned long long)prof_cnt[7]); }
  // diagnostic build only: the depth plane carries this pixel's shadow L1 test count, the index plane its exact evaluations
  if (live && p.depth) p.depth[PID] = (float)prof_cnt[3];
  if (live && p.index) p.index[PID] = (int)n_exact;
#endif
#ifdef RT_PROFILE_CLOCK
  // depth plane: cycles of this warp; index plane: records its shadow phases streamed (low 20 bits), cells walked (high bits);
  // rgb plane: shadow-phase L0 survivors this lane tested, candidates it kept, exact evaluations
  if (live && p.depth) p.depth[PID] = (float)(clock64() - prof_t0);
  if (live && p.index) p.index[PID] = (int)(min(prof_recs, 0xfffffu) | (min(prof_cells, 2047u) << 20));
  if (live && p.rgb) { p.rgb[3 * PID] = (float)prof_l1; p.rgb[3 * PID + 1] = (float)prof_l2; p.rgb[3 * PID + 2] = (float)(n_exact - prof_ex0); }
#endif
}

template <bool MULTI, bool GRID>
__global__ void __launch_bounds__(RT_THREADS, GRID ? 2 : RT_MIN_BLOCKS) rt_filtered_kernel(const __grid_constant__ RtKParams p) {
  rt_filtered_body<MULTI, GRID, false>(p, nullptr);
}
// Batched views: grid (x, y) = the 16x16 pixel blocks of one whole frame, z = view; p.row0 = 0, p.row1 = H, no interleave.
template <bool MULTI>
__global__ void __launch_bounds__(RT_THREADS, RT_MIN_BLOCKS) rt_filtered_views_kernel(const __grid_constant__ RtKParams p,
                                                                                      const __grid_constant__ RtViewsParams v) {
  rt_filtered_body<MULTI, false, true>(p, &v);
}
// The caller's sample pattern (render_raytrace_samples): launched as rt_filtered_kernel, with the table in s.
template <bool MULTI, bool GRID>
__global__ void __launch_bounds__(RT_THREADS, GRID ? 2 : RT_MIN_BLOCKS)
    rt_filtered_samples_kernel(const __grid_constant__ RtKParams p, const __grid_constant__ RtSamplesParams s) {
  rt_filtered_body<MULTI, GRID, false, true>(p, nullptr, &s);
}

int rt_launch_filtered(b200_ctx *ctx, const RtFrame &f, RtKParams &p, const RtSamplesParams *sp = nullptr);
