// rt_lattice_kernel: the scene-streaming kernel for frames whose sample rays form a lattice.
//
// A pixel's nine samples are (dir0 + 0.5 (kx - 1), dir1 + 0.5 (ky - 1), f) (skeleton.cpp:134-137).  When dir0
// depends on u only, dir1 on v only, and dir0(u) + 0.5 has the bits of dir0(u + 1) - 0.5 (and likewise in v),
// sample kx = 2 of pixel u IS sample kx = 0 of pixel u + 1: everything the reference derives from a sample
// (closest hit, shadow ray, DirectLight, colour) is a function of the camera position and that direction, so
// it is computed once.  A 16 x 16 pixel block then needs the 33 x 33 points of a half-pixel lattice instead of
// 256 x 9 rays; point (i, j) is sample (i - 2a, j - 2b) of block pixel (a, b).  rt_launch_filtered checks the
// condition on the host (rt_lattice_exact) per launch; every other frame runs rt_filtered_kernel.
//
// Threads and warps sit on the pixels as in rt_filtered_body (8 warps of 8 x 4 pixels).  Thread (a, b) traces
// the points (2a + di, 2b + dj), di, dj in {0, 1} (slots 0-3, slot 3 = its centre sample), and at most one of
// the 65 points of column 32 / row 32 (slot 4, rt_lat_extra).  Points no live pixel uses are not traced.  The
// primary and shadow phases are those of rt_filtered_body over the slots; each hit point's shade goes to
// shared memory under its lattice index, and after a block barrier every pixel sums its nine samples in the
// reference's order (:151-156).
#pragma once

constexpr int RT_LAT_N = 33;                        // lattice points per block edge
constexpr int RT_LAT_PTS = RT_LAT_N * RT_LAT_N;
constexpr int RT_LAT_SLOTS = 5;
// ring, then t / distance / index / ray length per (slot, thread), then pw[3] / col[3] per lattice point, then hit flags
constexpr size_t RT_LAT_SMEM = 2 * (size_t)RT_TILE * RT_REC_F4 * sizeof(float4) +
                               4 * (size_t)RT_LAT_SLOTS * RT_THREADS * sizeof(float) +
                               6 * (size_t)RT_LAT_PTS * sizeof(float) + ((RT_LAT_PTS + 3) & ~3);

// The point of column 32 or row 32 that (warp, lane) traces in slot 4: i | j << 8, or -1.  Row 32 goes to the two
// bottom pixel rows of the bottom warps, column 32 to the two right pixel columns of the right warps; the five
// points (32, 28..32) left over in the corner warp go to lanes near them.  Every point is traced exactly once.
__device__ __forceinline__ int rt_lat_extra(int warp, int lane) {
  const int cx = warp & 1, ry = warp >> 1, la = lane & 7, lb = lane >> 3;
  if (ry == 3 && lb >= 2) return (16 * cx + 2 * la + (lb == 2 ? 1 : 0)) | (32 << 8);
  if (cx == 1 && la >= 6) return 32 | ((8 * ry + 2 * lb + la - 6) << 8);
  if (cx == 1 && ry == 3 && la >= 3) {
    const int m = 2 * (la - 3) + lb;
    return m <= 4 ? 32 | ((28 + m) << 8) : -1;
  }
  return -1;
}

// Block pixel whose sample gives lattice column (row) i, and that sample's offset: i = 0 is sample 0 of pixel 0,
// odd i the centre sample of pixel (i - 1) / 2, other even i sample 2 of pixel i / 2 - 1.  A live pixel that uses
// point i is never to the left of rt_lat_pix(i): the point is needed exactly when that pixel is live.
__device__ __forceinline__ int rt_lat_pix(int i) { return max(i - 1, 0) >> 1; }
__device__ __forceinline__ float rt_lat_off(int i) {
  const int kx = i == 0 ? 0 : 2 - (i & 1);
  return xmul(0.5f, (float)(kx - 1));
}

__global__ void __launch_bounds__(RT_THREADS, RT_MIN_BLOCKS) rt_lattice_kernel(const __grid_constant__ RtKParams p) {
  extern __shared__ __align__(128) float4 tile_smem[];
  __shared__ __align__(8) uint64_t bars[2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int a = (warp & 1) * 8 + (lane & 7), b = (warp >> 1) * 4 + (lane >> 3);   // pixel of the block
  const int u0 = (int)blockIdx.x * 16;
  const int v0 = p.row0 + ((int)blockIdx.y * p.il_n + p.il_r) * 16;             // interleaved launches: as rt_filtered_body
  const int u = u0 + a, v = v0 + b;
  const bool live = (u < p.W) && (v < p.row1);
  const size_t pid = (size_t)v * p.W + u;
  const float *R = p.R;
  const float focal = p.focal, dz = focal;
  const float cx = p.cam[0], cy = p.cam[1], cz = p.cam[2];

  if (threadIdx.x == 0) {
    mbar_init(&bars[0], 1); mbar_init(&bars[1], 1);
    mbar_fence_init();
  }
  __syncthreads();
  RtRing ring;
  ring.smem = tile_smem; ring.bars = bars; ring.phase_bits = 0; ring.issued = 0; ring.smem_idx = nullptr;
  float *s_ht = reinterpret_cast<float *>(tile_smem + 2 * RT_TILE * RT_REC_F4);
  float *s_hd = s_ht + RT_LAT_SLOTS * RT_THREADS;
  int *s_hi = reinterpret_cast<int *>(s_hd + RT_LAT_SLOTS * RT_THREADS);
  float *s_len = s_hd + 2 * RT_LAT_SLOTS * RT_THREADS;
  float *s_shade = s_len + RT_LAT_SLOTS * RT_THREADS;   // [c][point]: pw 0-2, col 3-5
  unsigned char *s_hit = reinterpret_cast<unsigned char *>(s_shade + 6 * RT_LAT_PTS);
#define LT(s) s_ht[(s) * RT_THREADS + threadIdx.x]
#define LD(s) s_hd[(s) * RT_THREADS + threadIdx.x]
#define LI(s) s_hi[(s) * RT_THREADS + threadIdx.x]
#define LLEN(s) s_len[(s) * RT_THREADS + threadIdx.x]

  // ---- the thread's lattice points and their directions (the kernel's own expression for dir0 / dir1) ----
  const int nu = p.W - u0, nv = p.row1 - v0;          // live pixel columns / rows of the block, from the left / top
  const int ex = rt_lat_extra(warp, lane);
  const int ei = ex & 0xff, ej = ex >> 8;
  const float y_own = (float)(v - p.H / 2), x_own = (float)(u - p.W / 2);
  auto dir_x = [&](int i) {   // sample x of lattice column i (independent of y: R[4] == 0)
    const float x = (float)(u0 + rt_lat_pix(i) - p.W / 2);
    return xadd(xadd(xadd(xmul(R[0], x), xmul(R[4], y_own)), xadd(xmul(R[8], focal), xmul(R[12], 1.0f))), rt_lat_off(i));
  };
  auto dir_y = [&](int j) {
    const float y = (float)(v0 + rt_lat_pix(j) - p.H / 2);
    return xadd(xadd(xadd(xmul(R[1], x_own), xmul(R[5], y)), xadd(xmul(R[9], focal), xmul(R[13], 1.0f))), rt_lat_off(j));
  };
  const float dxA = dir_x(2 * a), dxB = dir_x(2 * a + 1), dyA = dir_y(2 * b), dyB = dir_y(2 * b + 1);
  const float dxE = ex >= 0 ? dir_x(ei) : 0.f, dyE = ex >= 0 ? dir_y(ej) : 0.f;
  unsigned valid = 0;   // slots whose point a live pixel uses
#pragma unroll
  for (int s = 0; s < 4; ++s)
    if (rt_lat_pix(2 * a + (s & 1)) < nu && rt_lat_pix(2 * b + (s >> 1)) < nv) valid |= 1u << s;
  if (ex >= 0 && rt_lat_pix(ei) < nu && rt_lat_pix(ej) < nv) valid |= 1u << 4;
#define SDX(s) ((s) == 4 ? dxE : (((s) & 1) ? dxB : dxA))
#define SDY(s) ((s) == 4 ? dyE : (((s) >> 1) & 1 ? dyB : dyA))
#define SPT(s) ((s) == 4 ? ej * RT_LAT_N + ei : (2 * b + ((s) >> 1)) * RT_LAT_N + 2 * a + ((s) & 1))

  float llo0 = INFINITY, lhi0 = -INFINITY, llo1 = INFINITY, lhi1 = -INFINITY;   // the thread's bundle box
#pragma unroll
  for (int s = 0; s < RT_LAT_SLOTS; ++s) {
    LT(s) = 0.f; LD(s) = FLT_MAX; LI(s) = 0;
    LLEN(s) = xsqrt(xdot3(SDX(s), SDY(s), dz, SDX(s), SDY(s), dz));
    if ((valid >> s) & 1u) {
      llo0 = fminf(llo0, SDX(s)); lhi0 = fmaxf(lhi0, SDX(s));
      llo1 = fminf(llo1, SDY(s)); lhi1 = fmaxf(lhi1, SDY(s));
    }
  }
  unsigned n_exact = 0;
  const float4 *T0 = ring.smem, *T1 = ring.smem + RT_TILE * RT_REC_F4;

  // ============================ primary rays ============================
  {
    const float lo0 = warp_min(llo0), hi0 = warp_max(lhi0), lo1 = warp_min(llo1), hi1 = warp_max(lhi1);
    const bool warp_live = hi0 >= lo0;
    const float wc0 = 0.5f * (lo0 + hi0), wc1 = 0.5f * (lo1 + hi1);
    const float wh0 = 0.5f * (hi0 - lo0) * 1.0001f + 1e-3f, wh1 = 0.5f * (hi1 - lo1) * 1.0001f + 1e-3f;
    const float lc0 = 0.5f * (llo0 + lhi0), lc1 = 0.5f * (llo1 + lhi1);
    const float lh0 = 0.5f * (lhi0 - llo0) * 1.0001f + 1e-3f, lh1 = 0.5f * (lhi1 - llo1) * 1.0001f + 1e-3f;

    RtCursor cursor = rt_cursor_scene(p.planes, p.n_tris);
    RtItem item;
    bool have = rt_cursor_next<false, RT_TILE>(p, cursor, item);
    if (threadIdx.x == 0 && have) rt_ring_issue<RT_TILE>(ring, item);
    while (have) {
      const int buf = ring.issued & 1;
      ++ring.issued;
      __syncthreads();   // everyone is done with the other buffer: refill it
      RtItem next_item;
      const bool have_next = rt_cursor_next<false, RT_TILE>(p, cursor, next_item);
      if (threadIdx.x == 0 && have_next) rt_ring_issue<RT_TILE>(ring, next_item);
      mbar_wait(&bars[buf], (ring.phase_bits >> buf) & 1u);
      ring.phase_bits ^= 1u << buf;
      const float4 *T = buf ? T1 : T0;
      const int base = item.base;
      const int cnt = warp_live ? item.cnt : 0;
#ifdef RT_PROFILE_COUNTERS
      if (threadIdx.x == 0) atomicAdd(p.counters + 12, (unsigned long long)item.cnt);
#endif
      item = next_item;
      have = have_next;
      for (int r0 = 0; r0 < cnt; r0 += 32) {
        // ---- L0: one triangle per lane vs the warp's bundle box ----
        bool pass = false;
        if (r0 + lane < cnt) {
          const float4 q0 = T[(r0 + lane) * 3], q1 = T[(r0 + lane) * 3 + 1], q2 = T[(r0 + lane) * 3 + 2];
          pass = rt_box_may_hit_cam<false>(q0, q1, q2, wc0, wc1, wh0, wh1);
        }
        unsigned mask = __ballot_sync(0xffffffffu, pass);
        // ---- L1: every lane tests its own bundle box against every survivor ----
        unsigned mine = 0;
        while (mask) {
          const int j = __ffs(mask) - 1;
          mask &= mask - 1;
          const float4 q0 = T[(r0 + j) * 3], q1 = T[(r0 + j) * 3 + 1], q2 = T[(r0 + j) * 3 + 2];
          if (valid && rt_box_may_hit_cam<false>(q0, q1, q2, lc0, lc1, lh0, lh1)) mine |= 1u << j;
        }
        // ---- L2 / EX: each lane walks its own candidates, per lattice point ----
        while (mine) {
          const int j = __ffs(mine) - 1;
          mine &= mine - 1;
          const int tri = base + r0 + j;
          const float4 q0 = T[(r0 + j) * 3], q1 = T[(r0 + j) * 3 + 1], q2 = T[(r0 + j) * 3 + 2];
          const float E = q2.y, dt_lo = q2.z;
#pragma unroll
          for (int s = 0; s < RT_LAT_SLOTS; ++s) {
            if (!((valid >> s) & 1u)) continue;
            const float dx = SDX(s), dy = SDY(s);
            const float mU = fmaf(q0.x, dx, fmaf(q0.y, dy, q0.z));
            const float mV = fmaf(q0.w, dx, fmaf(q1.x, dy, q1.y));
            const float mW = fmaf(q1.z, dx, fmaf(q1.w, dy, q2.x));
            const float m3 = fminf(fminf(mU, mV), mW);
            if (m3 >= -E) {
              const float mN = mU + mV + mW;
              RtHit hb;
              hb.dist = LD(s);
              const bool farther = (mN > E) && (dt_lo * LLEN(s) > hb.dist * (mN + E));
              if (!farther) {
                ++n_exact;
                hb.t = LT(s); hb.idx = LI(s);
                const RtHit nb = rt_ex_primary(p.geom, p.dt_cam, cx, cy, cz, tri, m3 >= E ? 1 : 0, dx, dy, dz, LLEN(s), hb);
                if (nb.idx != hb.idx || nb.dist != hb.dist) { LT(s) = nb.t; LD(s) = nb.dist; LI(s) = nb.idx; }
              }
            }
          }
        }
      }
    }
  }

  // spheres (skeleton.cpp:341-355), per lattice point in ascending sphere order
  for (int sp = 0; sp < p.n_sph && valid; ++sp) {
    // Bundle pre-test as in rt_filtered_body, over the thread's box of directions (centre c, half-widths h,
    // widened by the rounding of c): an upper bound of q + tolerance (rt_sphere_may_hit).  Negative: no point hits.
    {
      const float Lx = cx - __ldg(&p.sph[sp].centre[0]), Ly = cy - __ldg(&p.sph[sp].centre[1]),
                  Lz = cz - __ldg(&p.sph[sp].centre[2]);
      const float r2 = __ldg(&p.sph[sp].radius_squared);
      const float LL = fmaf(Lx, Lx, fmaf(Ly, Ly, Lz * Lz)), c = LL - r2;
      if (c > 0.0f) {                        // camera outside the sphere
        const float c0 = 0.5f * (llo0 + lhi0), c1 = 0.5f * (llo1 + lhi1);
        const float h0 = 0.5f * (lhi0 - llo0) * 1.0001f + 1e-6f * fabsf(c0) + 2e-4f;
        const float h1 = 0.5f * (lhi1 - llo1) * 1.0001f + 1e-6f * fabsf(c1) + 2e-4f;
        const float dL = fabsf(fmaf(c0, Lx, fmaf(c1, Ly, dz * Lz))) + h0 * fabsf(Lx) + h1 * fabsf(Ly);
        const float a_max = dL * dL * 1.00001f;
        const float ax0 = fmaxf(fabsf(c0) - h0, 0.0f), ay0 = fmaxf(fabsf(c1) - h1, 0.0f);
        const float ax1 = fabsf(c0) + h0, ay1 = fabsf(c1) + h1;
        const float dd_min = fmaf(ax0, ax0, fmaf(ay0, ay0, dz * dz)) * 0.99999f;
        const float dd_max = fmaf(ax1, ax1, fmaf(ay1, ay1, dz * dz)) * 1.00001f;
        if (a_max - dd_min * c < -1.001e-4f * (a_max + dd_max * (LL + r2))) continue;
      }
    }
#pragma unroll
    for (int s = 0; s < RT_LAT_SLOTS; ++s) {
      if (!((valid >> s) & 1u)) continue;
      const float dx = SDX(s), dy = SDY(s);
      if (!rt_sphere_may_hit(p.sph[sp], cx, cy, cz, dx, dy, dz)) continue;
      const RtSphT h = rt_ex_sphere(p.sph + sp, cx, cy, cz, dx, dy, dz);
      if (h.hit && h.t < LD(s)) { LT(s) = h.t; LD(s) = h.t; LI(s) = -1 - sp; }
    }
  }
  unsigned active = 0;
#pragma unroll
  for (int s = 0; s < RT_LAT_SLOTS; ++s)
    if (((valid >> s) & 1u) && LD(s) < FLT_MAX) active |= 1u << s;
  if (live) {   // slot 3 is the pixel's centre sample
    const bool hit3 = (active >> 3) & 1u;
    if (p.depth) p.depth[pid] = hit3 ? LD(3) : INFINITY;
    if (p.index) p.index[pid] = hit3 ? LI(3) : INT32_MIN;
  }

  // ============================ shadow rays (at most one light) ============================
  unsigned occluded = 0;
  const float Lx = p.lights[0][0], Ly = p.lights[0][1], Lz = p.lights[0][2];
  if (p.n_lights > 0) {
    // g = hit - light per point; boxes of the thread's and the warp's bundles
    float glo[3] = {INFINITY, INFINITY, INFINITY}, ghi[3] = {-INFINITY, -INFINITY, -INFINITY};
#pragma unroll
    for (int s = 0; s < RT_LAT_SLOTS; ++s) {
      if ((active >> s) & 1u) {
        const float gx = -xsub(Lx, xadd(cx, xmul(LT(s), SDX(s))));
        const float gy = -xsub(Ly, xadd(cy, xmul(LT(s), SDY(s))));
        const float gz = -xsub(Lz, xadd(cz, xmul(LT(s), dz)));
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
    const float wnorm = warp_max(pnorm) * 1.0001f;
    pnorm *= 1.0001f;
    const bool warp_active = __ballot_sync(0xffffffffu, active != 0) != 0;

    // the buffer about to be refilled last held the primary phase's next-to-last tile; every thread left it at
    // that phase's last barrier
    __syncthreads();
    RtCursor cursor = rt_cursor_scene(p.planes + (size_t)((p.n_tris + RT_TILE - 1) / RT_TILE) * RT_TILE * RT_REC_F4, p.n_tris);
    RtItem item;
    bool have = rt_cursor_next<false, RT_TILE>(p, cursor, item);
    if (threadIdx.x == 0 && have) rt_ring_issue<RT_TILE>(ring, item);
    while (have) {
      const int buf = ring.issued & 1;
      ++ring.issued;
      __syncthreads();
      RtItem next_item;
      const bool have_next = rt_cursor_next<false, RT_TILE>(p, cursor, next_item);
      if (threadIdx.x == 0 && have_next) rt_ring_issue<RT_TILE>(ring, next_item);
      mbar_wait(&bars[buf], (ring.phase_bits >> buf) & 1u);
      ring.phase_bits ^= 1u << buf;
      const float4 *T = buf ? T1 : T0;
      const int base = item.base;
      const int cnt = warp_active ? item.cnt : 0;
#ifdef RT_PROFILE_COUNTERS
      if (threadIdx.x == 0) atomicAdd(p.counters + 13, (unsigned long long)item.cnt);
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
          pass = rt_box_may_hit_light<false>(q0, q1, q2, wc, wh, Eg) && !(mN + 1.1f * Eg < q2.z);
        }
        unsigned mask = __ballot_sync(0xffffffffu, pass);
        // ---- L1: the thread's own bundle box against every survivor ----
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
          if ((active & ~occluded) && !((m3 < -Eg) || (mN + Eg < q2.z))) mine |= 1u << j;
        }
        // ---- L2 / EX: each lane walks its own candidates ----
        while (mine) {
          const int j = __ffs(mine) - 1;
          mine &= mine - 1;
          const unsigned todo = active & ~occluded;
          if (!todo) break;
          const int tri = base + r0 + j;
          const float4 q0 = T[(r0 + j) * 3], q1 = T[(r0 + j) * 3 + 1], q2 = T[(r0 + j) * 3 + 2];
          const float Eg = q2.y * pnorm;
          // ---- L2: per shadow ray; what it cannot decide is left in `amb` ----
          unsigned amb = 0;
#pragma unroll
          for (int s = 0; s < RT_LAT_SLOTS; ++s) {
            if (!((todo >> s) & 1u)) continue;
            const float px = xadd(cx, xmul(LT(s), SDX(s))), py = xadd(cy, xmul(LT(s), SDY(s))),
                        pz = xadd(cz, xmul(LT(s), dz));
            const float gx = -xsub(Lx, px), gy = -xsub(Ly, py), gz = -xsub(Lz, pz);
            const float mU = fmaf(q0.x, gx, fmaf(q0.y, gy, q0.z * gz));
            const float mV = fmaf(q0.w, gx, fmaf(q1.x, gy, q1.y * gz));
            const float mW = fmaf(q1.z, gx, fmaf(q1.w, gy, q2.x * gz));
            const float m3 = fminf(fminf(mU, mV), mW);
            const float mN = mU + mV + mW;
            if (m3 < -Eg || mN + Eg < q2.z) continue;          // definite miss / behind the start
            if (m3 >= Eg && mN - Eg >= q2.w && q2.z >= 1e-4f * mN) {
              occluded |= 1u << s;                              // definite occluder
              continue;
            }
            amb |= 1u << s;
          }
          // ---- the rays that start on this triangle: decided from self_D as in rt_filtered_body ----
          if (amb) {
            const float sD = p.self_D ? __ldg(p.self_D + tri) : 0.0f;
            const float4 g0 = __ldg(p.geom + 3 * tri), g1 = __ldg(p.geom + 3 * tri + 1);
            const float e2z = __ldg(&p.geom[3 * tri + 2].x);
            const float *n = p.src[tri].normal;
            const float n0 = __ldg(n), n1 = __ldg(n + 1), n2 = __ldg(n + 2);
            for (unsigned m = amb; m; m &= m - 1) {
              const int s = __ffs(m) - 1;
              if (sD == 0.0f || LI(s) != tri) continue;
              const float px = xadd(cx, xmul(LT(s), SDX(s))), py = xadd(cy, xmul(LT(s), SDY(s))),
                          pz = xadd(cz, xmul(LT(s), dz));
              const float ox = xadd(px, xmul(n0, 0.00001f)), oy = xadd(py, xmul(n1, 0.00001f)),
                          oz = xadd(pz, xmul(n2, 0.00001f));                                    // :394
              const float Dt = xdet3(xsub(ox, g0.x), xsub(oy, g0.y), xsub(oz, g0.z), g0.w, g1.x, g1.y, g1.z, g1.w, e2z);
              if (((Dt < 0.0f) != (sD < 0.0f)) && fabsf(Dt) > 1e-20f * fabsf(sD)) amb &= ~(1u << s);
            }
          }
          // ---- EX: the reference arithmetic, one copy of the code outside the unrolled loop ----
          while (amb) {
            const int s = __ffs(amb) - 1;
            amb &= amb - 1;
            const float px = xadd(cx, xmul(LT(s), SDX(s))), py = xadd(cy, xmul(LT(s), SDY(s))),
                        pz = xadd(cz, xmul(LT(s), dz));
            ++n_exact;
            if (rt_ex_shadow(p.geom, p.src, p.sph, tri, LI(s), px, py, pz, Lx, Ly, Lz)) occluded |= 1u << s;
          }
        }
      }
    }
  }

  // ---- sphere occluders + the lighting tail of DirectLight, and the surface colour, per hit point ----
#pragma unroll
  for (int s = 0; s < RT_LAT_SLOTS; ++s)
    if ((valid >> s) & 1u) s_hit[SPT(s)] = (active >> s) & 1u;
  for (unsigned m = active; m; m &= m - 1) {
    const int s = __ffs(m) - 1;
    const float px = xadd(cx, xmul(LT(s), SDX(s))), py = xadd(cy, xmul(LT(s), SDY(s))), pz = xadd(cz, xmul(LT(s), dz));
    const RtShade o = rt_ex_shade(p.src, p.sph, p.n_sph, LI(s), px, py, pz, Lx, Ly, Lz, p.lights[0][4], p.lights[0][5],
                                  p.lights[0][6], (occluded >> s) & 1u, p.n_lights > 0);
    const int pt = SPT(s);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      s_shade[c * RT_LAT_PTS + pt] = o.pw[c];
      s_shade[(3 + c) * RT_LAT_PTS + pt] = o.col[c];
    }
  }
  __syncthreads();

  // ---- each pixel sums its nine samples in the reference's order (:151-156) ----
  unsigned n_hit = 0;
  if (live) {
    float pix[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      const int pt = (2 * b + k % 3) * RT_LAT_N + 2 * a + k / 3;
      if (!s_hit[pt]) continue;
      ++n_hit;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        if (p.n_lights > 0) pix[c] = xadd(pix[c], s_shade[c * RT_LAT_PTS + pt]);
        pix[c] = xadd(pix[c], xmul(s_shade[(3 + c) * RT_LAT_PTS + pt], 0.5f));
      }
    }
    rt_store_pixel(p, pid, n_hit != 0, pix);
  }
  // the reference's counts: one shadow ray per hit sample of every pixel, shared points counted once per pixel
  rt_count(p.counters + 0, (unsigned long long)n_hit * p.n_lights);
  rt_count(p.counters + 1, (unsigned long long)n_exact);
#undef LT
#undef LD
#undef LI
#undef LLEN
#undef SDX
#undef SDY
#undef SPT
}
