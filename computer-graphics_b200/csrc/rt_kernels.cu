// Raytracer hot path on sm_100a: replaces Draw -> ClosestIntersection ->
// DirectLight of raytracer/Source/skeleton.cpp:104-169, 263-363, 366-415.
//
// Two kernels produce bit-identical frames:
//   rt_bruteforce_kernel  the reference arithmetic on every (ray, primitive)
//                         pair; the on-device cross-check.
//   rt_filtered_kernel    (rt_filtered.cuh) the production kernel: conservative
//                         edge-function filters decide almost every pair, the
//                         reference arithmetic runs only where it can matter.
//   rt_lattice_kernel     (rt_lattice_kernel.cuh) the same filters for frames whose
//                         sample rays form a half-pixel lattice: each shared sample
//                         ray is traced once per 16x16 pixel block.
// Frames with the caller's own sample offsets (render_raytrace_samples) run the *_samples_kernel instantiations
// of the filtered and brute-force bodies, never the lattice kernel.
#include "rt_exact.cuh"
#include "rt_filtered.cuh"
#include "rt_lattice_kernel.cuh"
#include "rt_grid.cuh"

// ------------------------------------------------------------------------------
// scene preparation: v0 / e1 / e2 per triangle (skeleton.cpp:283-284)
// ------------------------------------------------------------------------------
// bounds (optional): [0] max |vertex coordinate|, [1] max |normal component| capped at 1e30 (NaN / inf
// count as 1e30), as bit patterns of non-negative floats -- what rt_upload_scene's host loop computes
// for small scenes, here for large ones (100 800 triangles took 2.8 ms on the host per upload).
__global__ void rt_prep_geom_kernel(const rt_triangle *__restrict__ src, int n, float4 *__restrict__ geom,
                                    unsigned *__restrict__ bounds) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  float m = 0.f, nm = 0.f;
  if (i < n) {
    const rt_triangle t = src[i];
    float4 g0, g1, g2;
    g0.x = t.v0[0]; g0.y = t.v0[1]; g0.z = t.v0[2];
    g0.w = xsub(t.v1[0], t.v0[0]);
    g1.x = xsub(t.v1[1], t.v0[1]);
    g1.y = xsub(t.v1[2], t.v0[2]);
    g1.z = xsub(t.v2[0], t.v0[0]);
    g1.w = xsub(t.v2[1], t.v0[1]);
    g2.x = xsub(t.v2[2], t.v0[2]);
    g2.y = g2.z = g2.w = 0.f;
    geom[3 * i + 0] = g0;
    geom[3 * i + 1] = g1;
    geom[3 * i + 2] = g2;
    if (bounds) {
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        m = fmaxf(m, fmaxf(fabsf(t.v0[k]), fmaxf(fabsf(t.v1[k]), fabsf(t.v2[k]))));   // fmaxf drops NaN, like the host's
        const float a = fabsf(t.normal[k]);
        nm = fmaxf(nm, a <= 1e30f ? a : 1e30f);
      }
    }
  }
  if (bounds) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
      nm = fmaxf(nm, __shfl_xor_sync(0xffffffffu, nm, o));
    }
    if ((threadIdx.x & 31) == 0) {
      atomicMax(bounds, __float_as_uint(m));
      atomicMax(bounds + 1, __float_as_uint(nm));
    }
  }
}

// ------------------------------------------------------------------------------
// brute force, reference arithmetic everywhere
// ------------------------------------------------------------------------------
// SAMPLES: the caller's sample table sp (render_raytrace_samples) instead of the 3x3 grid.
template <bool SAMPLES>
__device__ __forceinline__ void rt_bruteforce_body(const RtKParams &p, const RtSamplesParams *sp) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // each warp owns an 8x4 pixel patch; a 128-thread block covers 16x8 pixels
  const int u = blockIdx.x * 16 + (warp & 1) * 8 + (lane & 7);
  const int v = p.row0 + ((blockIdx.y >> 1) * p.il_n + p.il_r) * 16 + (blockIdx.y & 1) * 8 + (warp >> 1) * 4 + (lane >> 3);
  unsigned long long n_shadow = 0;
  if (u < p.W && v < p.row1) {
    // dir = R * vec4(u - W/2, v - H/2, f, 1)   (skeleton.cpp:126-128)
    const float x = (float)(u - p.W / 2), y = (float)(v - p.H / 2);
    const float dir0 = xadd(xadd(xmul(p.R[0], x), xmul(p.R[4], y)), xadd(xmul(p.R[8], p.focal), xmul(p.R[12], 1.0f)));
    const float dir1 = xadd(xadd(xmul(p.R[1], x), xmul(p.R[5], y)), xadd(xmul(p.R[9], p.focal), xmul(p.R[13], 1.0f)));
    float pix[3] = {0.f, 0.f, 0.f};
    bool valid = false;
    const size_t pid = (size_t)v * p.W + u;
    // (SAMPLES: one loop over the table, i = 0 and j = k)
    for (int i = SAMPLES ? 0 : -1; i <= (SAMPLES ? 0 : 1); ++i) {
      for (int j = SAMPLES ? 0 : -1; j <= (SAMPLES ? sp->n - 1 : 1); ++j) {
        const float dx = SAMPLES ? xadd(dir0, sp->off[2 * j]) : xadd(dir0, xmul(0.5f, (float)i));   // :137
        const float dy = SAMPLES ? xadd(dir1, sp->off[2 * j + 1]) : xadd(dir1, xmul(0.5f, (float)j));
        const float dz = p.focal;
        const RtHit h = rt_closest_bruteforce(p, p.cam[0], p.cam[1], p.cam[2], dx, dy, dz);
        const bool hit = h.dist < FLT_MAX;
        if (SAMPLES ? j == sp->depth_sample : (i == 0 && j == 0)) {
          if (p.depth) p.depth[pid] = hit ? h.dist : INFINITY;
          if (p.index) p.index[pid] = hit ? h.idx : INT32_MIN;
        }
        if (!hit) continue;
        valid = true;
        // position = start + vec4(t * dir3, 0)   (:326 / :345)
        const float px = xadd(p.cam[0], xmul(h.t, dx));
        const float py = xadd(p.cam[1], xmul(h.t, dy));
        const float pz = xadd(p.cam[2], xmul(h.t, dz));
        float col[3], nx, ny, nz;
        rt_surface(p, h.idx, px, py, pz, col, nx, ny, nz);
        for (int l = 0; l < p.n_lights; ++l) {
          // DirectLight (:366-415)
          const float rx = xsub(p.lights[l][0], px), ry = xsub(p.lights[l][1], py), rz = xsub(p.lights[l][2], pz);
          const float r_mag = rt_exact_rmag(rx, ry, rz);
          const float ox = xadd(px, xmul(nx, 0.00001f)), oy = xadd(py, xmul(ny, 0.00001f)),
                      oz = xadd(pz, xmul(nz, 0.00001f));     // :394
          ++n_shadow;
          const RtHit sh = rt_closest_bruteforce(p, ox, oy, oz, rx, ry, rz);
          if (sh.dist < FLT_MAX && sh.dist < r_mag) continue;  // :395-397, adds (0,0,0)
          float pw[3];
          rt_exact_lambert(rx, ry, rz, r_mag, nx, ny, nz, col, &p.lights[l][4], pw);
          pix[0] = xadd(pix[0], pw[0]); pix[1] = xadd(pix[1], pw[1]); pix[2] = xadd(pix[2], pw[2]);
        }
        // pixelColour + objectColor * indirectLight   (:156, indirectLight = 0.5)
        pix[0] = xadd(pix[0], xmul(col[0], 0.5f));
        pix[1] = xadd(pix[1], xmul(col[1], 0.5f));
        pix[2] = xadd(pix[2], xmul(col[2], 0.5f));
      }
    }
    if (SAMPLES) rt_store_pixel_n(p, pid, valid, pix, sp->n);
    else rt_store_pixel(p, pid, valid, pix);
  }
  rt_count_shadow(p, n_shadow);
}

__global__ void __launch_bounds__(128) rt_bruteforce_kernel(const __grid_constant__ RtKParams p) {
  rt_bruteforce_body<false>(p, nullptr);
}
__global__ void __launch_bounds__(128) rt_bruteforce_samples_kernel(const __grid_constant__ RtKParams p,
                                                                    const __grid_constant__ RtSamplesParams s) {
  rt_bruteforce_body<true>(p, &s);
}

// ------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------
int rt_prepare_scene(b200_ctx *ctx) {
  const int n = ctx->rt_n_tris;
  if (int rc = ensure(ctx, ctx->rt_geom, sizeof(float4) * 3 * (size_t)(n > 0 ? n : 1))) return rc;
  if (n > 0) {
    unsigned *bounds = nullptr;
    if (ctx->rt_bounds_on_device) {
      if (int rc = ensure(ctx, ctx->rt_bounds, 2 * sizeof(unsigned))) return rc;
      bounds = (unsigned *)ctx->rt_bounds.p;
      CU_CHECK(ctx, cudaMemsetAsync(bounds, 0, 2 * sizeof(unsigned), ctx->stream));
    }
    rt_prep_geom_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>((const rt_triangle *)ctx->rt_src.p, n,
                                                                  (float4 *)ctx->rt_geom.p, bounds);
    ctx->stats.kernel_launches++;
    CU_CHECK(ctx, cudaGetLastError());
    if (bounds) {
      float *hb = (float *)((char *)ctx->pinned + 512);   // past both counter blocks of the pinned scratch
      CU_CHECK(ctx, cudaMemcpyAsync(hb, bounds, 2 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
      CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
      ctx->rt_world_abs = fmaxf(ctx->rt_world_abs, hb[0]);
      ctx->rt_normal_abs = fmaxf(ctx->rt_normal_abs, hb[1]);
    }
  }
  return B200_OK;
}

static void rt_kparams(b200_ctx *ctx, const RtFrame &f, float *d_rgb, float *d_depth, int32_t *d_index,
                       uint32_t *d_argb, RtKParams &p) {
  memset(&p, 0, sizeof p);
  memcpy(p.cam, f.cam, sizeof p.cam);
  p.focal = f.focal;
  memcpy(p.R, f.R, sizeof p.R);
  p.W = f.W; p.H = f.H; p.row0 = f.row0; p.row1 = f.row1;
  p.il_n = f.il_n > 1 ? f.il_n : 1; p.il_r = f.il_n > 1 ? f.il_r : 0;
  p.n_lights = f.n_lights;
  memcpy(p.lights, f.lights, sizeof p.lights);
  p.geom = (const float4 *)ctx->rt_geom.p;
  p.src = (const rt_triangle *)ctx->rt_src.p;
  p.sph = (const rt_sphere *)ctx->rt_spheres.p;
  p.n_tris = ctx->rt_n_tris; p.n_sph = ctx->rt_n_spheres;
  p.rgb = d_rgb; p.depth = d_depth; p.index = d_index; p.argb = d_argb;
  p.counters = (unsigned long long *)ctx->counters.p;
}

int rt_launch(b200_ctx *ctx, const RtFrame &f, float *d_rgb, float *d_depth, int32_t *d_index,
              uint32_t *d_argb, const RtSamplesParams *sp) {
  RtKParams p;
  rt_kparams(ctx, f, d_rgb, d_depth, d_index, d_argb, p);
  const int rows = f.row1 - f.row0;
  if (rows <= 0 || f.W <= 0) return B200_OK;
  p.blocks_y = (rows + 15) / 16;
  const int my_blocks = p.blocks_y > p.il_r ? (p.blocks_y - p.il_r + p.il_n - 1) / p.il_n : 0;   // this launch's 16-row blocks
  if (my_blocks == 0) return B200_OK;
  if (ctx->opt_rt_bruteforce) {
    dim3 grid((f.W + 15) / 16, 2 * my_blocks);
    if (sp) {
      rt_bruteforce_samples_kernel<<<grid, 128, 0, ctx->stream>>>(p, *sp);
      tl_mark(ctx, "rt_bruteforce_samples_kernel");
    } else {
      rt_bruteforce_kernel<<<grid, 128, 0, ctx->stream>>>(p);
      tl_mark(ctx, "rt_bruteforce_kernel");
    }
    ctx->stats.kernel_launches++;
    CU_CHECK(ctx, cudaGetLastError());
    return B200_OK;
  }
  return rt_launch_filtered(ctx, f, p, sp);
}

// scenes this large get direction grids (declared in common.cuh; measured crossover at 4K: ~800 triangles)
constexpr unsigned long long RT_GRID_MAX_ENTRIES = 1ull << 26;   // 64 Mi list entries = 3.25 GiB

// Upper bound of |d|inf over the primary rays of rows [row0, row1): dir.x / dir.y are affine in (u, v),
// extremes at the corners.
static float rt_cam_dmax(const RtFrame &f) {
  float dmax = fabsf(f.focal);
  const int us[2] = {0, f.W - 1}, vs[2] = {f.row0, f.row1 - 1};
  for (int a = 0; a < 2; ++a)
    for (int b = 0; b < 2; ++b) {
      const float x = (float)(us[a] - f.W / 2), y = (float)(vs[b] - f.H / 2);
      for (int r = 0; r < 2; ++r) {
        const float d = f.R[0 + r] * x + f.R[4 + r] * y + f.R[8 + r] * f.focal + f.R[12 + r];
        dmax = fmaxf(dmax, fabsf(d) + 0.5f);
      }
    }
  return dmax * 1.001f + 1.0f;
}

// Whether the frame's sample directions form a half-pixel lattice (rt_lattice_kernel.cuh): dir0 depends on u only and
// dir1 on v only (R[4] = R[1] = 0), every value is finite, and sample 2 of every pixel but the last of the band has the
// bits of sample 0 of its right (lower) neighbour.  The kernel's own expression for dir (skeleton.cpp:126-128), one
// rounding per operation like the device's __f*_rn (no FMA contraction on the host); O(W + rows) per launch.  With
// R[4] = 0 the y term is a zero, which can change only the sign of a zero dir0, and no sample (dir0 - 0.5, dir0 + 0,
// dir0 + 0.5) keeps that sign: one row stands for all (likewise x for dir1).
static float rt_dir_host(const RtFrame &f, int r, float x, float y) {
  const float a = f.R[r] * x, b = f.R[4 + r] * y, c = f.R[8 + r] * f.focal, d = f.R[12 + r] * 1.0f;
  return (a + b) + (c + d);
}
static bool rt_lattice_exact(const RtFrame &f) {
  if (f.R[1] != 0.0f || f.R[4] != 0.0f) return false;
  for (int r = 0; r < 2; ++r) {   // r = 0: dir0 over the columns, r = 1: dir1 over the band's rows
    const int lo = r ? f.row0 : 0, hi = r ? f.row1 : f.W;
    uint32_t prev = 0;
    for (int c = lo; c < hi; ++c) {
      const float d = r ? rt_dir_host(f, 1, (float)(0 - f.W / 2), (float)(c - f.H / 2))
                        : rt_dir_host(f, 0, (float)(c - f.W / 2), (float)(f.row0 - f.H / 2));
      const float s0 = d + 0.5f * -1.0f, s1 = d + 0.5f * 0.0f, s2 = d + 0.5f * 1.0f;
      if (!std::isfinite(s0) || !std::isfinite(s1) || !std::isfinite(s2)) return false;
      uint32_t b0, b2;
      memcpy(&b0, &s0, sizeof b0); memcpy(&b2, &s2, sizeof b2);
      if (c > lo && b0 != prev) return false;
      prev = b2;
    }
  }
  return true;
}

// The camera-independent part of the plane-record preparation: scene, lights, shadow-ray bounds, buffers.
static void rt_prep_common(b200_ctx *ctx, const RtFrame &f, size_t origin_stride, const float *self_D, RtPrepParams &q) {
  q.geom = (const float4 *)ctx->rt_geom.p;
  q.n_tris = ctx->rt_n_tris;
  // world_S bounds |start - v0|inf of SHADOW rays (the camera's own plane records use the exact
  // |camera - v0|): their starts are hit points, which lie on the scene's geometry, so the camera
  // position does not enter (it tripled S, and with it the filter's margin, on the Cornell box)
  float m = ctx->rt_world_abs;
  q.n_lights = f.n_lights;
  for (int l = 0; l < f.n_lights; ++l)
    for (int k = 0; k < 3; ++k) {
      q.lights[l][k] = f.lights[l][k];
      m = fmaxf(m, fabsf(f.lights[l][k]));
    }
  q.world_S = 2.0f * m * 1.001f + 1e-3f;
  q.n_scale = ctx->rt_normal_abs;
  q.planes = (float4 *)ctx->rt_planes.p;
  q.origin_stride_f4 = origin_stride;
  q.dt_cam = (float *)ctx->rt_dtcam.p;
  q.self_D = (float *)self_D;   // null: a grid frame (a grid frame that falls back to streaming decides every self pair exactly)
}

// per thread: t, distance, index of the nine samples; the scene-streaming kernel also their ray lengths and the colour sum
constexpr size_t RT_HIT_SMEM = 27 * (size_t)RT_THREADS * sizeof(float);
constexpr size_t RT_STREAM_SMEM = 2 * (size_t)RT_TILE * RT_REC_F4 * sizeof(float4) + RT_HIT_SMEM + 12 * (size_t)RT_THREADS * sizeof(float);

static int rt_set_smem_limits(b200_ctx *ctx) {
  if (ctx->rt_grid_smem_set) return B200_OK;      // per context: function attributes are per device
  const size_t most = (size_t)(RT_THREADS / 32) * 2 * RT_WTILE * (RT_REC_F4 * sizeof(float4) + sizeof(int)) + RT_HIT_SMEM;
  CU_CHECK(ctx, cudaFuncSetAttribute(rt_filtered_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)most));
  CU_CHECK(ctx, cudaFuncSetAttribute(rt_filtered_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)most));
  CU_CHECK(ctx, cudaFuncSetAttribute(rt_filtered_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RT_STREAM_SMEM));
  CU_CHECK(ctx, cudaFuncSetAttribute(rt_filtered_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RT_STREAM_SMEM));
  CU_CHECK(ctx, cudaFuncSetAttribute(rt_filtered_views_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RT_STREAM_SMEM));
  CU_CHECK(ctx, cudaFuncSetAttribute(rt_filtered_views_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RT_STREAM_SMEM));
  CU_CHECK(ctx, cudaFuncSetAttribute(rt_filtered_samples_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)most));
  CU_CHECK(ctx, cudaFuncSetAttribute(rt_filtered_samples_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)most));
  CU_CHECK(ctx, cudaFuncSetAttribute(rt_filtered_samples_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RT_STREAM_SMEM));
  CU_CHECK(ctx, cudaFuncSetAttribute(rt_filtered_samples_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RT_STREAM_SMEM));
  CU_CHECK(ctx, cudaFuncSetAttribute(rt_lattice_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RT_LAT_LAUNCH_SMEM));
  // four blocks per SM need 220 KB of it: all that the SM can give to shared memory
  CU_CHECK(ctx, cudaFuncSetAttribute(rt_lattice_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
  ctx->rt_grid_smem_set = 1;
  return B200_OK;
}

// sp (the caller's sample pattern): the filtered kernels' samples instantiations, never the lattice kernel, and
// the block plan of gridded frames is neither read nor written.
int rt_launch_filtered(b200_ctx *ctx, const RtFrame &f, RtKParams &p, const RtSamplesParams *sp) {
  const int n = ctx->rt_n_tris;
  const int n_tiles = (n + RT_TILE - 1) / RT_TILE;
  const size_t origin_stride = (size_t)n_tiles * RT_TILE * RT_REC_F4;
  if (int rc = ensure(ctx, ctx->rt_planes, sizeof(float4) * (origin_stride * (1 + f.n_lights) + 1))) return rc;
  p.planes = (const float4 *)ctx->rt_planes.p;
  if (int rc = ensure(ctx, ctx->rt_dtcam, sizeof(float) * (size_t)(n > 0 ? n : 1))) return rc;
  p.dt_cam = (const float *)ctx->rt_dtcam.p;
  // large scenes: per-frame direction grids, then the grid kernels stream cell lists (decided here, before the plane
  // records are made: the self-pair signs are made only for the scene-streaming kernel, which uses them)
  bool use_grid = n > 0 && (ctx->opt_rt_grid == 1 || (ctx->opt_rt_grid == 0 && n >= RT_GRID_AUTO_TRIS));
  p.self_D = nullptr;
  if (!use_grid) {
    if (int rc = ensure(ctx, ctx->rt_selfD, sizeof(float) * (size_t)(n > 0 ? n : 1) * (f.n_lights > 0 ? f.n_lights : 1))) return rc;
    p.self_D = (const float *)ctx->rt_selfD.p;
  }

  if (n > 0) {
    RtPrepParams q;
    rt_prep_common(ctx, f, origin_stride, p.self_D, q);
    q.cam[0] = f.cam[0]; q.cam[1] = f.cam[1]; q.cam[2] = f.cam[2];
    q.focal = f.focal;
    q.dmax = rt_cam_dmax(f);   // over the band
    dim3 grid((n + 127) / 128, 1 + f.n_lights);
    rt_prep_planes_kernel<<<grid, 128, 0, ctx->stream>>>(q);
    tl_mark(ctx, "rt_prep_planes_kernel");
    ctx->stats.kernel_launches++;
    CU_CHECK(ctx, cudaGetLastError());
  }

  const int my_blocks = (p.blocks_y - p.il_r + p.il_n - 1) / p.il_n;
  dim3 grid((f.W + 15) / 16, my_blocks);
  const size_t hit_smem = RT_HIT_SMEM, smem = RT_STREAM_SMEM;

  if (use_grid) {
    const size_t cells = (size_t)grid.x * p.blocks_y + (size_t)f.n_lights * 6 * RT_GRID_FACE;   // camera cells: every block of the range
    const size_t scan_tmp = cells / 4096 + 2;
    ctx->rt_n_cells = cells; ctx->rt_n_cam_cells = (size_t)grid.x * p.blocks_y;
    if (int rc = ensure(ctx, ctx->rt_cells, sizeof(unsigned) * (4 * cells + 1 + scan_tmp))) return rc;
    unsigned *cnt = (unsigned *)ctx->rt_cells.p, *cursor = cnt + cells, *padded = cursor + cells,
             *off = padded + cells, *tmp = off + cells + 1;
    RtGridParams g;
    g.planes = (const float4 *)ctx->rt_planes.p;
    g.origin_stride_f4 = origin_stride;
    g.n_tris = n;
    memcpy(g.R, f.R, sizeof g.R);
    g.focal = f.focal;
    g.W = f.W; g.H = f.H; g.row0 = f.row0; g.row1 = f.row1;
    g.gx = (int)grid.x; g.gy = p.blocks_y;
    g.n_lights = f.n_lights;
    g.cell_cnt = cnt; g.cell_cursor = cursor; g.cell_off = off;
    g.cell_rec = nullptr; g.cell_idx = nullptr; g.cap = 0;
    // The counting pass also writes its (cell, record) pairs down when the last gridded frame of this context tells
    // how many to expect (+5 %); the lists are then filled from the pairs instead of by a second descent.
    unsigned long long *dc = (unsigned long long *)ctx->counters.p;
    g.pairs = nullptr; g.pair_cap = 0; g.pair_cursor = dc + 15;
    if (ctx->rt_grid_pairs_seen > 0 && ctx->rt_grid_pairs_n == n) {
      const unsigned long long want = ctx->rt_grid_pairs_seen + ctx->rt_grid_pairs_seen / 20 + 4096;
      if (int rc = ensure(ctx, ctx->rt_cell_pairs, sizeof(uint2) * (size_t)want)) return rc;
      g.pairs = (uint2 *)ctx->rt_cell_pairs.p;
      g.pair_cap = want;
      CU_CHECK(ctx, cudaMemsetAsync(g.pair_cursor, 0, sizeof(unsigned long long), ctx->stream));
    }
    CU_CHECK(ctx, cudaMemsetAsync(cnt, 0, sizeof(unsigned) * 2 * cells, ctx->stream));   // counts and cursors
    const dim3 bgrid((n + 7) / 8, 1 + f.n_lights);
    rt_grid_bin_kernel<false><<<bgrid, 256, 0, ctx->stream>>>(g);
    rt_grid_pad_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, ctx->stream>>>(cnt, padded, (int)cells);
    ctx->stats.kernel_launches += 2;
    CU_CHECK(ctx, cudaGetLastError());
    if (int rc = scan_exclusive(ctx, padded, off, (int)cells, tmp, dc + 9)) return rc;
    // the lists are sized from the scanned total: one small read-back ([9] total, [15] pairs written down)
    unsigned long long *hc = (unsigned long long *)ctx->pinned;
    CU_CHECK(ctx, cudaMemcpyAsync(hc, dc + 9, 7 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    const unsigned long long total = hc[0], n_pairs = g.pairs ? hc[6] : 0;
    if (total > RT_GRID_MAX_ENTRIES) {
      use_grid = false;   // lists larger than the budget (huge triangles everywhere): stream the scene instead
    } else {
      if (int rc = ensure(ctx, ctx->rt_cell_rec, sizeof(float4) * RT_REC_F4 * (size_t)(total + 4))) return rc;
      if (int rc = ensure(ctx, ctx->rt_cell_idx, sizeof(int) * (size_t)(total + 4))) return rc;
      g.cell_rec = (float4 *)ctx->rt_cell_rec.p;
      g.cell_idx = (int *)ctx->rt_cell_idx.p;
      g.cap = total;
      if (g.pairs && n_pairs > 0 && n_pairs <= g.pair_cap)
        rt_grid_place_kernel<<<(unsigned)((n_pairs + 255) / 256), 256, 0, ctx->stream>>>(g, n_pairs);
      else
        rt_grid_bin_kernel<true><<<bgrid, 256, 0, ctx->stream>>>(g);
      // what the next frame's pair buffer is sized from: the entries of this one (padding included: an upper bound)
      ctx->rt_grid_pairs_seen = g.pairs && n_pairs > 0 ? n_pairs : total;
      ctx->rt_grid_pairs_n = n;
      ctx->stats.kernel_launches++;
      CU_CHECK(ctx, cudaGetLastError());
      p.cell_off = off; p.cell_cnt = cnt;
      p.cell_rec = g.cell_rec; p.cell_idx = g.cell_idx;
    }
  }

  if (int rc = rt_set_smem_limits(ctx)) return rc;
  if (use_grid) {
    // one private double-buffered ring per warp: records + triangle indices
    const size_t gsmem = (size_t)(RT_THREADS / 32) * 2 * RT_WTILE * (RT_REC_F4 * sizeof(float4) + sizeof(int)) + hit_smem;
    // Block order and splits from the block costs of the last gridded frame (rt_plan_kernel); this frame leaves its
    // own for the next one.  Costs are kept per block of the WHOLE frame (any row range / interleave class finds its
    // blocks).  Layout: cost[2][frame blocks], plan[nb + 7 * RT_PLAN_MAX_SPLIT], plan_n.
    const unsigned nb = grid.x * grid.y;
    dim3 lgrid = grid;
    p.plan = nullptr; p.plan_n = nullptr; p.block_cost = nullptr; p.gx = (int)grid.x;
    if (grid.x <= 4096 && grid.y <= 4096 && ctx->opt_rt_plan && !sp) {
      const size_t frame_blocks = (size_t)grid.x * (size_t)((f.H + 15) / 16 + 1);
      const size_t plan_cap = (size_t)nb + 7 * (size_t)RT_PLAN_MAX_SPLIT;
      // (sized for the whole frame whatever this launch's share: a buffer that grew would lose the cost history)
      const size_t plan_room = frame_blocks + 7 * (size_t)RT_PLAN_MAX_SPLIT;
      const void *before = ctx->rt_plan.p;
      if (int rc = ensure(ctx, ctx->rt_plan, sizeof(unsigned) * (2 * frame_blocks + plan_room + 4))) return rc;
      if (ctx->rt_plan.p != before) ctx->rt_plan_valid = 0;
      unsigned *cost = (unsigned *)ctx->rt_plan.p, *plan = cost + 2 * frame_blocks, *plan_n = plan + plan_room;
      const unsigned long long shape = ((unsigned long long)f.W << 44) ^ ((unsigned long long)f.H << 28) ^ ((unsigned long long)n << 4) ^ (unsigned long long)f.n_lights;
      const bool planned = ctx->rt_plan_shape == shape && ctx->rt_plan_valid;
      const int cur = planned ? ctx->rt_plan_flip ^ 1 : 0;
      CU_CHECK(ctx, cudaMemsetAsync(cost + (size_t)cur * frame_blocks, 0, sizeof(unsigned) * frame_blocks, ctx->stream));
      if (planned) {
        rt_plan_kernel<<<1, 1024, 0, ctx->stream>>>(cost + (size_t)(cur ^ 1) * frame_blocks, (int)grid.x, (int)nb, f.row0 >> 4, p.il_n, p.il_r,
                                                    plan, plan_n, ctx->rt_plan_heavy ? (unsigned)ctx->rt_plan_heavy : RT_PLAN_HEAVY);
        ctx->stats.kernel_launches++;
        p.plan = plan; p.plan_n = plan_n;
        lgrid = dim3((unsigned)plan_cap);
      }
      p.block_cost = cost + (size_t)cur * frame_blocks;
      ctx->rt_plan_shape = shape; ctx->rt_plan_valid = 1; ctx->rt_plan_flip = cur;
    }
    if (sp && f.n_lights > 1)
      rt_filtered_samples_kernel<true, true><<<lgrid, RT_THREADS, gsmem, ctx->stream>>>(p, *sp);
    else if (sp)
      rt_filtered_samples_kernel<false, true><<<lgrid, RT_THREADS, gsmem, ctx->stream>>>(p, *sp);
    else if (f.n_lights > 1)
      rt_filtered_kernel<true, true><<<lgrid, RT_THREADS, gsmem, ctx->stream>>>(p);
    else
      rt_filtered_kernel<false, true><<<lgrid, RT_THREADS, gsmem, ctx->stream>>>(p);
    tl_mark(ctx, sp ? "rt_filtered_samples_kernel<grid>" : "rt_filtered_kernel<grid>");
  } else if (sp) {
    if (f.n_lights > 1)
      rt_filtered_samples_kernel<true, false><<<grid, RT_THREADS, smem, ctx->stream>>>(p, *sp);
    else
      rt_filtered_samples_kernel<false, false><<<grid, RT_THREADS, smem, ctx->stream>>>(p, *sp);
    tl_mark(ctx, "rt_filtered_samples_kernel");
  } else if (f.n_lights <= 1 && rt_lattice_exact(f)) {
    rt_lattice_kernel<<<grid, RT_THREADS, RT_LAT_LAUNCH_SMEM, ctx->stream>>>(p);
    tl_mark(ctx, "rt_lattice_kernel");
  } else {
    if (f.n_lights > 1)
      rt_filtered_kernel<true, false><<<grid, RT_THREADS, smem, ctx->stream>>>(p);
    else
      rt_filtered_kernel<false, false><<<grid, RT_THREADS, smem, ctx->stream>>>(p);
    tl_mark(ctx, "rt_filtered_kernel");
  }
  ctx->stats.kernel_launches++;
  CU_CHECK(ctx, cudaGetLastError());
  return B200_OK;
}

// Whole frames of n_views cameras (same W, H, lights) into outputs that hold the frames back to back.  Scenes
// for the scene-streaming kernel render up to RT_VIEWS_MAX views per launch: one preparation launch makes each
// view's camera records and the shared light records, one render launch covers every view (blockIdx.z).  So
// the per-view buffers are sized for RT_VIEWS_MAX views whatever n_views.  Gridded scenes and the brute-force
// kernel render view by view: their grids are per camera.  So does a single view: the same frame through the
// single-view kernels, without the batch's 5 KB of launch parameters (measured 5 % slower at 320x256).
int rt_launch_views(b200_ctx *ctx, const RtFrame *fs, int n_views, float *d_rgb, float *d_depth, int32_t *d_index,
                    uint32_t *d_argb) {
  const RtFrame &f = fs[0];
  const size_t npix = (size_t)f.W * f.H;
  const int n = ctx->rt_n_tris;
  const bool use_grid = n > 0 && (ctx->opt_rt_grid == 1 || (ctx->opt_rt_grid == 0 && n >= RT_GRID_AUTO_TRIS));
  if (ctx->opt_rt_bruteforce || use_grid || n_views == 1) {
    for (int k = 0; k < n_views; ++k) {
      const size_t o = (size_t)k * npix;
      if (int rc = rt_launch(ctx, fs[k], d_rgb ? d_rgb + 3 * o : nullptr, d_depth ? d_depth + o : nullptr,
                             d_index ? d_index + o : nullptr, d_argb ? d_argb + o : nullptr))
        return rc;
    }
    return B200_OK;
  }
  if (npix == 0) return B200_OK;
  RtKParams p;
  rt_kparams(ctx, f, nullptr, nullptr, nullptr, nullptr, p);
  p.row0 = 0; p.row1 = f.H; p.il_n = 1; p.il_r = 0;
  p.blocks_y = (f.H + 15) / 16;
  const int per = n_views < RT_VIEWS_MAX ? n_views : RT_VIEWS_MAX;
  const size_t origin_stride = (size_t)((n + RT_TILE - 1) / RT_TILE) * RT_TILE * RT_REC_F4;
  if (int rc = ensure(ctx, ctx->rt_planes, sizeof(float4) * (origin_stride * (per + f.n_lights) + 1))) return rc;
  if (int rc = ensure(ctx, ctx->rt_dtcam, sizeof(float) * (size_t)(n > 0 ? n : 1) * per)) return rc;
  if (int rc = ensure(ctx, ctx->rt_selfD, sizeof(float) * (size_t)(n > 0 ? n : 1) * (f.n_lights > 0 ? f.n_lights : 1))) return rc;
  p.planes = (const float4 *)ctx->rt_planes.p;
  p.dt_cam = (const float *)ctx->rt_dtcam.p;
  p.self_D = (const float *)ctx->rt_selfD.p;
  if (int rc = rt_set_smem_limits(ctx)) return rc;

  for (int k0 = 0; k0 < n_views; k0 += RT_VIEWS_MAX) {
    const int nv = n_views - k0 < RT_VIEWS_MAX ? n_views - k0 : RT_VIEWS_MAX;
    RtViewsParams v;
    memset(&v, 0, sizeof v);
    v.n_views = nv;
    for (int j = 0; j < nv; ++j) {
      const RtFrame &fj = fs[k0 + j];
      memcpy(v.view[j].cam, fj.cam, sizeof v.view[j].cam);
      v.view[j].focal = fj.focal;
      memcpy(v.view[j].R, fj.R, sizeof v.view[j].R);
    }
    if (n > 0) {
      RtPrepParams q;
      rt_prep_common(ctx, f, origin_stride, p.self_D, q);
      q.cam[0] = q.cam[1] = q.cam[2] = 0.f; q.focal = 0.f; q.dmax = 0.f;   // per view, below
      RtPrepViews pv;
      memset(&pv, 0, sizeof pv);
      pv.n_views = nv;
      for (int j = 0; j < nv; ++j) {
        const RtFrame &fj = fs[k0 + j];
        for (int k = 0; k < 3; ++k) {
          pv.cam[j][k] = fj.cam[k];
          pv.cam_inf = fmaxf(pv.cam_inf, fabsf(fj.cam[k]));
        }
        pv.cam[j][3] = fj.focal;
        pv.dmax[j] = rt_cam_dmax(fj);
      }
      rt_prep_planes_views_kernel<<<dim3((n + 127) / 128, nv + f.n_lights), 128, 0, ctx->stream>>>(q, pv);
      ctx->stats.kernel_launches++;
      CU_CHECK(ctx, cudaGetLastError());
    }
    const size_t o = (size_t)k0 * npix;
    p.rgb = d_rgb ? d_rgb + 3 * o : nullptr;
    p.depth = d_depth ? d_depth + o : nullptr;
    p.index = d_index ? d_index + o : nullptr;
    p.argb = d_argb ? d_argb + o : nullptr;
    const dim3 grid((f.W + 15) / 16, p.blocks_y, nv);
    if (f.n_lights > 1)
      rt_filtered_views_kernel<true><<<grid, RT_THREADS, RT_STREAM_SMEM, ctx->stream>>>(p, v);
    else
      rt_filtered_views_kernel<false><<<grid, RT_THREADS, RT_STREAM_SMEM, ctx->stream>>>(p, v);
    tl_mark(ctx, "rt_filtered_views_kernel");
    ctx->stats.kernel_launches++;
    CU_CHECK(ctx, cudaGetLastError());
  }
  return B200_OK;
}

// Profiling: resident blocks per SM of rt_lattice_kernel at the shared memory and attributes of its launches.
extern "C" int b200_debug_rt_lattice_blocks_per_sm(b200_ctx *ctx, int *blocks) {
  if (!ctx || ctx->multi || !blocks) return B200_EINVAL;
  if (int rc = rt_set_smem_limits(ctx)) return rc;
  CU_CHECK(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks, rt_lattice_kernel, RT_THREADS, RT_LAT_LAUNCH_SMEM));
  return B200_OK;
}

// Tests / tuning: the factor over the mean block cost from which a block of a planned frame is split (0: the default).
extern "C" int b200_debug_rt_plan_heavy(b200_ctx *ctx, int factor) {
  if (!ctx || ctx->multi || factor < 0) return B200_EINVAL;
  ctx->rt_plan_heavy = factor;
  return B200_OK;
}
