// C ABI of include/b200render.h: context, uploads, host-pointer entry points.
#include "common.cuh"
#include <math.h>
#include <stdio.h>
#include <string.h>

int ctx_fail(b200_ctx *ctx, int code, const char *what, cudaError_t e) {
  if (ctx) {
    ctx->err = what ? what : "";
    if (e != cudaSuccess) {
      ctx->err += ": ";
      ctx->err += cudaGetErrorString(e);
    }
  }
  return code;
}

int ensure(b200_ctx *ctx, DevBuf &b, size_t bytes) {
  if (bytes <= b.cap && b.p) return B200_OK;
  size_t cap = bytes < 256 ? 256 : bytes;
  if (b.p) {
    // a buffer that has to grow grows by a quarter more than asked: frame-sized buffers (cell lists,
    // row tables, bands whose edges move) would otherwise be freed and allocated again -- ~1.5 ms
    // with its implicit synchronisation -- every time a frame needs a little more than the last
    cap += cap / 4;
    cudaStreamSynchronize(ctx->stream);
    cudaFree(b.p);
    b.p = nullptr; b.cap = 0;
  }
  cudaError_t e = cudaMalloc(&b.p, cap);
  if (e != cudaSuccess) { b.p = nullptr; return ctx_fail(ctx, B200_ENOMEM, "cudaMalloc", e); }
  b.cap = cap;
  return B200_OK;
}

static int ensure_pinned(b200_ctx *ctx, size_t bytes) {
  if (bytes <= ctx->pinned_cap) return B200_OK;
  if (ctx->pinned) { cudaStreamSynchronize(ctx->stream); cudaFreeHost(ctx->pinned); ctx->pinned = nullptr; ctx->pinned_cap = 0; }
  cudaError_t e = cudaMallocHost(&ctx->pinned, bytes);
  if (e != cudaSuccess) { ctx->pinned = nullptr; return ctx_fail(ctx, B200_ENOMEM, "cudaMallocHost", e); }
  ctx->pinned_cap = bytes;
  return B200_OK;
}

int band_slice_done(b200_ctx *ctx, int a, int b) {
  if (!ctx->slice_host || b <= a) return B200_OK;
  cudaEvent_t ev = ctx->ev_slice[ctx->slice_n++ % B200_SLICES];
  CU_CHECK(ctx, cudaEventRecord(ev, ctx->stream));
  CU_CHECK(ctx, cudaStreamWaitEvent(ctx->copy_stream, ev, 0));
  CU_CHECK(ctx, cudaMemcpyAsync(ctx->slice_host + (size_t)(a - ctx->slice_row0) * ctx->slice_w,
                                ctx->slice_dev + (size_t)a * ctx->slice_w, (size_t)(b - a) * ctx->slice_w * sizeof(uint32_t),
                                cudaMemcpyDeviceToHost, ctx->copy_stream));
  return B200_OK;
}

extern "C" {

int b200_init(int device, b200_ctx **out) {
  if (!out) return B200_EINVAL;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) return B200_ENODEV;
  if (device < 0 || device >= n) return B200_EINVAL;
  if (cudaSetDevice(device) != cudaSuccess) return B200_ECUDA;
  b200_ctx *ctx = new b200_ctx();
  ctx->device = device;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
  ctx->timeline = getenv("B200_TIMELINE") != nullptr;
  if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_main, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->ev_copied, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess) {
    delete ctx;
    return B200_ECUDA;
  }
  for (int i = 0; i < B200_SLICES; ++i)
    if (cudaEventCreateWithFlags(&ctx->ev_slice[i], cudaEventDisableTiming) != cudaSuccess) { delete ctx; return B200_ECUDA; }
  for (int i = 0; i < RAST_UP_CHUNKS; ++i)
    if (cudaEventCreateWithFlags(&ctx->ev_up[i], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_chunk[i], cudaEventDisableTiming) != cudaSuccess) { delete ctx; return B200_ECUDA; }
  ctx->stream = ctx->own_stream;
  if (ensure(ctx, ctx->counters, 32 * sizeof(unsigned long long)) != B200_OK || ensure_pinned(ctx, 1024) != B200_OK) {
    delete ctx;
    return B200_ENOMEM;
  }
  *out = ctx;
  return B200_OK;
}

// Entry points that only exist per device (device pointers, streams, intermediate buffers).
#define SINGLE_ONLY(ctx) \
  do { if ((ctx)->multi) return ctx_fail(ctx, B200_EINVAL, "not available on a multi-GPU context: use one context per device"); } while (0)

void b200_destroy(b200_ctx *ctx) {
  if (!ctx) return;
  if (ctx->multi) { multi_destroy(ctx); delete ctx; return; }
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  DevBuf *bufs[] = {&ctx->rt_src, &ctx->rt_geom, &ctx->rt_spheres, &ctx->rt_planes, &ctx->rt_dtcam, &ctx->rt_selfD, &ctx->rt_bounds, &ctx->rt_cells, &ctx->rt_cell_rec, &ctx->rt_cell_idx, &ctx->rast_src,
                    &ctx->rast_setup, &ctx->rast_rowsA, &ctx->rast_rowsB, &ctx->rast_bins, &ctx->rast_tile_count, &ctx->rast_tile_bits,
                    &ctx->rast_tmp, &ctx->rast_keys, &ctx->rast_trimeta, &ctx->rast_big, &ctx->rast_orig, &ctx->rast_shadow8, &ctx->rast_srowsB, &ctx->rast_srowsL, &ctx->rast_row_owner, &ctx->rast_world, &ctx->rast_geom_tmp, &ctx->rast_screen, &ctx->rast_low, &ctx->rast_high, &ctx->rast_shadow,
                    &ctx->rast_depth, &ctx->rast_index, &ctx->out_rgb, &ctx->out_depth, &ctx->out_index,
                    &ctx->out_argb, &ctx->counters, &ctx->rt_plan, &ctx->rt_cell_pairs, &ctx->rast_tex_images, &ctx->rast_tex_noise,
                    &ctx->rast_colour_keys, &ctx->rast_colour_rgb, &ctx->rast_colour_tmp, &ctx->rt_query};
  for (DevBuf *b : bufs) if (b->p) cudaFree(b->p);
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  cudaEventDestroy(ctx->ev0);
  cudaEventDestroy(ctx->ev1);
  cudaEventDestroy(ctx->ev_copied);
  for (int i = 0; i < B200_SLICES; ++i) cudaEventDestroy(ctx->ev_slice[i]);
  for (int i = 0; i < 64; ++i) if (ctx->tl_ev[i]) cudaEventDestroy(ctx->tl_ev[i]);
  for (int i = 0; i < RAST_UP_CHUNKS; ++i) { cudaEventDestroy(ctx->ev_up[i]); cudaEventDestroy(ctx->ev_chunk[i]); }
  cudaEventDestroy(ctx->ev_join);
  cudaEventDestroy(ctx->ev_main);
  cudaStreamDestroy(ctx->aux_stream);
  cudaStreamDestroy(ctx->copy_stream);
  cudaStreamDestroy(ctx->own_stream);
  delete ctx;
}

const char *b200_last_error(const b200_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }
void *b200_stream(b200_ctx *ctx) { return ctx && !ctx->multi ? (void *)ctx->stream : nullptr; }

static int finish_stats(b200_ctx *ctx);

// Also the point where a pipelined raster frame is verified (and re-rendered if its
// size guess was too small), so what is on the device afterwards is always exact.
int b200_synchronize(b200_ctx *ctx) {
  if (!ctx) return B200_EINVAL;
  if (ctx->multi) return multi_synchronize(ctx);
  return finish_stats(ctx);
}

int b200_set_stream(b200_ctx *ctx, void *cuda_stream) {
  if (!ctx) return B200_EINVAL;
  SINGLE_ONLY(ctx);
  if (int rc = finish_stats(ctx)) return rc;
  ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
  return B200_OK;
}

int b200_set_option(b200_ctx *ctx, int option, int value) {
  if (!ctx) return B200_EINVAL;
  if (ctx->multi) return multi_set_option(ctx, option, value);
  switch (option) {
    case B200_OPT_RT_BRUTEFORCE: ctx->opt_rt_bruteforce = value != 0; return B200_OK;
    case B200_OPT_RAST_PATH:
      if (value < 0 || value > 2) return ctx_fail(ctx, B200_EINVAL, "raster path must be 0, 1 or 2");
      ctx->opt_rast_path = value;
      return B200_OK;
    case B200_OPT_RT_INTERLEAVE_N:
      if (value < 1 || value > 4096) return ctx_fail(ctx, B200_EINVAL, "interleave count must be 1..4096");
      ctx->opt_rt_il_n = value;
      if (ctx->opt_rt_il_r >= value) ctx->opt_rt_il_r = 0;
      return B200_OK;
    case B200_OPT_RT_INTERLEAVE_R:
      if (value < 0 || value >= ctx->opt_rt_il_n) return ctx_fail(ctx, B200_EINVAL, "interleave index must be below the count");
      ctx->opt_rt_il_r = value;
      return B200_OK;
    case B200_OPT_RT_GRID:
      if (value < 0 || value > 2) return ctx_fail(ctx, B200_EINVAL, "grid mode must be 0, 1 or 2");
      ctx->opt_rt_grid = value;
      return B200_OK;
    case B200_OPT_RAST_PIPELINED:
      ctx->opt_rast_pipelined = value != 0;
      ctx->rast_spec.valid = 0;
      return B200_OK;
    case B200_OPT_RT_PLAN:
      ctx->opt_rt_plan = value != 0;
      ctx->rt_plan_valid = 0;
      return B200_OK;
    case B200_OPT_RAST_COLOUR_MODE:
      if (value < 0 || value > 2) return ctx_fail(ctx, B200_EINVAL, "colour mode must be 0, 1 or 2");
      ctx->opt_rast_colour = value;
      ctx->rast_spec.valid = 0;
      return B200_OK;
    case B200_OPT_RAST_BAND_CULL:
      ctx->opt_rast_band_cull = value != 0;
      ctx->rast_spec.valid = 0;
      return B200_OK;
    case B200_OPT_RAST_TILE_LOG2:
      if (value < 3 || value > 5) return ctx_fail(ctx, B200_EINVAL, "tile log2 must be 3..5");
      ctx->opt_rast_tile_log2 = value;
      return B200_OK;
  }
  return ctx_fail(ctx, B200_EINVAL, "unknown option");
}

int b200_get_stats(b200_ctx *ctx, b200_stats *out) {
  if (!ctx || !out) return B200_EINVAL;
  if (ctx->multi) { *out = ctx->stats; return B200_OK; }   // summed over the devices by the last frame
  if (int rc = finish_stats(ctx)) return rc;
  *out = ctx->stats;
  return B200_OK;
}

// Every render ends by copying its counters into the second half of the pinned scratch
// (the first half takes the mid-frame read-backs).
static int enqueue_counter_readback(b200_ctx *ctx) {
  CU_CHECK(ctx, cudaMemcpyAsync((unsigned long long *)ctx->pinned + 32, ctx->counters.p, 32 * sizeof(unsigned long long),
                                cudaMemcpyDeviceToHost, ctx->stream));
  return B200_OK;
}

// ---- RT ---------------------------------------------------------------------------

static int check_camera(b200_ctx *ctx, const camera_t *cam) {
  if (!cam) return ctx_fail(ctx, B200_EINVAL, "null camera");
  if (cam->width <= 0 || cam->height <= 0 || cam->width > 32768 || cam->height > 32768)
    return ctx_fail(ctx, B200_EINVAL, "bad resolution");
  return B200_OK;
}

int rt_upload_scene(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres,
                    int n_spheres) {
  if (!ctx) return B200_EINVAL;
  SINGLE_ONLY(ctx);
  if (n_tris < 0 || n_spheres < 0 || (n_tris > 0 && !tris) || (n_spheres > 0 && !spheres))
    return ctx_fail(ctx, B200_EINVAL, "bad scene arguments");
  cudaSetDevice(ctx->device);
  if (int rc = ensure(ctx, ctx->rt_src, sizeof(rt_triangle) * (size_t)(n_tris ? n_tris : 1))) return rc;
  if (int rc = ensure(ctx, ctx->rt_spheres, sizeof(rt_sphere) * (size_t)(n_spheres ? n_spheres : 1))) return rc;
  if (n_tris) CU_CHECK(ctx, cudaMemcpyAsync(ctx->rt_src.p, tris, sizeof(rt_triangle) * (size_t)n_tris,
                                            cudaMemcpyHostToDevice, ctx->stream));
  if (n_spheres) CU_CHECK(ctx, cudaMemcpyAsync(ctx->rt_spheres.p, spheres, sizeof(rt_sphere) * (size_t)n_spheres,
                                               cudaMemcpyHostToDevice, ctx->stream));
  ctx->rt_n_tris = n_tris;
  ctx->rt_n_spheres = n_spheres;
  // bound of |coordinate| over the scene, for the shadow filter's error budget: small scenes on the
  // host (no synchronisation), large ones inside the preparation kernel (one 8-byte read-back)
  float m = 0.f, nm = 1.f;
  ctx->rt_bounds_on_device = n_tris > 4096;
  if (!ctx->rt_bounds_on_device)
    for (int i = 0; i < n_tris; ++i)
      for (int k = 0; k < 3; ++k) {
        nm = fabsf(tris[i].normal[k]) <= 1e30f ? fmaxf(nm, fabsf(tris[i].normal[k])) : 1e30f;   // NaN / inf: widest margins
        m = fmaxf(m, fabsf(tris[i].v0[k]));
        m = fmaxf(m, fabsf(tris[i].v1[k]));
        m = fmaxf(m, fabsf(tris[i].v2[k]));
      }
  for (int i = 0; i < n_spheres; ++i)
    for (int k = 0; k < 3; ++k) m = fmaxf(m, fabsf(spheres[i].centre[k]) + fabsf(spheres[i].radius));
  ctx->rt_world_abs = m;
  ctx->rt_normal_abs = nm;
  return rt_prepare_scene(ctx);
}

static int fill_frame(b200_ctx *ctx, const camera_t *cam, const light_t *lights, int n_lights, int row0,
                      int row1, RtFrame &f) {
  if (int rc = check_camera(ctx, cam)) return rc;
  if (n_lights < 0 || n_lights > B200_MAX_LIGHTS || (n_lights > 0 && !lights))
    return ctx_fail(ctx, B200_EINVAL, "bad lights (at most 8)");
  if (row0 < 0 || row1 > cam->height || row0 > row1) return ctx_fail(ctx, B200_EINVAL, "bad row band");
  memcpy(f.cam, cam->pos, sizeof f.cam);
  f.focal = cam->focal;
  memcpy(f.R, cam->R, sizeof f.R);
  f.W = cam->width; f.H = cam->height; f.row0 = row0; f.row1 = row1;
  f.il_n = 1; f.il_r = 0;
  f.n_lights = n_lights;
  memset(f.lights, 0, sizeof f.lights);
  for (int l = 0; l < n_lights; ++l) {
    memcpy(&f.lights[l][0], lights[l].pos, 4 * sizeof(float));
    memcpy(&f.lights[l][4], lights[l].colour, 3 * sizeof(float));
  }
  return B200_OK;
}

// One RT frame on device buffers; il_n / il_r: the 16-row block interleave (1, 0 = every row).
static int rt_frame_device(b200_ctx *ctx, const camera_t *cam, const light_t *lights, int n_lights,
                           int row_begin, int row_end, float *d_rgb, float *d_depth, int32_t *d_index,
                           uint32_t *d_argb, int il_n, int il_r) {
  RtFrame f;
  if (int rc = fill_frame(ctx, cam, lights, n_lights, row_begin, row_end, f)) return rc;
  cudaSetDevice(ctx->device);
  if (ctx->rast_inflight.active) if (int rc = finish_stats(ctx)) return rc;   // the counters are shared
  f.il_n = il_n; f.il_r = il_r;
  ctx->stats.kernel_launches = 0;
  CU_CHECK(ctx, cudaMemsetAsync(ctx->counters.p, 0, 32 * sizeof(unsigned long long), ctx->stream));
  CU_CHECK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  ctx->tl_n = 0;
  tl_mark(ctx, "frame start");
  if (int rc = rt_launch(ctx, f, d_rgb, d_depth, d_index, d_argb)) return rc;
  CU_CHECK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  uint64_t my_rows = 0;   // rows of this context's 16-row blocks
  for (int b = f.il_r; b * 16 < row_end - row_begin; b += f.il_n)
    my_rows += (uint64_t)((row_end - row_begin - b * 16) < 16 ? (row_end - row_begin - b * 16) : 16);
  ctx->stats.primary_rays = (uint64_t)f.W * my_rows * 9u;
  if (int rc = enqueue_counter_readback(ctx)) return rc;
  ctx->pending = 1;
  return B200_OK;
}

// The interleave options apply to this entry only (see the header); the host-pointer
// entries always render every row of their band.
int rt_render_device(b200_ctx *ctx, const camera_t *cam, const light_t *lights, int n_lights,
                     int row_begin, int row_end, float *d_rgb, float *d_depth, int32_t *d_index,
                     uint32_t *d_argb) {
  if (!ctx) return B200_EINVAL;
  SINGLE_ONLY(ctx);
  return rt_frame_device(ctx, cam, lights, n_lights, row_begin, row_end, d_rgb, d_depth, d_index, d_argb,
                         ctx->opt_rt_il_n, ctx->opt_rt_il_r);
}

}  // extern "C"

// ---- RT, batched views: whole frames of n_views cameras of one size ---------------------
// (also the multi-GPU context's check, before the views are shared out)
int check_views(b200_ctx *ctx, const camera_t *cams, int n_views, const light_t *lights, int n_lights) {
  if (n_views < 1) return ctx_fail(ctx, B200_EINVAL, "n_views must be at least 1");
  if (!cams) return ctx_fail(ctx, B200_EINVAL, "null cameras");
  for (int k = 0; k < n_views; ++k) {
    if (int rc = check_camera(ctx, &cams[k])) return rc;
    if (cams[k].width != cams[0].width || cams[k].height != cams[0].height)
      return ctx_fail(ctx, B200_EINVAL, "every view must have the same width and height");
  }
  if (n_lights < 0 || n_lights > B200_MAX_LIGHTS || (n_lights > 0 && !lights))
    return ctx_fail(ctx, B200_EINVAL, "bad lights (at most 8)");
  return B200_OK;
}

extern "C" {

static int copy_out(b200_ctx *ctx, void *host, const void *dev, size_t bytes);

static int rt_views_device(b200_ctx *ctx, const camera_t *cams, int n_views, const light_t *lights, int n_lights,
                           float *d_rgb, float *d_depth, int32_t *d_index, uint32_t *d_argb) {
  if (int rc = check_views(ctx, cams, n_views, lights, n_lights)) return rc;
  std::vector<RtFrame> fs((size_t)n_views);
  for (int k = 0; k < n_views; ++k)
    if (int rc = fill_frame(ctx, &cams[k], lights, n_lights, 0, cams[0].height, fs[k])) return rc;
  cudaSetDevice(ctx->device);
  if (ctx->rast_inflight.active) if (int rc = finish_stats(ctx)) return rc;   // the counters are shared
  ctx->stats.kernel_launches = 0;
  CU_CHECK(ctx, cudaMemsetAsync(ctx->counters.p, 0, 32 * sizeof(unsigned long long), ctx->stream));
  CU_CHECK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  ctx->tl_n = 0;
  tl_mark(ctx, "frame start");
  if (int rc = rt_launch_views(ctx, fs.data(), n_views, d_rgb, d_depth, d_index, d_argb)) return rc;
  CU_CHECK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  ctx->stats.primary_rays = (uint64_t)n_views * (uint64_t)cams[0].width * (uint64_t)cams[0].height * 9u;
  if (int rc = enqueue_counter_readback(ctx)) return rc;
  ctx->pending = 1;
  return B200_OK;
}

int rt_render_views_device(b200_ctx *ctx, const camera_t *cams, int n_views, const light_t *lights, int n_lights,
                           float *d_rgb, float *d_depth, int32_t *d_index, uint32_t *d_argb) {
  if (!ctx) return B200_EINVAL;
  SINGLE_ONLY(ctx);
  return rt_views_device(ctx, cams, n_views, lights, n_lights, d_rgb, d_depth, d_index, d_argb);
}

// The host-pointer views entries: the views into the staging buffers, then one copy per output.
static int rt_views_host(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres, int n_spheres,
                         const camera_t *cams, int n_views, const light_t *lights, int n_lights, float *rgb_out,
                         float *depth_out, int32_t *index_out, uint32_t *argb_out) {
  if (int rc = check_views(ctx, cams, n_views, lights, n_lights)) return rc;
  if (int rc = rt_upload_scene(ctx, tris, n_tris, spheres, n_spheres)) return rc;
  const size_t npix = (size_t)n_views * cams[0].width * cams[0].height;
  if (rgb_out) if (int rc = ensure(ctx, ctx->out_rgb, npix * 3 * sizeof(float))) return rc;
  if (depth_out) if (int rc = ensure(ctx, ctx->out_depth, npix * sizeof(float))) return rc;
  if (index_out) if (int rc = ensure(ctx, ctx->out_index, npix * sizeof(int32_t))) return rc;
  if (argb_out) if (int rc = ensure(ctx, ctx->out_argb, npix * sizeof(uint32_t))) return rc;
  if (int rc = rt_views_device(ctx, cams, n_views, lights, n_lights, rgb_out ? (float *)ctx->out_rgb.p : nullptr,
                               depth_out ? (float *)ctx->out_depth.p : nullptr,
                               index_out ? (int32_t *)ctx->out_index.p : nullptr,
                               argb_out ? (uint32_t *)ctx->out_argb.p : nullptr))
    return rc;
  if (int rc = copy_out(ctx, rgb_out, ctx->out_rgb.p, npix * 3 * sizeof(float))) return rc;
  if (int rc = copy_out(ctx, depth_out, ctx->out_depth.p, npix * sizeof(float))) return rc;
  if (int rc = copy_out(ctx, index_out, ctx->out_index.p, npix * sizeof(int32_t))) return rc;
  if (int rc = copy_out(ctx, argb_out, ctx->out_argb.p, npix * sizeof(uint32_t))) return rc;
  return finish_stats(ctx);
}

int render_raytrace_views(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres, int n_spheres,
                          const camera_t *cams, int n_views, const light_t *lights, int n_lights, float *rgb_out,
                          float *depth_out, int32_t *index_out) {
  if (!ctx) return B200_EINVAL;
  if (ctx->multi)
    return multi_raytrace_views(ctx, tris, n_tris, spheres, n_spheres, cams, n_views, lights, n_lights, rgb_out,
                                depth_out, index_out, nullptr);
  return rt_views_host(ctx, tris, n_tris, spheres, n_spheres, cams, n_views, lights, n_lights, rgb_out, depth_out,
                       index_out, nullptr);
}

int draw_raytrace_views(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres, int n_spheres,
                        const camera_t *cams, int n_views, const light_t *lights, int n_lights, uint32_t *argb_out) {
  if (!ctx) return B200_EINVAL;
  if (!argb_out) return ctx_fail(ctx, B200_EINVAL, "null framebuffer");
  if (ctx->multi)
    return multi_raytrace_views(ctx, tris, n_tris, spheres, n_spheres, cams, n_views, lights, n_lights, nullptr,
                                nullptr, nullptr, argb_out);
  return rt_views_host(ctx, tris, n_tris, spheres, n_spheres, cams, n_views, lights, n_lights, nullptr, nullptr,
                       nullptr, argb_out);
}

}  // extern "C"

// ---- RT, ray queries: ClosestIntersection / DirectLight's shadow test for caller-supplied rays --------------
static int check_ray_buffers(b200_ctx *ctx, const void *rays, const float *max_distance, int n_rays, const void *out,
                             bool occlusion) {
  if (n_rays < 0) return ctx_fail(ctx, B200_EINVAL, "negative ray count");
  if (n_rays > 0 && (!rays || !out || (occlusion && !max_distance)))
    return ctx_fail(ctx, B200_EINVAL, "null rays, limits or output");
  return B200_OK;
}

// (also the multi-GPU context's check, before the rays are shared out)
int check_rays(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres, int n_spheres,
               const rt_ray *rays, const float *max_distance, int n_rays, const void *out, bool occlusion) {
  if (n_tris < 0 || n_spheres < 0 || (n_tris > 0 && !tris) || (n_spheres > 0 && !spheres))
    return ctx_fail(ctx, B200_EINVAL, "bad scene arguments");
  return check_ray_buffers(ctx, rays, max_distance, n_rays, out, occlusion);
}

// One query on device buffers and the uploaded scene: d_hits for closest hits, d_occ (+ d_max) for occlusion.
static int rt_query_device(b200_ctx *ctx, const rt_ray *d_rays, const float *d_max, int n_rays, rt_intersection *d_hits,
                           uint8_t *d_occ) {
  cudaSetDevice(ctx->device);
  if (ctx->rast_inflight.active) if (int rc = finish_stats(ctx)) return rc;   // the counters are shared
  ctx->stats.kernel_launches = 0;
  CU_CHECK(ctx, cudaMemsetAsync(ctx->counters.p, 0, 32 * sizeof(unsigned long long), ctx->stream));
  CU_CHECK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  ctx->tl_n = 0;
  tl_mark(ctx, "query start");
  if (int rc = rt_launch_rays(ctx, d_rays, d_max, n_rays, d_hits, d_occ)) return rc;
  CU_CHECK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  ctx->stats.primary_rays = d_occ ? 0 : (uint64_t)n_rays;
  ctx->stats.shadow_rays = d_occ ? (uint64_t)n_rays : 0;
  if (int rc = enqueue_counter_readback(ctx)) return rc;
  ctx->pending = 3;
  return B200_OK;
}

// The host-pointer query entries: rays (and limits) to a staging buffer, the query, the results back.
static int rt_query_host(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres, int n_spheres,
                         const rt_ray *rays, const float *max_distance, int n_rays, rt_intersection *out,
                         uint8_t *occ_out, bool occlusion) {
  if (int rc = check_rays(ctx, tris, n_tris, spheres, n_spheres, rays, max_distance, n_rays,
                          occlusion ? (const void *)occ_out : (const void *)out, occlusion))
    return rc;
  if (n_rays == 0) return B200_OK;
  if (int rc = rt_upload_scene(ctx, tris, n_tris, spheres, n_spheres)) return rc;
  const size_t n = (size_t)n_rays;
  const size_t off_max = n * sizeof(rt_ray), off_out = (off_max + n * sizeof(float) + 255) & ~(size_t)255;
  const size_t out_bytes = occlusion ? n : n * sizeof(rt_intersection);
  if (int rc = ensure(ctx, ctx->rt_query, off_out + out_bytes)) return rc;
  char *buf = (char *)ctx->rt_query.p;
  CU_CHECK(ctx, cudaMemcpyAsync(buf, rays, n * sizeof(rt_ray), cudaMemcpyHostToDevice, ctx->stream));
  if (occlusion)
    CU_CHECK(ctx, cudaMemcpyAsync(buf + off_max, max_distance, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  if (int rc = rt_query_device(ctx, (const rt_ray *)buf, occlusion ? (const float *)(buf + off_max) : nullptr, n_rays,
                               occlusion ? nullptr : (rt_intersection *)(buf + off_out),
                               occlusion ? (uint8_t *)(buf + off_out) : nullptr))
    return rc;
  if (int rc = copy_out(ctx, occlusion ? (void *)occ_out : (void *)out, buf + off_out, out_bytes)) return rc;
  return finish_stats(ctx);
}

extern "C" {

int rt_closest_hits(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres, int n_spheres,
                    const rt_ray *rays, int n_rays, rt_intersection *out) {
  if (!ctx) return B200_EINVAL;
  if (ctx->multi) return multi_rays(ctx, tris, n_tris, spheres, n_spheres, rays, nullptr, n_rays, out, nullptr, false);
  return rt_query_host(ctx, tris, n_tris, spheres, n_spheres, rays, nullptr, n_rays, out, nullptr, false);
}

int rt_occluded(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres, int n_spheres,
                const rt_ray *rays, const float *max_distance, int n_rays, uint8_t *out) {
  if (!ctx) return B200_EINVAL;
  if (ctx->multi) return multi_rays(ctx, tris, n_tris, spheres, n_spheres, rays, max_distance, n_rays, nullptr, out, true);
  return rt_query_host(ctx, tris, n_tris, spheres, n_spheres, rays, max_distance, n_rays, nullptr, out, true);
}

int rt_closest_hits_device(b200_ctx *ctx, const rt_ray *d_rays, int n_rays, rt_intersection *d_out) {
  if (!ctx) return B200_EINVAL;
  SINGLE_ONLY(ctx);
  if (int rc = check_ray_buffers(ctx, d_rays, nullptr, n_rays, d_out, false)) return rc;
  if (n_rays == 0) return B200_OK;
  return rt_query_device(ctx, d_rays, nullptr, n_rays, d_out, nullptr);
}

int rt_occluded_device(b200_ctx *ctx, const rt_ray *d_rays, const float *d_max_distance, int n_rays, uint8_t *d_out) {
  if (!ctx) return B200_EINVAL;
  SINGLE_ONLY(ctx);
  if (int rc = check_ray_buffers(ctx, d_rays, d_max_distance, n_rays, d_out, true)) return rc;
  if (n_rays == 0) return B200_OK;
  return rt_query_device(ctx, d_rays, d_max_distance, n_rays, nullptr, d_out);
}

static int rast_frame(b200_ctx *ctx, bool whole_draw, const camera_t *cam, const rast_light_t *light, int row_begin,
                      int row_end, float *d_rgb, float *d_depth, int32_t *d_index, uint32_t *d_argb, bool allow_spec);

// Waits for the last render and reads its device counters back.  A pipelined raster
// frame is checked here against the sizes it was launched with.
static int finish_stats(b200_ctx *ctx) {
  CU_CHECK(ctx, cudaSetDevice(ctx->device));   // a re-render below allocates and launches: on this context's GPU
  CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
  if (!ctx->pending) return B200_OK;
  const unsigned long long *c = (const unsigned long long *)ctx->pinned + 32;
  if (ctx->pending == 2 && ctx->rast_inflight.active) {
    b200_ctx::RastInflight &f = ctx->rast_inflight;
    f.active = 0;
    bool ok = c[5] == 0 && (f.fast || c[3] <= f.cap_bins);
    if (f.whole_draw) {
      const int has_shadow = (ctx->rast_n_boxes > 0 || (c[7] & 2ull)) ? 1 : 0;
      ok = ok && c[24] <= f.cap_tris && !(c[7] & 1ull) && has_shadow == ctx->rast_has_shadow;
    }
    if (!ok) {
      // the frame outgrew the guess: render it again with exact sizes
      ctx->rast_spec.valid = 0;
      ctx->pending = 0;
      ctx->stats.respeculated++;
      if (int rc = rast_frame(ctx, f.whole_draw != 0, &f.cam, &f.light, f.row0, f.row1, f.rgb, f.depth, f.index,
                              f.argb, false))
        return rc;
      CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    } else if (f.whole_draw) {
      ctx->rast_n_tris = (int)c[24];
    }
  }
  float ms = 0.f;
  cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
  ctx->stats.gpu_ms = ms;
  if (ctx->timeline && ctx->pending && ctx->tl_n > 1) {
    for (int i = 1; i < ctx->tl_n; ++i) {
      float d = 0.f;
      cudaEventElapsedTime(&d, ctx->tl_ev[i - 1], ctx->tl_ev[i]);
      fprintf(stderr, "[b200 timeline] %-28s %8.1f us\n", ctx->tl_name[i], d * 1000.f);
    }
    fprintf(stderr, "[b200 timeline] frame %.1f us\n", ms * 1000.f);
  }
  if (ctx->pending == 1 || ctx->pending == 3) {
    if (ctx->pending == 1) ctx->stats.shadow_rays = c[0];   // a ray query (3) set its ray counts when it was enqueued
    ctx->stats.exact_evals = c[1];
    ctx->stats.prim_tests = (ctx->stats.primary_rays + ctx->stats.shadow_rays) *
                            (uint64_t)(ctx->rt_n_tris + ctx->rt_n_spheres);
  } else {
    ctx->stats.fragments = c[16];
    ctx->stats.bin_entries = c[3];
    // what this frame needed sizes the next pipelined frame of the same shape
    b200_ctx::RastSpec &sp = ctx->rast_spec;
    sp.tris = (unsigned long long)ctx->rast_n_tris;
    sp.rows = c[4]; sp.bins = c[3]; sp.big = c[10];
    sp.has_shadow = ctx->rast_has_shadow;
    sp.valid = 1;
  }
  ctx->pending = 0;
  return B200_OK;
}

// ---- sliced return of the packed framebuffer (see b200_ctx::copy_stream) ------------------
static void band_slices_begin(b200_ctx *ctx, uint32_t *host_row0, const uint32_t *dev_frame, int row0, int width) {
  ctx->slice_host = host_row0; ctx->slice_dev = dev_frame; ctx->slice_row0 = row0; ctx->slice_w = width;
  ctx->slice_n = 0;
}
// every slice copy is ordered before whatever is enqueued on ctx->stream next
static int band_slices_end(b200_ctx *ctx) {
  ctx->slice_host = nullptr;   // first: cleared even when the event calls below fail
  CU_CHECK(ctx, cudaEventRecord(ctx->ev_copied, ctx->copy_stream));
  CU_CHECK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_copied, 0));
  return B200_OK;
}

static int copy_out(b200_ctx *ctx, void *host, const void *dev, size_t bytes) {
  if (!host) return B200_OK;
  CU_CHECK(ctx, cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  return B200_OK;
}

int render_raytrace_band(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres,
                         int n_spheres, const camera_t *cam, const light_t *lights, int n_lights,
                         int row_begin, int row_end, float *rgb_out, float *depth_out,
                         int32_t *index_out) {
  if (!ctx) return B200_EINVAL;
  if (ctx->multi)
    return multi_raytrace(ctx, tris, n_tris, spheres, n_spheres, cam, lights, n_lights, row_begin, row_end, rgb_out,
                          depth_out, index_out, nullptr);
  if (int rc = check_camera(ctx, cam)) return rc;
  if (int rc = rt_upload_scene(ctx, tris, n_tris, spheres, n_spheres)) return rc;
  const size_t npix = (size_t)cam->width * cam->height;
  if (rgb_out) if (int rc = ensure(ctx, ctx->out_rgb, npix * 3 * sizeof(float))) return rc;
  if (depth_out) if (int rc = ensure(ctx, ctx->out_depth, npix * sizeof(float))) return rc;
  if (index_out) if (int rc = ensure(ctx, ctx->out_index, npix * sizeof(int32_t))) return rc;
  if (int rc = rt_frame_device(ctx, cam, lights, n_lights, row_begin, row_end,
                               rgb_out ? (float *)ctx->out_rgb.p : nullptr,
                               depth_out ? (float *)ctx->out_depth.p : nullptr,
                               index_out ? (int32_t *)ctx->out_index.p : nullptr, nullptr, 1, 0))
    return rc;
  const size_t off = (size_t)row_begin * cam->width, cnt = (size_t)(row_end - row_begin) * cam->width;
  if (int rc = copy_out(ctx, rgb_out, (float *)ctx->out_rgb.p + 3 * off, cnt * 3 * sizeof(float))) return rc;
  if (int rc = copy_out(ctx, depth_out, (float *)ctx->out_depth.p + off, cnt * sizeof(float))) return rc;
  if (int rc = copy_out(ctx, index_out, (int32_t *)ctx->out_index.p + off, cnt * sizeof(int32_t))) return rc;
  return finish_stats(ctx);
}

int render_raytrace(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres,
                    int n_spheres, const camera_t *cam, const light_t *lights, int n_lights,
                    float *rgb_out, float *depth_out, int32_t *index_out) {
  if (!ctx) return B200_EINVAL;
  if (int rc = check_camera(ctx, cam)) return rc;
  return render_raytrace_band(ctx, tris, n_tris, spheres, n_spheres, cam, lights, n_lights, 0, cam->height,
                              rgb_out, depth_out, index_out);
}

int draw_raytrace_band(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres,
                       int n_spheres, const camera_t *cam, const light_t *lights, int n_lights,
                       int row_begin, int row_end, uint32_t *argb_out) {
  if (!ctx) return B200_EINVAL;
  if (!argb_out) return ctx_fail(ctx, B200_EINVAL, "null framebuffer");
  if (ctx->multi)
    return multi_raytrace(ctx, tris, n_tris, spheres, n_spheres, cam, lights, n_lights, row_begin, row_end, nullptr,
                          nullptr, nullptr, argb_out);
  if (int rc = check_camera(ctx, cam)) return rc;
  if (int rc = rt_upload_scene(ctx, tris, n_tris, spheres, n_spheres)) return rc;
  const size_t npix = (size_t)cam->width * cam->height;
  if (int rc = ensure(ctx, ctx->out_argb, npix * sizeof(uint32_t))) return rc;
  RtFrame f;
  if (int rc = fill_frame(ctx, cam, lights, n_lights, row_begin, row_end, f)) return rc;
  if (ctx->rast_inflight.active) if (int rc = finish_stats(ctx)) return rc;   // the counters are shared
  ctx->stats.kernel_launches = 0;
  CU_CHECK(ctx, cudaMemsetAsync(ctx->counters.p, 0, 32 * sizeof(unsigned long long), ctx->stream));
  CU_CHECK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  ctx->tl_n = 0;
  tl_mark(ctx, "frame start");
  // Large frames are rendered in slices of whole 16-row blocks so that the copy of one slice to
  // the host overlaps the rendering of the next (scenes with per-frame grids: one slice, the
  // grids are built per launch).
  const int rows = row_end - row_begin;
  const bool gridded = ctx->opt_rt_grid == 1 || (ctx->opt_rt_grid == 0 && n_tris >= RT_GRID_AUTO_TRIS);
  const int k = (!gridded && (size_t)rows * cam->width >= B200_SLICE_MIN_PIXELS) ? B200_SLICES : 1;
  band_slices_begin(ctx, argb_out, (const uint32_t *)ctx->out_argb.p, row_begin, cam->width);
  int rc_loop = B200_OK;
  for (int i = 0; i < k && rc_loop == B200_OK; ++i) {
    RtFrame fi = f;
    fi.row0 = band_slice_edge(row_begin, rows, i, k, 16);
    fi.row1 = band_slice_edge(row_begin, rows, i + 1, k, 16);
    if (fi.row1 <= fi.row0) continue;
    rc_loop = rt_launch(ctx, fi, nullptr, nullptr, nullptr, (uint32_t *)ctx->out_argb.p);
    if (rc_loop == B200_OK && i + 1 == k && cudaEventRecord(ctx->ev1, ctx->stream) != cudaSuccess)
      rc_loop = ctx_fail(ctx, B200_ECUDA, "cudaEventRecord");
    if (rc_loop == B200_OK) rc_loop = band_slice_done(ctx, fi.row0, fi.row1);
  }
  if (rc_loop == B200_OK && rows <= 0 && cudaEventRecord(ctx->ev1, ctx->stream) != cudaSuccess)
    rc_loop = ctx_fail(ctx, B200_ECUDA, "cudaEventRecord");
  // always: clears slice_host, so that no later launch on this context copies into the caller's buffer
  const int rc_end = band_slices_end(ctx);
  if (rc_loop) return rc_loop;
  if (rc_end) return rc_end;
  ctx->stats.primary_rays = (uint64_t)f.W * (uint64_t)rows * 9u;
  if (int rc = enqueue_counter_readback(ctx)) return rc;
  ctx->pending = 1;
  return finish_stats(ctx);
}

int draw_raytrace(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres,
                  int n_spheres, const camera_t *cam, const light_t *lights, int n_lights,
                  uint32_t *argb_out) {
  if (!ctx) return B200_EINVAL;
  if (int rc = check_camera(ctx, cam)) return rc;
  return draw_raytrace_band(ctx, tris, n_tris, spheres, n_spheres, cam, lights, n_lights, 0, cam->height,
                            argb_out);
}

// ---- roofline denominator: FP32 FFMA peak of this GPU ------------------------------------
__global__ void b200_ffma_peak_kernel(float *out, int iters, float a, float b) {
  float x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
      x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}

int b200_measure_fp32_peak(b200_ctx *ctx, float *tflops_out) {
  if (!ctx || !tflops_out) return B200_EINVAL;
  SINGLE_ONLY(ctx);
  cudaSetDevice(ctx->device);
  if (int rc = finish_stats(ctx)) return rc;   // ev0 / ev1 still time a pending frame
  const int blocks = ctx->sm_count * 2, threads = 1024, iters = 4096;
  DevBuf tmp;
  if (int rc = ensure(ctx, tmp, sizeof(float) * (size_t)blocks * threads)) return rc;
  float best = 0.f;
  for (int rep = 0; rep < 4; ++rep) {
    cudaEventRecord(ctx->ev0, ctx->stream);
    b200_ffma_peak_kernel<<<blocks, threads, 0, ctx->stream>>>((float *)tmp.p, iters, 1.0001f, 0.5f);
    cudaEventRecord(ctx->ev1, ctx->stream);
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) { cudaFree(tmp.p); return ctx_fail(ctx, B200_ECUDA, "ffma peak"); }
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
    const double fl = 2.0 * 128.0 * iters * (double)blocks * threads;
    if (rep > 0 && ms > 0.f) best = fmaxf(best, (float)(fl / ms / 1e9));
  }
  cudaFree(tmp.p);
  *tflops_out = best;
  return B200_OK;
}

// ---- RAST -------------------------------------------------------------------------------

int rast_set_textures(b200_ctx *ctx, const rast_textures_t *tex) {
  if (!ctx) return B200_EINVAL;
  if (ctx->multi) return multi_rast_set_textures(ctx, tex);
  cudaSetDevice(ctx->device);
  if (ctx->pending == 2 || ctx->rast_inflight.active) if (int rc = finish_stats(ctx)) return rc;   // a frame in flight reads the old images
  ctx->rast_spec.valid = 0;
  if (!tex) { ctx->rast_tex_on = 0; return B200_OK; }
  // order of RastTex::img (rast_tex.cuh): bytes read per pixel, smallest edge
  const rast_image_t *im[8] = {&tex->marble, &tex->grill, &tex->grill_opacity, &tex->grill_normal,
                               &tex->woven, &tex->woven_occlusion, &tex->woven_opacity, &tex->woven_normal};
  const int elem[8] = {3, 3, 1, 3, 3, 1, 1, 3}, edge[8] = {2000, 1024, 1024, 1024, 1024, 1024, 1024, 1024};
  size_t off[8], total = 0;
  for (int k = 0; k < 8; ++k) {
    if (!im[k]->data || im[k]->rows < edge[k] || im[k]->cols < edge[k] || (long long)im[k]->step < (long long)im[k]->cols * elem[k])
      return ctx_fail(ctx, B200_EINVAL, "texture image missing, smaller than findU / findV address (2000 marble, 1024 others) or step < cols * element");
    off[k] = total;
    total += ((size_t)im[k]->rows * (size_t)im[k]->step + 255) & ~(size_t)255;
  }
  if (!tex->marble_noise || tex->marble_noise_len < 1) return ctx_fail(ctx, B200_EINVAL, "marble_noise missing");
  ctx->rast_tex_on = 0;   // until everything below has succeeded (the buffers may move: no stale pointers behind an error)
  if (int rc = ensure(ctx, ctx->rast_tex_images, total)) return rc;
  if (int rc = ensure(ctx, ctx->rast_tex_noise, (size_t)tex->marble_noise_len * sizeof(float4))) return rc;
  RastTex &t = ctx->rast_tex;
  for (int k = 0; k < 8; ++k) {
    t.img[k] = (const unsigned char *)ctx->rast_tex_images.p + off[k];
    t.step[k] = im[k]->step;
    CU_CHECK(ctx, cudaMemcpyAsync((void *)t.img[k], im[k]->data, (size_t)im[k]->rows * (size_t)im[k]->step, cudaMemcpyHostToDevice, ctx->stream));
  }
  t.marble_rows = tex->marble.rows;
  t.noise = (const float4 *)ctx->rast_tex_noise.p;
  t.noise_len = tex->marble_noise_len;
  CU_CHECK(ctx, cudaMemcpyAsync(ctx->rast_tex_noise.p, tex->marble_noise, (size_t)tex->marble_noise_len * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
  CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));   // the caller's arrays are free again on return
  ctx->rast_tex_on = 1;
  return B200_OK;
}

int rast_upload_clipped(b200_ctx *ctx, const rast_triangle *clipped, int n_tris) {
  if (!ctx) return B200_EINVAL;
  SINGLE_ONLY(ctx);
  if (n_tris < 0 || (n_tris > 0 && !clipped)) return ctx_fail(ctx, B200_EINVAL, "bad triangle list");
  cudaSetDevice(ctx->device);
  if (ctx->rast_inflight.active) if (int rc = finish_stats(ctx)) return rc;   // a re-render must see its own scene
  int has_shadow = 0;
  for (int i = 0; i < n_tris; ++i) {
    if (clipped[i].texture != 0 && !ctx->rast_tex_on) return ctx_fail(ctx, B200_EINVAL, "texture != 0 needs rast_set_textures");
    if (clipped[i].texture < 0 || clipped[i].texture > 3) return ctx_fail(ctx, B200_EINVAL, "texture must be 0..3");
    has_shadow |= !(clipped[i].color[0] >= 0);
  }
  ctx->rast_has_shadow = has_shadow;
  if (int rc = ensure(ctx, ctx->rast_src, sizeof(rast_triangle) * (size_t)(n_tris ? n_tris : 1))) return rc;
  if (n_tris) CU_CHECK(ctx, cudaMemcpyAsync(ctx->rast_src.p, clipped, sizeof(rast_triangle) * (size_t)n_tris,
                                            cudaMemcpyHostToDevice, ctx->stream));
  ctx->rast_n_tris = n_tris;
  return B200_OK;
}

// One raster frame: the triangle loop on the uploaded clipped list, or (whole_draw) the
// geometry stage first.  With allow_spec and a verified frame of the same shape behind
// it, the frame is enqueued without any host synchronisation (see common.cuh).
static int rast_frame(b200_ctx *ctx, bool whole_draw, const camera_t *cam, const rast_light_t *light, int row_begin,
                      int row_end, float *d_rgb, float *d_depth, int32_t *d_index, uint32_t *d_argb, bool allow_spec) {
  if (ctx->pending == 2) if (int rc = finish_stats(ctx)) return rc;   // settles a pipelined frame still in flight
  b200_ctx::RastSpec &sp = ctx->rast_spec;
  const int n_list = whole_draw ? -1 : ctx->rast_n_tris;
  const bool same = sp.valid && sp.whole_draw == (whole_draw ? 1 : 0) && sp.W == cam->width && sp.H == cam->height &&
                    sp.row0 == row_begin && sp.row1 == row_end && sp.ts == ctx->opt_rast_tile_log2 &&
                    sp.fast == ctx->opt_rast_path && sp.n_list == n_list && sp.cull == ctx->opt_rast_band_cull &&
                    (!whole_draw || (sp.n_room == ctx->rast_n_room && sp.n_boxes == ctx->rast_n_boxes));
  const bool spec = allow_spec && same && !ctx->opt_rast_colour;   // a colour-mode frame reads its fragment count back mid-frame
  sp.valid = 0;
  sp.whole_draw = whole_draw ? 1 : 0; sp.W = cam->width; sp.H = cam->height; sp.row0 = row_begin; sp.row1 = row_end;
  sp.ts = ctx->opt_rast_tile_log2; sp.fast = ctx->opt_rast_path; sp.n_list = n_list; sp.cull = ctx->opt_rast_band_cull;
  sp.n_room = ctx->rast_n_room; sp.n_boxes = ctx->rast_n_boxes;
  b200_ctx::RastInflight &f = ctx->rast_inflight;
  f.active = 0;
  if (spec) {
    if (whole_draw) ctx->rast_has_shadow = sp.has_shadow;   // checked against this frame's own flags later
    f.whole_draw = whole_draw ? 1 : 0;
    f.cam = *cam; f.light = *light; f.row0 = row_begin; f.row1 = row_end;
    f.rgb = d_rgb; f.depth = d_depth; f.index = d_index; f.argb = d_argb;
    f.cap_tris = 0; f.cap_bins = 0;
  }
  ctx->stats.kernel_launches = 0;
  CU_CHECK(ctx, cudaMemsetAsync(ctx->counters.p, 0, 32 * sizeof(unsigned long long), ctx->stream));
  CU_CHECK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  ctx->tl_n = 0;
  tl_mark(ctx, "frame start");
  rast_light_t lc = *light;
  ctx->rast_clear_ptr = nullptr; ctx->rast_keys_cleared = 0; ctx->rast_cull_on = 0; ctx->rast_geom_chunks = 1;
  // the path rast_launch will take, for the list bound a pipelined geometry stage writes under (that stage also
  // caps it at 2^30 - 1, which is past the scatter path's limit either way)
  const bool to_scatter = rast_scatter_path(ctx, whole_draw ? (long long)rast_spec_cap(sp.tris) : (long long)ctx->rast_n_tris);
  if (ctx->rast_up_chunks > 1) {
    if (spec && whole_draw && to_scatter) {
      ctx->rast_geom_chunks = ctx->rast_up_chunks;   // the frame consumes the upload chunk by chunk
    } else {                                        // any other frame: the whole scene first
      CU_CHECK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_up[ctx->rast_up_chunks - 1], 0));
    }
    ctx->rast_up_chunks = 1;
  }
  if (!whole_draw) ctx->rast_culled = 0;   // the caller's own list
  if (whole_draw) {
    if (spec && to_scatter) {
      // the frame is bound for the scatter path: its geometry kernel clears the key rows on the way
      const size_t W = (size_t)cam->width;
      const int fb0 = row_begin - 2 > 0 ? row_begin - 2 : 0, fb1 = row_end + 2 < cam->height ? row_end + 2 : cam->height;
      if (int rc = ensure(ctx, ctx->rast_keys, W * cam->height * sizeof(unsigned long long))) return rc;
      if (fb1 > fb0) {
        ctx->rast_clear_ptr = (unsigned long long *)ctx->rast_keys.p + (size_t)fb0 * W;
        ctx->rast_clear_bytes = (size_t)(fb1 - fb0) * W * sizeof(unsigned long long);
      }
      // ... and, asked to, keeps only the triangles that reach the band's rows.  (Not when the entry
      // value of the indirect light is in play: its one fragment is found on the complete list.)
      if (ctx->opt_rast_band_cull && !rast_indirect_entry_differs(light) && (fb0 > 0 || fb1 < cam->height)) {
        ctx->rast_cull_on = 1; ctx->rast_cull0 = fb0; ctx->rast_cull1 = fb1;
      }
    }
    if (int rc = rast_geometry(ctx, cam, light, &lc, spec)) return rc;
    if (spec) f.cap_tris = (unsigned long long)ctx->rast_n_tris;
  }
  if (int rc = rast_launch(ctx, cam, &lc, row_begin, row_end, d_rgb, d_depth, d_index, d_argb, spec)) return rc;
  CU_CHECK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  if (int rc = enqueue_counter_readback(ctx)) return rc;
  f.active = spec ? 1 : 0;
  ctx->pending = 2;
  return B200_OK;
}

static int rast_check_frame_args(b200_ctx *ctx, const camera_t *cam, const rast_light_t *light, int row_begin,
                                 int row_end) {
  if (int rc = check_camera(ctx, cam)) return rc;
  if (!light) return ctx_fail(ctx, B200_EINVAL, "null light");
  if (row_begin < 0 || row_end > cam->height || row_begin > row_end) return ctx_fail(ctx, B200_EINVAL, "bad row band");
  cudaSetDevice(ctx->device);
  return B200_OK;
}

int rast_render_device(b200_ctx *ctx, const camera_t *cam, const rast_light_t *light, int row_begin,
                       int row_end, float *d_rgb, float *d_depth, int32_t *d_index, uint32_t *d_argb) {
  if (!ctx) return B200_EINVAL;
  SINGLE_ONLY(ctx);
  if (int rc = rast_check_frame_args(ctx, cam, light, row_begin, row_end)) return rc;
  return rast_frame(ctx, false, cam, light, row_begin, row_end, d_rgb, d_depth, d_index, d_argb,
                    ctx->opt_rast_pipelined != 0);
}

static int raster_host_outputs(b200_ctx *ctx, const camera_t *cam, float *rgb_out, float *depth_out,
                               int32_t *index_out, uint32_t *argb_out) {
  const size_t npix = (size_t)cam->width * cam->height;
  if (rgb_out) if (int rc = ensure(ctx, ctx->out_rgb, npix * 3 * sizeof(float))) return rc;
  if (depth_out) if (int rc = ensure(ctx, ctx->out_depth, npix * sizeof(float))) return rc;
  if (index_out) if (int rc = ensure(ctx, ctx->out_index, npix * sizeof(int32_t))) return rc;
  if (argb_out) if (int rc = ensure(ctx, ctx->out_argb, npix * sizeof(uint32_t))) return rc;
  return B200_OK;
}

int render_raster_clipped(b200_ctx *ctx, const rast_triangle *clipped, int n_tris, const camera_t *cam,
                          const rast_light_t *light, float *rgb_out, float *depth_out, int32_t *index_out) {
  if (!ctx) return B200_EINVAL;
  SINGLE_ONLY(ctx);
  if (int rc = check_camera(ctx, cam)) return rc;
  if (int rc = rast_upload_clipped(ctx, clipped, n_tris)) return rc;
  if (int rc = raster_host_outputs(ctx, cam, rgb_out, depth_out, index_out, nullptr)) return rc;
  if (int rc = rast_check_frame_args(ctx, cam, light, 0, cam->height)) return rc;
  if (int rc = rast_frame(ctx, false, cam, light, 0, cam->height, rgb_out ? (float *)ctx->out_rgb.p : nullptr,
                          depth_out ? (float *)ctx->out_depth.p : nullptr,
                          index_out ? (int32_t *)ctx->out_index.p : nullptr, nullptr, true))
    return rc;
  if (ctx->rast_inflight.active) if (int rc = finish_stats(ctx)) return rc;   // verified before anything leaves
  const size_t npix = (size_t)cam->width * cam->height;
  if (int rc = copy_out(ctx, rgb_out, ctx->out_rgb.p, npix * 3 * sizeof(float))) return rc;
  if (int rc = copy_out(ctx, depth_out, ctx->out_depth.p, npix * sizeof(float))) return rc;
  if (int rc = copy_out(ctx, index_out, ctx->out_index.p, npix * sizeof(int32_t))) return rc;
  return finish_stats(ctx);
}

// ---- RAST tier 2: the whole Draw (geometry stage + triangle loop + post pass) ----------

int rast_upload_scene(b200_ctx *ctx, const rast_triangle *room, int n_room, const rast_triangle *boxes,
                      int n_boxes) {
  if (!ctx) return B200_EINVAL;
  SINGLE_ONLY(ctx);
  if (n_room < 0 || n_boxes < 0 || (n_room > 0 && !room) || (n_boxes > 0 && !boxes))
    return ctx_fail(ctx, B200_EINVAL, "bad scene arguments");
  if ((long long)n_room + 7ll * n_boxes > 0x3fffffffll) return ctx_fail(ctx, B200_EINVAL, "scene too large");
  cudaSetDevice(ctx->device);
  if (ctx->rast_inflight.active) if (int rc = finish_stats(ctx)) return rc;   // a re-render must see its own scene
  // texture != 0 and shadow-coloured input triangles are detected by the geometry
  // kernel on the device (no host pass over the triangles)
  ctx->rast_has_shadow = n_boxes > 0;   // createShadowVolume wraps every box triangle (:215)
  const size_t n = (size_t)n_room + (size_t)n_boxes;
  if (int rc = ensure(ctx, ctx->rast_world, sizeof(rast_triangle) * (n ? n : 1))) return rc;
  rast_triangle *d = (rast_triangle *)ctx->rast_world.p;
  ctx->rast_up_chunks = 1;
  if (ctx->rast_chunk_next_upload && n_boxes == 0 && (size_t)n_room * sizeof(rast_triangle) >= ((size_t)16 << 20)) {
    // a frame follows at once (host-pointer entries): the list travels in chunks on the copy stream,
    // and that frame's geometry / scatter work on chunk k while chunk k + 1 is on the link
    CU_CHECK(ctx, cudaEventRecord(ctx->ev_main, ctx->stream));
    CU_CHECK(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_main, 0));
    for (int c = 0; c <= RAST_UP_CHUNKS; ++c)
      ctx->rast_up_edge[c] = c == RAST_UP_CHUNKS ? n_room : (int)((long long)n_room * c / RAST_UP_CHUNKS) / 128 * 128;
    for (int c = 0; c < RAST_UP_CHUNKS; ++c) {
      const size_t a = (size_t)ctx->rast_up_edge[c], b = (size_t)ctx->rast_up_edge[c + 1];
      if (b > a) CU_CHECK(ctx, cudaMemcpyAsync(d + a, room + a, sizeof(rast_triangle) * (b - a), cudaMemcpyHostToDevice, ctx->copy_stream));
      CU_CHECK(ctx, cudaEventRecord(ctx->ev_up[c], ctx->copy_stream));
    }
    ctx->rast_up_chunks = RAST_UP_CHUNKS;
  } else {
    if (n_room) CU_CHECK(ctx, cudaMemcpyAsync(d, room, sizeof(rast_triangle) * (size_t)n_room, cudaMemcpyHostToDevice, ctx->stream));
    if (n_boxes) CU_CHECK(ctx, cudaMemcpyAsync(d + n_room, boxes, sizeof(rast_triangle) * (size_t)n_boxes, cudaMemcpyHostToDevice, ctx->stream));
  }
  ctx->rast_chunk_next_upload = 0;
  ctx->rast_n_room = n_room;
  ctx->rast_n_boxes = n_boxes;
  return B200_OK;
}

int rast_draw_device(b200_ctx *ctx, const camera_t *cam, const rast_light_t *light, int row_begin, int row_end,
                     float *d_rgb, float *d_depth, int32_t *d_index, uint32_t *d_argb) {
  if (!ctx) return B200_EINVAL;
  SINGLE_ONLY(ctx);
  if (int rc = rast_check_frame_args(ctx, cam, light, row_begin, row_end)) return rc;
  return rast_frame(ctx, true, cam, light, row_begin, row_end, d_rgb, d_depth, d_index, d_argb,
                    ctx->opt_rast_pipelined != 0);
}

}  // extern "C"

// Rows [row_begin, row_end) of the whole Draw on the scene already uploaded to this context,
// into band-sized HOST buffers.  With only the packed frame asked for, the rows leave for the
// host slice by slice while the next slice is resolved.
int rast_band_resident(b200_ctx *ctx, const camera_t *cam, const rast_light_t *light, int row_begin, int row_end,
                       float *rgb_out, float *depth_out, int32_t *index_out, uint32_t *argb_out) {
  if (int rc = check_camera(ctx, cam)) return rc;
  if (int rc = raster_host_outputs(ctx, cam, rgb_out, depth_out, index_out, argb_out)) return rc;
  if (int rc = rast_check_frame_args(ctx, cam, light, row_begin, row_end)) return rc;
  const size_t off = (size_t)row_begin * cam->width, cnt = (size_t)(row_end - row_begin) * cam->width;
  const bool sliced = argb_out && !rgb_out && !depth_out && !index_out;
  if (sliced) band_slices_begin(ctx, argb_out, (const uint32_t *)ctx->out_argb.p, row_begin, cam->width);
  const int rc_frame = rast_frame(ctx, true, cam, light, row_begin, row_end, rgb_out ? (float *)ctx->out_rgb.p : nullptr,
                                  depth_out ? (float *)ctx->out_depth.p : nullptr,
                                  index_out ? (int32_t *)ctx->out_index.p : nullptr,
                                  argb_out ? (uint32_t *)ctx->out_argb.p : nullptr, true);
  if (sliced) if (int rc = band_slices_end(ctx)) return rc;
  if (rc_frame) return rc_frame;
  const uint64_t twice = ctx->stats.respeculated;
  if (int rc = finish_stats(ctx)) return rc;     // verifies a pipelined frame; renders it again if it outgrew its guess
  if (sliced && ctx->stats.respeculated == twice) return B200_OK;   // every row already left with its slice
  if (int rc = copy_out(ctx, rgb_out, (float *)ctx->out_rgb.p + 3 * off, cnt * 3 * sizeof(float))) return rc;
  if (int rc = copy_out(ctx, depth_out, (float *)ctx->out_depth.p + off, cnt * sizeof(float))) return rc;
  if (int rc = copy_out(ctx, index_out, (int32_t *)ctx->out_index.p + off, cnt * sizeof(int32_t))) return rc;
  if (int rc = copy_out(ctx, argb_out, (uint32_t *)ctx->out_argb.p + off, cnt * sizeof(uint32_t))) return rc;
  return finish_stats(ctx);
}

extern "C" {

int render_raster_band(b200_ctx *ctx, const rast_triangle *room, int n_room, const rast_triangle *boxes, int n_boxes,
                       const camera_t *cam, const rast_light_t *light, int row_begin, int row_end, float *rgb_out,
                       float *depth_out, int32_t *index_out) {
  if (!ctx) return B200_EINVAL;
  if (ctx->multi)
    return multi_raster(ctx, room, n_room, boxes, n_boxes, cam, light, row_begin, row_end, rgb_out, depth_out, index_out, nullptr);
  if (int rc = check_camera(ctx, cam)) return rc;
  ctx->rast_chunk_next_upload = 1;
  if (int rc = rast_upload_scene(ctx, room, n_room, boxes, n_boxes)) return rc;
  return rast_band_resident(ctx, cam, light, row_begin, row_end, rgb_out, depth_out, index_out, nullptr);
}

int render_raster(b200_ctx *ctx, const rast_triangle *room, int n_room, const rast_triangle *boxes, int n_boxes,
                  const camera_t *cam, const rast_light_t *light, float *rgb_out, float *depth_out,
                  int32_t *index_out) {
  if (!ctx) return B200_EINVAL;
  if (int rc = check_camera(ctx, cam)) return rc;
  return render_raster_band(ctx, room, n_room, boxes, n_boxes, cam, light, 0, cam->height, rgb_out, depth_out, index_out);
}

int draw_raster_band(b200_ctx *ctx, const rast_triangle *room, int n_room, const rast_triangle *boxes,
                     int n_boxes, const camera_t *cam, const rast_light_t *light, int row_begin, int row_end,
                     uint32_t *argb_out) {
  if (!ctx) return B200_EINVAL;
  if (!argb_out) return ctx_fail(ctx, B200_EINVAL, "null framebuffer");
  if (ctx->multi)
    return multi_raster(ctx, room, n_room, boxes, n_boxes, cam, light, row_begin, row_end, nullptr, nullptr, nullptr, argb_out);
  if (int rc = check_camera(ctx, cam)) return rc;
  ctx->rast_chunk_next_upload = 1;
  if (int rc = rast_upload_scene(ctx, room, n_room, boxes, n_boxes)) return rc;
  return rast_band_resident(ctx, cam, light, row_begin, row_end, nullptr, nullptr, nullptr, argb_out);
}

int draw_raster(b200_ctx *ctx, const rast_triangle *room, int n_room, const rast_triangle *boxes, int n_boxes,
                const camera_t *cam, const rast_light_t *light, uint32_t *argb_out) {
  if (!ctx) return B200_EINVAL;
  if (int rc = check_camera(ctx, cam)) return rc;
  return draw_raster_band(ctx, room, n_room, boxes, n_boxes, cam, light, 0, cam->height, argb_out);
}

int raster_read_clipped(b200_ctx *ctx, rast_triangle *out, int cap, int *n_out) {
  if (!ctx || !n_out) return B200_EINVAL;
  SINGLE_ONLY(ctx);
  if (int rc = finish_stats(ctx)) return rc;
  *n_out = ctx->rast_n_tris;
  const int n = ctx->rast_n_tris < cap ? ctx->rast_n_tris : cap;
  if (out && n > 0) CU_CHECK(ctx, cudaMemcpy(out, ctx->rast_src.p, sizeof(rast_triangle) * (size_t)n, cudaMemcpyDeviceToHost));
  return B200_OK;
}

int raster_read_buffers(b200_ctx *ctx, float *screen_out, float *low_out, float *high_out, int32_t *shadow_out) {
  if (!ctx) return B200_EINVAL;
  SINGLE_ONLY(ctx);
  if (ctx->rast_w <= 0)
    return ctx_fail(ctx, B200_EINVAL, "no intermediate buffers: nothing rendered yet, or the last frame took the "
                                      "scatter path (set B200_OPT_RAST_PATH to 1 to keep them)");
  const size_t npix = (size_t)ctx->rast_w * ctx->rast_h;
  if (int rc = finish_stats(ctx)) return rc;
  if (screen_out) CU_CHECK(ctx, cudaMemcpy(screen_out, ctx->rast_screen.p, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost));
  if (low_out) CU_CHECK(ctx, cudaMemcpy(low_out, ctx->rast_low.p, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost));
  if (high_out) CU_CHECK(ctx, cudaMemcpy(high_out, ctx->rast_high.p, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost));
  if (shadow_out) CU_CHECK(ctx, cudaMemcpy(shadow_out, ctx->rast_shadow.p, npix * sizeof(int32_t), cudaMemcpyDeviceToHost));
  return B200_OK;
}

// ---- headless framebuffer -------------------------------------------------------------

void b200_quantise(const float *rgb, size_t n_pixels, uint32_t *argb_out) {
  for (size_t i = 0; i < n_pixels; ++i) argb_out[i] = put_pixel_argb(rgb[3 * i], rgb[3 * i + 1], rgb[3 * i + 2]);
}

// 32-bpp BMP with a BITMAPV4-style header and ARGB masks, rows bottom-up: the
// layout SDL_SaveBMP writes for the ARGB8888 surface the reference builds in
// SDL_SaveImage (SDLauxiliary.h:24-53); pixel bytes are identical.
int b200_save_bmp(const char *path, const uint32_t *argb, int width, int height) {
  if (!path || !argb || width <= 0 || height <= 0) return B200_EINVAL;
  FILE *f = fopen(path, "wb");
  if (!f) return B200_EINVAL;
  const uint32_t hdr = 14, info = 108, off = hdr + info;
  const uint32_t img = (uint32_t)width * (uint32_t)height * 4u;
  unsigned char h[122];
  memset(h, 0, sizeof h);
  auto put32 = [&](int at, uint32_t v) { h[at] = v & 255; h[at + 1] = (v >> 8) & 255; h[at + 2] = (v >> 16) & 255; h[at + 3] = (v >> 24) & 255; };
  auto put16 = [&](int at, uint32_t v) { h[at] = v & 255; h[at + 1] = (v >> 8) & 255; };
  h[0] = 'B'; h[1] = 'M';
  put32(2, off + img); put32(10, off);
  put32(14, info); put32(18, (uint32_t)width); put32(22, (uint32_t)height);
  put16(26, 1); put16(28, 32); put32(30, 3 /* BI_BITFIELDS */); put32(34, img);
  put32(38, 2835); put32(42, 2835);
  put32(54, 0x00FF0000u); put32(58, 0x0000FF00u); put32(62, 0x000000FFu); put32(66, 0xFF000000u);
  put32(70, 0x57696E20u);  // 'Win ' colour space
  bool ok = fwrite(h, 1, off, f) == off;
  for (int y = height - 1; y >= 0 && ok; --y)
    ok = fwrite(argb + (size_t)y * width, 4, (size_t)width, f) == (size_t)width;
  fclose(f);
  return ok ? B200_OK : B200_EINVAL;
}

}  // extern "C"

// Raw device counters of the last render (diagnostics; not part of the public header).
extern "C" int b200_debug_counters(b200_ctx *ctx, unsigned long long *out8) {
  if (!ctx || !out8) return B200_EINVAL;
  CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
  CU_CHECK(ctx, cudaMemcpy(out8, ctx->counters.p, 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return B200_OK;
}

// List length of every direction-grid cell of the last gridded RT frame (diagnostics).
extern "C" int b200_debug_rt_cells(b200_ctx *ctx, unsigned *out, int cap, int *n_cells, int *n_cam_cells) {
  if (!ctx || !n_cells || !n_cam_cells) return B200_EINVAL;
  CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
  *n_cells = (int)ctx->rt_n_cells; *n_cam_cells = (int)ctx->rt_n_cam_cells;
  const size_t n = ctx->rt_n_cells < (size_t)cap ? ctx->rt_n_cells : (size_t)cap;
  if (out && n) CU_CHECK(ctx, cudaMemcpy(out, ctx->rt_cells.p, n * sizeof(unsigned), cudaMemcpyDeviceToHost));
  return B200_OK;
}
