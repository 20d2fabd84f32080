// Shared device helpers and the context object behind include/b200render.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>
#include <functional>
#include <string>
#include <vector>

#include "../../include/b200render.h"

// ---- strictly-rounded arithmetic ---------------------------------------------
// The reference is built without FMA contraction (raytracer/Makefile:15: g++ -O3,
// no -march), so every product and sum below is rounded on its own.  These
// wrappers stop nvcc from fusing them; they compile to plain FMUL/FADD/FFMA-free
// SASS.  Division and square root are the IEEE-exact variants.
__device__ __forceinline__ float xmul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float xadd(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float xsub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float xdiv(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ float xsqrt(float a) { return __fsqrt_rn(a); }
// a / den for a finite den > 0: a zero numerator (an edge with dx = 0, a row whose two ends are the
// same sample, ...) sends the whole warp through __fdiv_rn's slow path (ncu: 13 % of the small-
// triangle kernel's instructions at 9 of 32 lanes); 0 / den = a exactly, sign included.
__device__ __forceinline__ float xdiv_pos(float a, float den) { return a == 0.0f ? a : __fdiv_rn(a, den); }
// On x86 an invalid operation (0 * inf, inf - inf, 0 / 0) yields the indefinite NaN 0xffc00000 and later
// operations pass it on unchanged; here it yields 0x7fffffff.  Outputs whose every NaN begins as such an operation
// store it as the reference's bits (the rasteriser's clipped list, DESIGN §4.1; rt_direct_light, §3.4).
__device__ __forceinline__ float x86_nan(float v) { return v != v ? __int_as_float(0xffc00000) : v; }

// IEEE-exact x / C for the constants the reference divides by (5, 3, 9):
// q = x*rc; r = fma(-C, q, x); q' = fma(r, rc, q) with rc = RN(1/C) is the
// correctly rounded quotient for EVERY finite x except -0.0 (sign of zero);
// checked exhaustively over all 2^32 inputs by oracle/tools/check_constdiv.c.
template <int C>
__device__ __forceinline__ float xdiv_const(float x) {
  constexpr float c = (float)C, rc = 1.0f / (float)C;
  const float q = __fmul_rn(x, rc);
  const float r = __fmaf_rn(-c, q, x);
  const float v = __fmaf_rn(r, rc, q);
  return (x == 0.0f || !(fabsf(x) < INFINITY)) ? x : v;   // +-0, +-inf and NaN divide to themselves
}

// glm::determinant(mat3) with columns a, b, c
// (glm/glm/detail/func_matrix.inl:235-238), one rounding per operation.
__device__ __forceinline__ float xdet3(float ax, float ay, float az, float bx, float by, float bz,
                                       float cx, float cy, float cz) {
  float c0 = xsub(xmul(by, cz), xmul(cy, bz));
  float c1 = xsub(xmul(ay, cz), xmul(cy, az));
  float c2 = xsub(xmul(ay, bz), xmul(by, az));
  return xadd(xsub(xmul(ax, c0), xmul(bx, c1)), xmul(cx, c2));
}

// glm::dot(vec3) (glm/glm/detail/func_geometric.inl:65-73)
__device__ __forceinline__ float xdot3(float ax, float ay, float az, float bx, float by, float bz) {
  return xadd(xadd(xmul(ax, bx), xmul(ay, by)), xmul(az, bz));
}

// PutPixelSDL (raytracer/Source/SDLauxiliary.h:149-161): clamp(255*c, 0, 255),
// truncate, pack 0x80RRGGBB.
__host__ __device__ __forceinline__ uint32_t put_pixel_argb(float r, float g, float b) {
  float c[3] = {r, g, b};
  uint32_t ch[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float v = 255.0f * c[k];
    v = v < 0.f ? 0.f : v;
    v = v > 255.f ? 255.f : v;
    ch[k] = (uint32_t)v;
  }
  return (128u << 24) + (ch[0] << 16) + (ch[1] << 8) + ch[2];
}

// ---- context -------------------------------------------------------------------
#define B200_SLICES 4
// Bands below this many pixels come back in one piece: four launches of a quarter of a ~1 Mpixel band (what one of
// eight GPUs gets of a 4K frame) leave most of the GPU idle in each -- measured 0.15 -> 0.30 ms per band -- and
// made the adaptive bands of a multi-GPU context oscillate around the threshold.
#define B200_SLICE_MIN_PIXELS ((size_t)3 << 20)
constexpr int RAST_UP_CHUNKS = 4;   // a large raster scene travels to the device in this many chunks (draw_raster_band)
struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
};

struct b200_multi;   // multi.cu
// Texture state of the rasteriser (rast_set_textures; device pointers; see rast_tex.cuh)
struct RastTex {
  const unsigned char *img[8];
  int step[8];
  int marble_rows;             // normalMap_marble is indexed y * marble.rows + x (:593)
  const float4 *noise;
  long long noise_len;
  float cam[4];                // cameraPos
  float Rinv[16];              // glm::inverse(R), column-major
  int use_rinv;                // the reference's "yaw != 0" (:1761): R is not the identity
};

struct b200_ctx {
  b200_multi *multi = nullptr;        // set on a context made by b200_init_multi: it only fans out to one ordinary context per device
  int device = 0;
  cudaStream_t stream = nullptr;      // where work is enqueued (own_stream unless overridden)
  cudaStream_t own_stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  // Host-pointer entries return the packed framebuffer in slices: while the kernels render
  // slice i + 1, slice i travels to the host on a second stream (band_begin .. band_slice_done).
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_slice[B200_SLICES] = {}, ev_copied = nullptr;
  // Chunked scene upload of the host-pointer raster entries: chunk k is copied on copy_stream, the
  // single-pass geometry kernel runs per chunk behind its copy, and the scatter of chunk k runs on
  // aux_stream while chunk k + 1 is still on the link.
  cudaStream_t aux_stream = nullptr;
  cudaEvent_t ev_up[RAST_UP_CHUNKS] = {}, ev_chunk[RAST_UP_CHUNKS] = {}, ev_join = nullptr, ev_main = nullptr;
  int rast_chunk_next_upload = 0;   // set by the host-pointer entries: the next rast_upload_scene may travel in chunks
  int rast_up_chunks = 1, rast_up_edge[RAST_UP_CHUNKS + 1] = {};   // chunks of the upload in flight; their first triangles (multiples of 128)
  int rast_geom_chunks = 1, rast_geom_chunk_tris[RAST_UP_CHUNKS] = {};   // of the frame being enqueued
  uint32_t *slice_host = nullptr;       // destination of row `slice_row0`; null = no sliced copy in progress
  const uint32_t *slice_dev = nullptr;  // device frame (full-frame addressing)
  int slice_row0 = 0, slice_w = 0, slice_n = 0;
  std::string err;
  b200_stats stats{};
  int opt_rt_bruteforce = 0;
  int opt_rast_tile_log2 = 5;
  int sm_count = 148;

  // RT scene (device)
  DevBuf rt_src;      // rt_triangle[n] as uploaded (normal/colour gathered from here)
  DevBuf rt_geom;     // float4[3n]: v0, e1, e2 for the exact test
  DevBuf rt_spheres;  // rt_sphere[n]
  DevBuf rt_planes;   // float4[..]: per-origin edge-function planes for the filter
  DevBuf rt_dtcam;    // float[n]: per-frame numerator of t for primary rays (batched views: [views][n])
  DevBuf rt_selfD;    // float[lights][n]: per-frame sign and bound of D for a shadow ray on its own triangle
  DevBuf rt_bounds;   // two words: coordinate / normal bounds of a large scene, reduced on the device
  int rt_bounds_on_device = 0;
  DevBuf rt_cells;    // direction grids: per-cell counts, cursors, padded counts, offsets, scan scratch
  DevBuf rt_cell_rec, rt_cell_idx;   // the cells' lists: plane records and triangle indices
  DevBuf rt_query;   // host-pointer ray queries: rays or hits, limits and results (rt_closest_hits, rt_occluded, rt_direct_light)
  DevBuf rt_plan;                    // gridded frames: two per-block cost arrays, the block plan, its length (rt_plan_kernel)
  unsigned long long rt_plan_shape = 0;
  int rt_plan_valid = 0, rt_plan_flip = 0;
  int opt_rt_plan = 1;               // B200_OPT_RT_PLAN
  int rt_plan_heavy = 0;             // b200_debug_rt_plan_heavy (0: RT_PLAN_HEAVY)
  DevBuf rt_cell_pairs;              // (cell, record) pairs written down by the counting pass
  unsigned long long rt_grid_pairs_seen = 0;   // pairs (or list entries) of the last gridded frame, of a scene of ...
  int rt_grid_pairs_n = 0;                     // ... this many triangles
  size_t rt_n_cells = 0, rt_n_cam_cells = 0;   // of the last gridded frame (diagnostics)
  int rt_grid_smem_set = 0;                    // the grid kernels' dynamic shared-memory limit has been raised
  int opt_rt_il_n = 1, opt_rt_il_r = 0;        // row-block interleave of rt_render_device (see the header)
  int opt_rt_grid = 0;               // 0 auto (scenes of RT_GRID_AUTO_TRIS triangles or more), 1 always, 2 never
  int rt_n_tris = 0, rt_n_spheres = 0;
  float rt_world_abs = 0.f;   // max |coordinate| over the uploaded scene
  float rt_normal_abs = 1.f;  // max(1, max |normal component|): scales the 1e-5 * normal shadow-ray offset (:394)
  int pending = 0;            // 1 = RT frame or direct-light query, 2 = RAST render, 3 = RT ray query whose counters are
                              // not read back yet

  // RAST scene (device)
  DevBuf rast_src;    // rast_triangle[n] clipped list
  int rast_n_tris = 0;
  DevBuf rast_setup, rast_rowsA, rast_rowsB, rast_bins, rast_tile_count, rast_tmp, rast_tile_bits;
  DevBuf rast_keys;      // fast path: 64-bit (zinv, triangle) key per pixel
  int opt_rast_band_cull = 0;        // B200_OPT_RAST_BAND_CULL
  int rast_cull_on = 0, rast_cull0 = 0, rast_cull1 = 0;   // this frame's geometry stage should keep only rows [cull0, cull1) ...
  int rast_culled = 0;               // ... and did: rast_src is the band's list, rast_orig its indices in the complete list
  DevBuf rast_orig;
  void *rast_clear_ptr = nullptr;    // key rows the single-pass geometry kernel should clear (set per frame by rast_frame)
  size_t rast_clear_bytes = 0;
  int rast_keys_cleared = 0;         // ... and whether it did (rast_launch then skips its memset)
  DevBuf rast_shadow8;               // ordered path, fused: shadowBuffer as one byte per pixel
  DevBuf rast_srowsB, rast_srowsL;   // fast path: row records of the small triangles
  DevBuf rast_trimeta, rast_big;   // fast path: per-triangle row-table origin; list of the triangles too big for the small-triangle kernel
  int rast_has_shadow = 0;   // the uploaded list can contain shadow-volume triangles
  int rast_tex_on = 0;       // rast_set_textures: texture / index fields are honoured, frames take the ordered path
  RastTex rast_tex{};
  DevBuf rast_tex_images, rast_tex_noise;
  int opt_rast_colour = 0;   // B200_OPT_RAST_COLOUR_MODE: randColourSelect (0, 1 random colours, 2 night vision)
  DevBuf rast_colour_keys, rast_colour_rgb, rast_colour_tmp;
  int opt_rast_path = 0;     // 0 auto, 1 ordered tiles, 2 scatter (shadow-free lists only)
  DevBuf rast_row_owner;   // per slot of the row tables: the triangle that owns it (RastParams::row_owner)
  DevBuf rast_world;     // tier 2: world-space room then boxes, as uploaded
  DevBuf rast_geom_tmp;  // tier 2: per-triangle output counts and their scan
  int rast_n_room = 0, rast_n_boxes = 0;
  DevBuf rast_screen, rast_low, rast_high, rast_shadow, rast_depth, rast_index;
  int rast_w = 0, rast_h = 0;

  // Pipelined raster frames (B200_OPT_RAST_PIPELINED): buffer sizes and grids come from
  // the last verified frame of the same shape instead of two mid-frame read-backs; the
  // frame's own counters are checked when it is waited for and a frame that outgrew the
  // guess is re-rendered synchronously before anything is handed out.
  int opt_rast_pipelined = 0;
  struct RastSpec {
    int valid = 0, has_shadow = 0, n_room = 0, n_boxes = 0, n_list = 0, W = 0, H = 0, row0 = 0, row1 = 0, fast = 0, ts = 0, whole_draw = 0, cull = 0;
    unsigned long long tris = 0, rows = 0, bins = 0, big = 0;
  } rast_spec;
  struct RastInflight {
    int active = 0, whole_draw = 0, fast = 0;
    camera_t cam;
    rast_light_t light;
    int row0 = 0, row1 = 0;
    float *rgb = nullptr, *depth = nullptr;
    int32_t *index = nullptr;
    uint32_t *argb = nullptr;
    unsigned long long cap_tris = 0, cap_bins = 0;
  } rast_inflight;

  // outputs / staging (device) used by the host-pointer entry points
  DevBuf out_rgb, out_depth, out_index, out_argb;
  // diagnostics (environment B200_TIMELINE=1): an event after every launch, printed by finish_stats
  int timeline = 0, tl_n = 0;
  cudaEvent_t tl_ev[64] = {};
  const char *tl_name[64] = {};
  DevBuf counters;    // unsigned long long[32]
  void *pinned = nullptr;
  size_t pinned_cap = 0;
};

int ctx_fail(b200_ctx *ctx, int code, const char *what, cudaError_t e = cudaSuccess);
int ensure(b200_ctx *ctx, DevBuf &b, size_t bytes);

#define CU_CHECK(ctx, call)                                          \
  do {                                                               \
    cudaError_t e__ = (call);                                        \
    if (e__ != cudaSuccess) return ctx_fail(ctx, B200_ECUDA, #call, e__); \
  } while (0)

// ---- kernels' host launchers (defined in rt_kernels.cu / rast_kernels.cu) ------
struct RtFrame {
  float cam[4];
  float focal;
  float R[16];
  int W, H, row0, row1;
  int il_n, il_r;      // this launch renders the 16-row blocks b of [row0, row1) with b % il_n == il_r
  int n_lights;
  float lights[8][7];  // pos[4], colour[3]
};
#define B200_MAX_LIGHTS 8
// The caller's per-pixel sample pattern (render_raytrace_samples): sample k of a pixel is the ray along
// (dir.x + off[2k], dir.y + off[2k+1], f), k < n; depth / index are those of sample depth_sample.  A kernel
// parameter of its own (__grid_constant__), so that RtKParams -- and every other kernel -- stays as it is.
struct RtSamplesParams {
  int n;
  int depth_sample;
  float off[2 * B200_RT_MAX_SAMPLES];
};
constexpr int RT_GRID_AUTO_TRIS = 1024;   // B200_OPT_RT_GRID = 0: scenes this large get direction grids

// spec = true: pipelined (no host synchronisation; see b200_ctx::rast_spec)
int rast_colour_sort(b200_ctx *ctx, const unsigned long long *in, unsigned long long *out, unsigned long long n, int end_bit);   // rast_colour.cu
int rast_launch(b200_ctx *ctx, const camera_t *cam, const rast_light_t *light, int row0, int row1,
                float *d_rgb, float *d_depth, int32_t *d_index, uint32_t *d_argb, bool spec);
int rast_geometry(b200_ctx *ctx, const camera_t *cam, const rast_light_t *light, rast_light_t *light_out,
                  bool spec);
// true: the frame takes the scatter path, false: ordered screen tiles (n: the list length or a bound on it)
bool rast_scatter_path(const b200_ctx *ctx, long long n);
static inline unsigned long long rast_spec_cap(unsigned long long seen) { return seen + seen / 32 + 1024; }   // +3 %
// PixelShader leaves indirectLightPowerPerArea at 0.2 (:585): whether a Draw is entered with another value, which
// then reaches its first shaded fragment
static inline bool rast_indirect_entry_differs(const rast_light_t *light) {
  const float steady = 0.2f * 1.0f;
  for (int k = 0; k < 3; ++k)
    if (memcmp(&light->indirect[k], &steady, sizeof steady)) return true;
  return false;
}
int scan_exclusive(b200_ctx *ctx, const unsigned *counts, unsigned *offs, int n, unsigned *tmp,
                   unsigned long long *total_out);   // rast_geom.cu; tmp: n / 4096 + 2 words
int rt_prepare_scene(b200_ctx *ctx);
static inline void tl_mark(b200_ctx *ctx, const char *name) {
  if (!ctx->timeline || ctx->tl_n >= 64) return;
  if (!ctx->tl_ev[ctx->tl_n]) cudaEventCreate(&ctx->tl_ev[ctx->tl_n]);
  cudaEventRecord(ctx->tl_ev[ctx->tl_n], ctx->stream);
  ctx->tl_name[ctx->tl_n++] = name;
}
// rows [a, b) of the packed frame are final on ctx->stream: start their copy to the host (no-op unless sliced)
int band_slice_done(b200_ctx *ctx, int a, int b);
// slice boundaries of a band of `rows` rows split k ways on multiples of `align` rows
// (slices shrink towards the end, 1 - ((k - i) / k)^2 of the rows before edge i: the copy of the
// last slice is the only one that nothing overlaps)
static inline int band_slice_edge(int row0, int rows, int i, int k, int align) {
  if (i >= k) return row0 + rows;
  const long long rem = (long long)(k - i) * (k - i), all = (long long)k * k;
  const int e = (int)((long long)rows * (all - rem) / all) / align * align;
  return row0 + e;
}
// sp: the caller's sample pattern (render_raytrace_samples), or null for Draw's nine samples
int rt_launch(b200_ctx *ctx, const RtFrame &f, float *d_rgb, float *d_depth, int32_t *d_index,
              uint32_t *d_argb, const RtSamplesParams *sp = nullptr);
// rt_rays.cu: one ray query on the uploaded scene, n > 0 rays; d_hits (closest hits) or d_occ + d_max (occlusion)
int rt_launch_rays(b200_ctx *ctx, const rt_ray *d_rays, const float *d_max, int n, rt_intersection *d_hits,
                   uint8_t *d_occ);
// rt_rays.cu: DirectLight for n > 0 hits and 1..8 lights on the uploaded scene, d_power[(i * n_lights + l) * 3 + c]
int rt_launch_direct_light(b200_ctx *ctx, const rt_intersection *d_hits, int n, const light_t *lights, int n_lights,
                           float *d_power);
// whole frames of n_views cameras of one size, frame k of each output at k * W * H (rgb: times 3)
int rt_launch_views(b200_ctx *ctx, const RtFrame *fs, int n_views, float *d_rgb, float *d_depth, int32_t *d_index,
                    uint32_t *d_argb);
// The four outputs of a frame, host or device pointers; a null pointer is an output nobody asked for.
struct Outputs {
  float *rgb = nullptr, *depth = nullptr;
  int32_t *index = nullptr;
  uint32_t *argb = nullptr;
  // the same outputs from pixel `px` on
  Outputs at(size_t px) const {
    return {rgb ? rgb + 3 * px : nullptr, depth ? depth + px : nullptr, index ? index + px : nullptr,
            argb ? argb + px : nullptr};
  }
};
// api.cu: rows [row_begin, row_end) of the whole Draw on the scene already uploaded, into band-sized host outputs
int rast_band_resident(b200_ctx *ctx, const camera_t *cam, const rast_light_t *light, int row_begin, int row_end,
                       const Outputs &host);
// multi.cu: entry points of a multi-GPU context (api.cu forwards to these)
void multi_destroy(b200_ctx *ctx);
int multi_synchronize(b200_ctx *ctx);
int multi_set_option(b200_ctx *ctx, int option, int value);
int multi_rast_set_textures(b200_ctx *ctx, const rast_textures_t *tex);
// job(child, a, b): the single-device work of items [a, b) on one device of a multi-GPU context
using MultiJob = std::function<int(b200_ctx *, int, int)>;
// Items [0, count) in even shares of whole `align`-item units, one share per device; sums the devices' stats.
int multi_split(b200_ctx *ctx, int count, int align, const MultiJob &job);
// Rows [0, rows) of a raytraced frame in bands balanced on the measured cost of earlier frames.
int multi_raytrace(b200_ctx *ctx, int rows, const MultiJob &job);
// The whole Draw of rows [row_begin, row_end) in balanced bands; the arguments have been checked (api.cu).
int multi_raster(b200_ctx *ctx, const rast_triangle *room, int n_room, const rast_triangle *boxes, int n_boxes,
                 const camera_t *cam, const rast_light_t *light, int row_begin, int row_end, const Outputs &host);
