/* b200render.h -- C ABI of the B200-native renderer.
 *
 * Drop-in boundary for the two hot paths of fznsakib/Computer-Graphics
 * (citations are file:line in that repository):
 *
 *   RT   raytracer/Source/skeleton.cpp   Draw :104-169 -> ClosestIntersection
 *        :263-363 -> DirectLight :366-415        (per-pixel primary + shadow rays)
 *   RAST rasteriser/Source/skeleton.cpp  Draw :203-308 -> DrawPolygon :420-431
 *        -> VertexShader :510-522 -> ComputePolygonRows :433-498
 *        -> DrawPolygonRows :500-508 -> PixelShader :559-672
 *        -> calculateIllumination :674-688, then the post pass :283-307.
 *
 * The reference's entry point is `void Draw(screen*)` with every other input a
 * file-scope global (RT :56-60, RAST :30-86).  This ABI carries what those
 * globals carry, as plain pointers and sizes.  All structs are byte-compatible
 * with the reference's own types so a caller can pass `&triangles[0]` directly.
 *
 * Conventions
 *   - every function returns B200_OK (0) or a negative B200_E* code; nothing
 *     ever calls exit();
 *   - "host" entry points take HOST pointers and do the H2D/D2H copies
 *     themselves; "_device" entry points take DEVICE pointers (they may be peer
 *     mappings of another GPU's memory -- the kernels store bands straight
 *     through them) and enqueue on the context's stream without synchronising;
 *   - one context per GPU and per host thread; calls on a context serialise;
 *   - there is no CPU fallback: without a CUDA device b200_init fails.
 */
#ifndef B200RENDER_H
#define B200RENDER_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_OK 0
#define B200_EINVAL (-1) /* bad argument (null pointer, bad size, bad band) */
#define B200_ECUDA (-2)  /* CUDA runtime error; see b200_last_error()        */
#define B200_ENOMEM (-3) /* device or pinned-host allocation failed          */
#define B200_ENODEV (-4) /* no usable CUDA device (no CPU fallback exists)   */

/* index_out value for "no hit" (RT) / "no opaque fragment" (RAST is -1). */
#define B200_INDEX_MISS INT32_MIN

/* ---- types (byte-compatible with the reference) ---------------------------*/

/* raytracer/Source/TestModelH.h:80-115 `class Triangle`: 76 bytes. */
typedef struct rt_triangle {
  float v0[4], v1[4], v2[4];
  float normal[4]; /* w = 1.0 in the reference (TestModelH.h:104)            */
  float color[3];
} rt_triangle;

/* raytracer/Source/TestModelH.h:14-77 `class Sphere`: 44 bytes. */
typedef struct rt_sphere {
  float radius, radius_squared;
  float centre[3], color[3];
  float normal[3]; /* never initialised nor read by the reference            */
} rt_sphere;

/* rasteriser/Source/TestModelH.h:13-42 `class Triangle`: 84 bytes. */
typedef struct rast_triangle {
  float v0[4], v1[4], v2[4];
  float normal[4];
  float color[3];  /* color[0] < 0 marks a shadow-volume triangle (:1705)    */
  int32_t texture; /* 0 untextured, 1 marble, 2 metal grill, 3 woven wood
                    * (TestModelH.h:21-22); non-zero needs rast_set_textures  */
  int32_t index;   /* object the texture is laid over (TestModelH.h:23-24): 0
                    * back, 1 ceiling, 2 floor, 3 left wall, 4 right wall     */
} rast_triangle;

/* RT globals cameraPos / focalLength / R (skeleton.cpp:56-60) and RAST globals
 * cameraPos / focalLength / R (skeleton.cpp:30-35), plus the resolution that
 * the reference fixes with #define SCREEN_WIDTH / SCREEN_HEIGHT. */
typedef struct camera_t {
  float pos[4];
  float focal;
  float R[16]; /* column-major, R[4*c + r] == glm R[c][r]                    */
  int32_t width, height;
} camera_t;

/* raytracer `struct Light` (skeleton.cpp:47-50). */
typedef struct light_t {
  float pos[4];
  float colour[3];
} light_t;

/* rasteriser light globals: sceneCoordinatesLightPos (or, for the clipped-list
 * entry, the camera-space lightPos), lightPower, indirectLightPowerPerArea
 * (skeleton.cpp:51-54).  `indirect` is the value the global holds when Draw is
 * entered (0.15 at start-up :54, 0.2 +- 0.005 after keys 1 / 2): PixelShader
 * resets the global to 0.2 after every shaded fragment (:585), so, exactly like
 * the reference, only the first shaded fragment of the frame sees `indirect`
 * and every other one 0.2. */
typedef struct rast_light_t {
  float pos[4];
  float power[3];
  float indirect[3];
} rast_light_t;

typedef struct b200_ctx b200_ctx;

/* ---- context ---------------------------------------------------------------*/

/* Creates a context on CUDA device `device` (one process per GPU: pass
 * LOCAL_RANK).  Fails with B200_ENODEV when there is no GPU. */
int b200_init(int device, b200_ctx **out);
/* One context for the first n_gpus devices of the box (0: all of them).  This is the
 * `b200_init(n_gpus)` of the drop-in contract: behind `Draw(screen*)` the HOST-pointer entry
 * points (render_raytrace*, draw_raytrace*, render_raster, render_raster_band, draw_raster*)
 * share every frame among the devices by row bands -- one host thread and one ordinary context
 * per device, the raytracer's bands following the measured cost of the previous frame, the
 * rasteriser's scene uploaded in N slices and all-gathered between the devices over NVLink --
 * and return when the assembled frame is in the caller's buffers.  Results are bit-identical to
 * a single device's.  The device-pointer entries, streams and intermediate buffers exist per
 * device only (B200_EINVAL here).  b200_get_stats: sums over the devices, gpu_ms the slowest. */
int b200_init_multi(int n_gpus, b200_ctx **out);
int b200_device_count(const b200_ctx *ctx);
void b200_destroy(b200_ctx *ctx);
/* Human-readable text of the last error on this context ("" if none). */
const char *b200_last_error(const b200_ctx *ctx);
/* The CUDA stream (cudaStream_t) every call on this context is enqueued on. */
void *b200_stream(b200_ctx *ctx);
/* Waits for everything enqueued on the context.  Also the point where a pipelined
 * raster frame (B200_OPT_RAST_PIPELINED) is verified, and rendered again if needed. */
int b200_synchronize(b200_ctx *ctx);
/* Makes the context enqueue on a caller-owned stream (e.g. the one the caller's
 * collectives run on); NULL restores the context's own stream. */
int b200_set_stream(b200_ctx *ctx, void *cuda_stream);

/* Tunables.  B200_OPT_RT_BRUTEFORCE = 1 switches the raytracer to the
 * unfiltered kernel that runs the reference arithmetic on every ray/triangle
 * pair (on-device cross-check of the filtered kernel; results are identical).
 * It also switches the ray queries (rt_closest_hits, rt_occluded) to the
 * per-ray exact loop over every pair, without cull or early exit. */
#define B200_OPT_RT_BRUTEFORCE 1
#define B200_OPT_RAST_TILE_LOG2 2   /* ordered-tile path: log2 of the screen-tile edge, 3..5 (default 5) */
/* Rasteriser strategy: 0 = automatic, 1 = ordered screen tiles (any list; keeps
 * the intermediate buffers readable), 2 = atomic scatter + fused resolve
 * (lists without shadow-volume triangles only).  Results are identical. */
#define B200_OPT_RAST_PATH 3
/* Pipelined rasteriser frames for the device-pointer entries (rast_render_device,
 * rast_draw_device): 0 (default) = every frame reads its list/table sizes back
 * mid-frame (two short host waits); 1 = a frame of the same shape as the last
 * verified one is enqueued without any host wait, sized from that frame plus a
 * margin.  Its own counters are checked in b200_synchronize / b200_get_stats and a
 * frame that outgrew the guess is rendered again there with exact sizes, so the
 * output buffers are final only after one of those two calls returns.  The
 * host-pointer entries always work this way internally.  Results are identical. */
#define B200_OPT_RAST_PIPELINED 4
/* Raytracer direction grids (per-frame lists of the triangles each 16x16 pixel
 * block and each cube-map cell around a light can see): 0 = automatic (scenes of
 * 1024 triangles or more), 1 = always, 2 = never.  Results are identical. */
#define B200_OPT_RT_GRID 5
/* Raytracer work split for N cooperating contexts (one per GPU) that render the SAME row
 * range into one full-frame buffer: with INTERLEAVE_N = n > 1 and INTERLEAVE_R = r this
 * context renders the 16-row blocks b of the range with b % n == r and leaves the others
 * untouched, which balances the GPUs better than contiguous bands.  Device-pointer entry
 * (rt_render_device) only; the default (1, 0) renders every row of the range. */
#define B200_OPT_RT_INTERLEAVE_N 6
#define B200_OPT_RT_INTERLEAVE_R 7
/* Rasteriser, whole-Draw entries rendering a BAND of the frame (row_begin > 0 or row_end < H)
 * with pipelined frames on the scatter path: 1 = the geometry stage keeps only the triangles
 * whose rows reach the band (+ its 2-row halo), so that setup / scatter / resolve work on 1/N of
 * the list when N devices share a frame.  Pixels, depth and owner indices are identical;
 * raster_read_clipped then returns the band's list.  Default 0; on in the per-device contexts
 * of b200_init_multi. */
#define B200_OPT_RAST_BAND_CULL 8
/* Rasteriser colour mode = the reference's randColourSelect (skeleton.cpp:81, toggled by SPACE :407):
 * 0 (default) the shaded / textured colours; 1 random colours; 2 "night vision" (:647-662).  In modes 1
 * and 2 every ACCEPTED fragment draws three values from the C library's rand(), in the serial order of
 * the reference's loops; the library numbers the accepted fragments in that order on the device and
 * then calls rand() itself, three times per fragment, so the pixels AND the process's rand() stream
 * end up as after the reference's Draw (seed with srand as the reference's process would be).  Only
 * screenBuffer is written (:653, :661), the texture fields are ignored, and indirectLightPowerPerArea is
 * not reset (`indirect` applies to every fragment).  Whole frames only (no row bands; a multi-GPU
 * context draws such frames on its first device). */
#define B200_OPT_RAST_COLOUR_MODE 9
/* Raytracer, gridded (large-scene) frames: 1 (default) = a frame that follows a gridded frame of the same shape
 * runs its 16x16 pixel blocks in an order planned from that frame's measured block costs -- the few blocks that
 * cost several times the mean first, and split into eight launches of four pixels per warp; 0 = launch order.
 * Results are identical. */
#define B200_OPT_RT_PLAN 10
int b200_set_option(b200_ctx *ctx, int option, int value);

/* Counters of the last render on this context (b200_get_stats synchronises). */
typedef struct b200_stats {
  uint64_t primary_rays;     /* RT: W * rows * 9                              */
  uint64_t shadow_rays;      /* RT: primary hits * n_lights                   */
  uint64_t prim_tests;       /* RT: rays * (n_tris + n_spheres)               */
  uint64_t exact_evals;      /* RT: pairs that ran the reference arithmetic   */
  uint64_t kernel_launches;  /* kernels of this library launched by the call  */
  uint64_t fragments;        /* RAST: fragments shaded or depth-tested        */
  uint64_t bin_entries;      /* RAST: (tile, triangle) pairs                  */
  uint64_t respeculated;     /* RAST: pipelined frames rendered twice (context lifetime) */
  float gpu_ms;              /* device time of the call, CUDA events          */
} b200_stats;
int b200_get_stats(b200_ctx *ctx, b200_stats *out);

/* ---- RT: replaces raytracer Draw(screen*) (skeleton.cpp:104-169) -----------*/

/* Host-pointer entry.  Renders rows [0, cam->height).
 *   rgb_out   W*H*3 floats: the colour the reference hands to PutPixelSDL
 *             (averageLight, or black), before quantisation.   May be NULL.
 *   depth_out W*H floats: closestIntersection.distance of the centre sample
 *             (i = j = 0), +inf on miss.                        May be NULL.
 *   index_out W*H: centre-sample triangleIndex, or -1 - sphereIndex, or
 *             B200_INDEX_MISS.                                  May be NULL.
 */
int render_raytrace(b200_ctx *ctx, const rt_triangle *tris, int n_tris,
                    const rt_sphere *spheres, int n_spheres, const camera_t *cam,
                    const light_t *lights, int n_lights, float *rgb_out, float *depth_out,
                    int32_t *index_out);

/* Same, but only rows [row_begin, row_end) (one GPU's band); the outputs are
 * band-sized: (row_end - row_begin) * W pixels. */
int render_raytrace_band(b200_ctx *ctx, const rt_triangle *tris, int n_tris,
                         const rt_sphere *spheres, int n_spheres, const camera_t *cam,
                         const light_t *lights, int n_lights, int row_begin, int row_end,
                         float *rgb_out, float *depth_out, int32_t *index_out);

/* Exactly what `Draw(screen*)` leaves in screen->buffer: W*H packed 0x80RRGGBB
 * with the PutPixelSDL truncation rule (SDLauxiliary.h:149-161). */
int draw_raytrace(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres,
                  int n_spheres, const camera_t *cam, const light_t *lights, int n_lights,
                  uint32_t *argb_out);

/* Band variant: argb_out is band-sized, (row_end - row_begin) * W.  Frames of
 * three megapixels or more come back in slices copied on a second stream while the next
 * slice is rendered (pass pinned memory to benefit); the call returns when the
 * whole band is in argb_out. */
int draw_raytrace_band(b200_ctx *ctx, const rt_triangle *tris, int n_tris,
                       const rt_sphere *spheres, int n_spheres, const camera_t *cam,
                       const light_t *lights, int n_lights, int row_begin, int row_end,
                       uint32_t *argb_out);

/* Measures this GPU's FP32 FFMA rate (the raytracer's roofline denominator). */
int b200_measure_fp32_peak(b200_ctx *ctx, float *tflops_out);

/* Device-resident path: upload the scene once, render many times. */
int rt_upload_scene(b200_ctx *ctx, const rt_triangle *tris, int n_tris,
                    const rt_sphere *spheres, int n_spheres);
/* All output pointers are DEVICE pointers addressed as full-frame arrays
 * (pixel (x, y) at y*W + x); only rows [row_begin, row_end) are written.  Any
 * of them may be NULL.  Asynchronous on b200_stream(ctx). */
int rt_render_device(b200_ctx *ctx, const camera_t *cam, const light_t *lights, int n_lights,
                     int row_begin, int row_end, float *d_rgb, float *d_depth,
                     int32_t *d_index, uint32_t *d_argb);

/* ---- RT, batched views: many cameras of one scene in one call ----------------
 * n_views cameras (same width and height, any pos / focal / R) of one scene and one set of lights.
 * Outputs hold n_views whole frames back to back: view k's pixel (x, y) is at
 * k*W*H + y*W + x (rgb: times 3).  Each frame is bit-identical to render_raytrace /
 * draw_raytrace / rt_render_device with cams[k].  Any output of render_raytrace_views and
 * rt_render_views_device may be NULL; draw_raytrace_views needs argb_out.
 *   - n_views >= 1, cams non-null, every camera a valid resolution and the same W, H as
 *     cams[0]; at most 8 lights (non-null when n_lights > 0): otherwise B200_EINVAL.
 *   - Whole frames only: no row band, and B200_OPT_RT_INTERLEAVE_N / _R do not apply.
 *   - Scenes that take the scene-streaming kernel (fewer than 1024 triangles, or
 *     B200_OPT_RT_GRID = 2) render up to 64 views in one launch; larger batches take several
 *     launches inside the call, and the per-view device buffers stay sized for 64 views.
 *     Gridded scenes, B200_OPT_RT_BRUTEFORCE = 1 and a batch of one view render view by view.
 *   - b200_get_stats afterwards: primary_rays = n_views * W * H * 9, shadow_rays and
 *     exact_evals summed over the views, gpu_ms the device time of the whole call.
 *   - On a b200_init_multi context the host-pointer entries give each device a contiguous run
 *     of whole views; rt_render_views_device is per device (B200_EINVAL there). */
int render_raytrace_views(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres,
                          int n_spheres, const camera_t *cams, int n_views, const light_t *lights,
                          int n_lights, float *rgb_out, float *depth_out, int32_t *index_out);
int draw_raytrace_views(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres,
                        int n_spheres, const camera_t *cams, int n_views, const light_t *lights,
                        int n_lights, uint32_t *argb_out);
/* Device-resident: the scene of rt_upload_scene, DEVICE output pointers (n_views * W * H pixels
 * each), asynchronous on b200_stream(ctx). */
int rt_render_views_device(b200_ctx *ctx, const camera_t *cams, int n_views, const light_t *lights,
                           int n_lights, float *d_rgb, float *d_depth, int32_t *d_index,
                           uint32_t *d_argb);

/* ---- RT, the caller's own sample pattern per pixel -----------------------------
 * Draw (skeleton.cpp:123-168) with the 3x3 sample grid replaced by the caller's n_samples offsets.
 * Sample k of pixel (u, v) is the ray from cam->pos along (dir.x + offsets[2k], dir.y + offsets[2k+1], focal),
 *   where dir = R * vec4(u - W/2, v - H/2, focal, 1) exactly as in Draw, and the offset is added to the rotated
 *   direction in float32, one rounding.  The reference's pattern is offsets = 0.5*(i, j) with i = -1..1 outer
 *   and j = -1..1 inner.
 * Per pixel, samples are taken in the caller's order.  A sample that hits adds DirectLight for each light in order,
 *   then colour * 0.5f.  The pixel is pix / (float)n_samples if any sample hit, else 0.
 * depth / index are those of sample depth_sample.  The meaning is render_raytrace's (distance or +inf;
 *   triangle, -1 - sphere, or B200_INDEX_MISS).  Passing the reference's pattern with depth_sample = 4 gives
 *   render_raytrace's frame bit for bit.
 *   - 1 <= n_samples <= 64; every offset finite with |offset| <= 0.5 (+-0.5 and -0.0 allowed);
 *     0 <= depth_sample < n_samples; camera and lights as render_raytrace.  Otherwise B200_EINVAL.
 *   - b200_get_stats: primary_rays = W * rows * n_samples, shadow_rays = hit samples * n_lights (device-counted),
 *     prim_tests, exact_evals, kernel_launches, gpu_ms as for frames.
 *   - Any output may be NULL, except that draw_raytrace_samples needs argb_out.  B200_OPT_RT_BRUTEFORCE = 1 runs
 *     the per-pixel exact loop; B200_OPT_RT_GRID chooses streaming or gridded as for frames.  The samples run in
 *     groups of up to nine per walk of the scene, so a frame costs about ceil(n_samples / 9) nine-sample frames of
 *     the filtered kernel; the half-pixel lattice kernel of render_raytrace is never used, and the gridded-frame
 *     block plan of B200_OPT_RT_PLAN is neither read nor written.
 *   - On a b200_init_multi context the host entries give each device an even, 16-row-aligned band of rows,
 *     returned straight into its slice of the caller's buffers; rt_render_samples_device returns B200_EINVAL
 *     there.  A pipelined raster frame in flight is finished first. */
#define B200_RT_MAX_SAMPLES 64
int render_raytrace_samples(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres,
                            int n_spheres, const camera_t *cam, const light_t *lights, int n_lights,
                            const float *offsets, int n_samples, int depth_sample,
                            float *rgb_out, float *depth_out, int32_t *index_out);
int draw_raytrace_samples(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres,
                          int n_spheres, const camera_t *cam, const light_t *lights, int n_lights,
                          const float *offsets, int n_samples, int depth_sample, uint32_t *argb_out);
/* The scene of rt_upload_scene, DEVICE outputs addressed as full frames, rows [row_begin, row_end),
 * asynchronous on b200_stream(ctx).  Offsets are HOST memory, as lights are.  B200_OPT_RT_INTERLEAVE_N / _R
 * apply as for rt_render_device. */
int rt_render_samples_device(b200_ctx *ctx, const camera_t *cam, const light_t *lights, int n_lights,
                             const float *offsets, int n_samples, int depth_sample, int row_begin, int row_end,
                             float *d_rgb, float *d_depth, int32_t *d_index, uint32_t *d_argb);

/* ---- RT, ray queries: ClosestIntersection for rays the caller supplies --------
 * raytracer/Source/skeleton.cpp:40-45 (struct Intersection), :263-363 (ClosestIntersection) and
 * :394-397 (DirectLight's shadow test `ClosestIntersection(...) && distance < r_mag`), for any rays:
 * picking from any point, visibility between two points, other sampling patterns, code that calls
 * ClosestIntersection directly.  Every result is bit-identical to the reference's.
 *   - One thread per ray, in the caller's order.  There is no spatial index: the cost of a call is
 *     rays x (triangles + spheres) minus what a per-warp cull removes; coherent rays (neighbouring
 *     pixels, shadow rays of neighbouring points) cull far better than incoherent ones.  Scenes of
 *     1024 triangles or more stream all their triangles like small ones.
 *   - n_rays < 0, a null rays / out / max_distance with n_rays > 0, or bad scene arguments:
 *     B200_EINVAL.  n_rays == 0: B200_OK, nothing written.  An empty scene misses everywhere.
 *   - b200_get_stats afterwards: primary_rays = n_rays (closest) or shadow_rays = n_rays (occlusion),
 *     prim_tests = n_rays * (n_tris + n_spheres), exact_evals = ray/triangle pairs that ran the
 *     reference arithmetic, kernel_launches and gpu_ms as for frames.
 *   - B200_OPT_RT_BRUTEFORCE = 1: the per-ray exact loop over every pair (on-device cross-check).
 *   - A query leaves the context as it was for the next frame (pixels, the gridded-frame block plan
 *     of B200_OPT_RT_PLAN); a pipelined raster frame in flight is finished first.
 *   - On a b200_init_multi context the host-pointer entries give each device a contiguous run of the
 *     rays, returned straight into its slice of out; the _device entries return B200_EINVAL there. */

/* The (start, dir) arguments of ClosestIntersection: 32 bytes.  Only xyz of dir is read
 * (glm::length(dir3) :307, mat3(-dir, e1, e2) :289); start.w only reaches position.w. */
typedef struct rt_ray {
  float start[4];
  float dir[4];
} rt_ray;

/* raytracer/Source/skeleton.cpp:40-45 `struct Intersection`: 28 bytes, offsets 0 / 16 / 20 / 24. */
typedef struct rt_intersection {
  float position[4];       /* start + vec4(t * dir3, 0): position.w = start.w + 0.0f (so -0 becomes +0) */
  float distance;          /* t * |dir3| for triangles, the raw t for spheres (:350); FLT_MAX on a miss  */
  int32_t triangle_index;  /* -1 when a sphere or nothing was hit                                      */
  int32_t sphere_index;    /* -1 when a triangle or nothing was hit                                    */
} rt_intersection;

/* out[i] = the Intersection ClosestIntersection(rays[i].start, rays[i].dir, ...) leaves behind.  A ray
 * hit something iff distance < FLT_MAX; on a miss the reference leaves every other field untouched,
 * and the library sets position to 0 and both indices to -1.  Host pointers; uploads the scene like
 * render_raytrace. */
int rt_closest_hits(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres,
                    int n_spheres, const rt_ray *rays, int n_rays, rt_intersection *out);
/* out[i] = 1 iff ClosestIntersection returns true AND distance < max_distance[i] (DirectLight's shadow
 * test, :394-397, sphere distances included as the reference has them); a NaN or non-positive limit
 * gives 0.  Host pointers. */
int rt_occluded(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres,
                int n_spheres, const rt_ray *rays, const float *max_distance, int n_rays, uint8_t *out);
/* Device-resident: the scene of rt_upload_scene, DEVICE pointers, asynchronous on b200_stream(ctx). */
int rt_closest_hits_device(b200_ctx *ctx, const rt_ray *d_rays, int n_rays, rt_intersection *d_out);
int rt_occluded_device(b200_ctx *ctx, const rt_ray *d_rays, const float *d_max_distance, int n_rays,
                       uint8_t *d_out);

/* ---- RT, DirectLight for hits the caller supplies --------------------------------
 * skeleton.cpp:366-415 for every (hit, light) pair, bit for bit, so that Draw composes from library calls for any
 * set of sample rays: rt_closest_hits -> rt_direct_light -> the caller's own accumulation.
 *   - Per light, not summed: Draw adds each light's DirectLight into its running pixel sum one at a time
 *     (:151-153), and a sum over the lights would round differently.
 *   - The entry rule of the reference's `if (triangleIndex != -1)`: triangle_index != -1 names that triangle,
 *     which must lie in [0, n_tris); otherwise sphere_index names a sphere in [0, n_spheres).  Any other entry
 *     (the miss records of rt_closest_hits, indices out of range) gives 0 and traces nothing.
 *   - position is read; position.w reaches only the shadow ray's start.w, so no output.  distance is not read.
 *   - A NaN output component that the arithmetic creates from NaN-free inputs (a light exactly at the hit point, a
 *     hit at a sphere's centre, inf - inf) is stored as 0xffc00000, the NaN the reference makes on x86.  Where an
 *     input carries a NaN the NaN's payload is not specified.
 *   - n_hits < 0, n_lights < 0 or > B200_MAX_LIGHTS (8), a null hits / power_out when n_hits > 0 and n_lights > 0,
 *     a null lights when n_lights > 0, or bad scene arguments: B200_EINVAL.  n_hits == 0 or n_lights == 0:
 *     B200_OK, nothing written.
 *   - One thread per (hit, light) pair; the shadow ray walks the scene like rt_occluded (per-warp cull, exact early
 *     exit).  B200_OPT_RT_BRUTEFORCE = 1: the per-ray exact loop over every pair, without cull or early exit.
 *   - b200_get_stats afterwards: primary_rays = 0, shadow_rays = pairs that traced a shadow ray (entries naming a
 *     primitive x n_lights, counted on the device), prim_tests = shadow_rays * (n_tris + n_spheres), exact_evals,
 *     kernel_launches and gpu_ms as for the ray queries.
 *   - The context is left as the ray queries leave it; a pipelined raster frame in flight is finished first.
 *   - On a b200_init_multi context rt_direct_light gives each device a contiguous run of the hits;
 *     rt_direct_light_device returns B200_EINVAL there. */

/* power_out[(i * n_lights + l) * 3 + c] = DirectLight(hits[i]) for lights[l] (skeleton.cpp:366-415), bit for bit.
 * Host pointers; uploads the scene like render_raytrace. */
int rt_direct_light(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres, int n_spheres,
                    const rt_intersection *hits, int n_hits, const light_t *lights, int n_lights, float *power_out);
/* Device-resident: the scene of rt_upload_scene, DEVICE hits / power, HOST lights (as rt_render_device),
 * asynchronous on b200_stream(ctx). */
int rt_direct_light_device(b200_ctx *ctx, const rt_intersection *d_hits, int n_hits, const light_t *lights,
                           int n_lights, float *d_power);

/* ---- RAST: replaces rasteriser Draw(screen*) (skeleton.cpp:203-308) --------*/

/* Tier 1: the triangle loop + post pass (skeleton.cpp:243-307) on an
 * already-clipped list (camera space, w = z/f, in draw order).  light->pos is
 * the camera-space, rotated `lightPos` (skeleton.cpp:211-212,223).
 *   rgb_out   W*H*3: colour handed to PutPixelSDL (border pixels stay 0)
 *   depth_out W*H: depthBuffer (1/z, 0 = empty)
 *   index_out W*H: index of the opaque triangle owning the pixel, -1 if none
 */
int render_raster_clipped(b200_ctx *ctx, const rast_triangle *clipped, int n_tris,
                          const camera_t *cam, const rast_light_t *light, float *rgb_out,
                          float *depth_out, int32_t *index_out);

/* Tier 2: the whole Draw on a world-space scene: camera transform, shadow
 * volumes for `boxes`, rotation, clip-space w, six-plane clip, then tier 1.
 * light->pos is sceneCoordinatesLightPos (world space). */
int render_raster(b200_ctx *ctx, const rast_triangle *room, int n_room,
                  const rast_triangle *boxes, int n_boxes, const camera_t *cam,
                  const rast_light_t *light, float *rgb_out, float *depth_out,
                  int32_t *index_out);

/* Rows [row_begin, row_end) of render_raster; the outputs are band-sized. */
int render_raster_band(b200_ctx *ctx, const rast_triangle *room, int n_room,
                       const rast_triangle *boxes, int n_boxes, const camera_t *cam,
                       const rast_light_t *light, int row_begin, int row_end, float *rgb_out,
                       float *depth_out, int32_t *index_out);

/* ---- RAST textures: PixelShader's texture branches (skeleton.cpp:588-645) --------------
 * The reference's main() decodes eight image files with OpenCV into cv::Mat globals
 * (:63-75, :133-155) and draws normalMap_marble from rand() (:157-168); PixelShader then
 * reads pixels, at<T>(findU, findV).  The library takes exactly that state: DECODED images
 * (decoding stays with the caller), addressed like cv::Mat -- `rows` x `step` bytes,
 * at<T>(r, c) = *(T *)(data + r * step + c * sizeof(T)). */
typedef struct rast_image_t {
  const uint8_t *data; /* host memory; copied by rast_set_textures           */
  int32_t rows, cols;
  int32_t step;        /* bytes per row (cols * channels when continuous)    */
} rast_image_t;
typedef struct rast_textures_t {
  rast_image_t marble;          /* `marble` :64, read as Vec3b (BGR) at (findU(p, 2000), findV(p, 2000)) */
  const float *marble_noise;    /* `normalMap_marble` :75: vec4 per entry, added to the normal (:593)    */
  int64_t marble_noise_len;     /* entries; indexed y * marble.rows + x of the SCREEN pixel              */
  rast_image_t grill;           /* `metalGrill` :70 (Vec3b)                                               */
  rast_image_t grill_opacity;   /* `metalGrillOpacity` after cv::threshold (:152): uchar, 255 = solid    */
  rast_image_t grill_normal;    /* `metalGrillNormalMap` :72 (Vec3b)                                      */
  rast_image_t woven;           /* `woven` :65 (Vec3b)                                                    */
  rast_image_t woven_occlusion; /* `woven_ambientOcclusion` :66, read as uchar at byte column findV (:626) */
  rast_image_t woven_opacity;   /* `woven_opacity` after cv::threshold (:155): uchar                      */
  rast_image_t woven_normal;    /* `wovenNormal` :68 (Vec3b)                                              */
} rast_textures_t;
/* Copies the images to the device(s) of the context; from then on the `texture` / `index` fields
 * of the triangles are honoured (without textures set, a list with texture != 0 is refused with
 * B200_EINVAL) and every raster frame is drawn by the ordered path: a metal-grill / woven-wood
 * fragment whose opacity is not 255 passes the depth test, keeps the pixel's colours and sets its
 * depth back to 0 (:619, :643, :665), which only an in-order fold reproduces.  The marble must be
 * at least 2000 x 2000 and the others 1024 x 1024 (the sizes findU / findV are called with).
 * findU / findV use cam->pos and glm::inverse(cam->R) (the reference's `yaw != 0` branch is taken
 * when cam->R is not the identity).  Where the reference reads outside an image (negative
 * findU / findV, normalMap_marble on screens taller than the marble) the coordinate wraps /
 * the index is clamped.  NULL switches textures off again.  (Colour modes 1 and 2: see
 * B200_OPT_RAST_COLOUR_MODE.) */
int rast_set_textures(b200_ctx *ctx, const rast_textures_t *textures);

/* screen->buffer of the whole rasteriser Draw. */
int draw_raster(b200_ctx *ctx, const rast_triangle *room, int n_room,
                const rast_triangle *boxes, int n_boxes, const camera_t *cam,
                const rast_light_t *light, uint32_t *argb_out);

/* Intermediate buffers of the last render_raster* call, for parity checks
 * against the reference's file-scope buffers (skeleton.cpp:39-46).  HOST
 * pointers, any may be NULL: screenBuffer before the in-place shadow darkening,
 * lowLightBuffer, highLightBuffer (W*H*3 each), shadowBuffer (W*H). */
int raster_read_buffers(b200_ctx *ctx, float *screen_out, float *low_out, float *high_out,
                        int32_t *shadow_out);
/* The clipped list the last render_raster built (tier 2); returns its length
 * in *n_out, copies min(cap, n) triangles. */
int raster_read_clipped(b200_ctx *ctx, rast_triangle *out, int cap, int *n_out);

/* Band variant of draw_raster: argb_out is band-sized, (row_end - row_begin) * W. */
int draw_raster_band(b200_ctx *ctx, const rast_triangle *room, int n_room,
                     const rast_triangle *boxes, int n_boxes, const camera_t *cam,
                     const rast_light_t *light, int row_begin, int row_end, uint32_t *argb_out);

/* Device-resident path, tier 1 (clipped list + camera-space light).  Output
 * pointers are DEVICE pointers addressed as full frames; rows [row_begin,
 * row_end) are written; asynchronous on b200_stream(ctx). */
int rast_upload_clipped(b200_ctx *ctx, const rast_triangle *clipped, int n_tris);
int rast_render_device(b200_ctx *ctx, const camera_t *cam, const rast_light_t *light,
                       int row_begin, int row_end, float *d_rgb, float *d_depth,
                       int32_t *d_index, uint32_t *d_argb);
/* Device-resident path, tier 2 (world-space scene + world-space light): the
 * geometry stage runs on the GPU every frame, like the reference's Draw. */
int rast_upload_scene(b200_ctx *ctx, const rast_triangle *room, int n_room,
                      const rast_triangle *boxes, int n_boxes);
int rast_draw_device(b200_ctx *ctx, const camera_t *cam, const rast_light_t *light,
                     int row_begin, int row_end, float *d_rgb, float *d_depth,
                     int32_t *d_index, uint32_t *d_argb);

/* ---- scenes (host-side data builders) ---------------------------------------*/

/* The raytracer's LoadTestModel (raytracer/Source/TestModelH.h:121-279): 28
 * triangles + 1 sphere, byte-identical to the reference's vectors. */
int b200_scene_cornell_rt(rt_triangle *tris, int tri_cap, rt_sphere *spheres, int sph_cap,
                          int *n_tris, int *n_spheres);
/* BASELINE config 5: each Cornell triangle split into n*n (n = 60: 100 800). */
int b200_scene_cornell_rt_tessellated(int n, rt_triangle *tris, int tri_cap, int *n_tris);
/* The rasteriser's LoadTestModel with setting = settingBoxes = 0
 * (rasteriser/Source/TestModelH.h:48-312): 10 room + 20 box triangles. */
int b200_scene_cornell_rast(rast_triangle *room, int room_cap, rast_triangle *boxes, int boxes_cap,
                            int *n_room, int *n_boxes);
/* BASELINE config 4: n-triangle random soup (mt19937(seed), edges in +-edge). */
int b200_scene_soup_rast(int n, uint32_t seed, float edge, rast_triangle *tris);

/* ---- headless framebuffer (replaces SDL_SaveImage, SDLauxiliary.h:24-53) ---*/

/* Quantises float RGB to 0x80RRGGBB with the PutPixelSDL rule (host helper). */
void b200_quantise(const float *rgb, size_t n_pixels, uint32_t *argb_out);
/* Writes a 32-bpp top-down-flipped BMP like SDL_SaveBMP of an ARGB8888 surface. */
int b200_save_bmp(const char *path, const uint32_t *argb, int width, int height);

#ifdef __cplusplus
}
#endif
#endif /* B200RENDER_H */
