// Multi-GPU contexts: one handle, N devices of one box.
//
// SURVEY 8(b) asks for `b200_init(n_gpus)` behind the reference's single entry point
// `void Draw(screen*)` (raytracer/Source/skeleton.cpp:104, rasteriser/Source/skeleton.cpp:203),
// and 8(e) for "each GPU renders its band, assembled over NVLink".  A context made by
// b200_init_multi owns one ordinary context per device and one host thread per device (a
// frame at 4K is ~0.2 ms of GPU time per device at N = 8: enqueueing eight devices' launches
// and copies from one thread would take longer than the frame).  The host-pointer entry
// points split the frame into row bands and run the per-device work concurrently:
//
//   raytracer  the scene (2 KB ... 7.6 MB) goes to every device over its own PCIe link; device
//              i renders rows [b_i, b_i+1) and returns them straight into the caller's buffer
//              (N links in parallel -- for a HOST destination that beats funnelling the frame
//              through one GPU).  Band edges follow the measured cost of the previous frame
//              (the Cornell box is 3x more expensive in its lower half than at the top).
//   rasteriser device i uploads only slice i of the world-space triangles (1/N of 84 MB at 1 M
//              triangles) and pushes it to the N-1 peers over NVLink (peer copies, ordered by
//              events): an all-gather whose host traffic is the scene ONCE, not N times.
//              Then the geometry stage on every device (a pure per-triangle stream) keeps only
//              the triangles whose rows meet the device's band (B200_OPT_RAST_BAND_CULL), so
//              setup / scatter / resolve shard with the pixels.
//
// The device-pointer entries are per device by nature and stay on ordinary contexts; bench.py
// uses one process per GPU for those (torchrun) and a multi context for the end-to-end figure.
#include "common.cuh"

#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>

// Hand-offs between the calling thread and the device threads are short and frequent (a frame is a
// fraction of a millisecond): both sides spin for a while before they go to sleep on the condition
// variable (a wake-up through the kernel costs 20-50 us, several times per frame).
static int MULTI_SPIN = 20000;   // iterations; B200_MULTI_SPIN overrides (0: sleep at once)

struct MultiWorker {
  std::thread th;
  std::mutex m;
  std::condition_variable cv;
  std::function<int()> job;
  std::atomic<int> has_job{0}, done{1};
  bool quit = false;
  int rc = 0;
};

// Reusable barrier of the worker threads (phases of one frame: buffers exist -> slices pushed).
struct MultiBarrier {
  std::atomic<int> waiting{0};
  std::atomic<unsigned long long> gen{0};
  int n = 0;
  void wait() {
    const unsigned long long g = gen.load(std::memory_order_acquire);
    if (waiting.fetch_add(1, std::memory_order_acq_rel) + 1 == n) {
      waiting.store(0, std::memory_order_relaxed);
      gen.fetch_add(1, std::memory_order_release);
      return;
    }
    for (long long spins = 0; gen.load(std::memory_order_acquire) == g; ++spins)
      if (spins > MULTI_SPIN) std::this_thread::yield();
  }
};

struct b200_multi {
  int n = 0;
  std::vector<b200_ctx *> child;
  std::vector<MultiWorker *> worker;
  std::vector<cudaEvent_t> pushed;      // per device: its scene slice has reached every peer
  std::vector<int> phase_rc;            // per device: result of the phase before a barrier
  MultiBarrier barrier;
  // band edges of the last frame of each kind and what each band cost (adaptive split)
  std::vector<int> edges[2];
  std::vector<float> cost[2];
  int edges_h[2] = {0, 0};
  int settled[2] = {0, 0};              // the last frame of the kind ran on the same bands as the one before it
  int peer_ok = 0;                      // every pair of devices can address each other's memory
};

static void worker_main(MultiWorker *w, int device) {
  cudaSetDevice(device);
  for (;;) {
    for (int spins = 0; spins < MULTI_SPIN && !w->has_job.load(std::memory_order_acquire); ++spins) {}
    if (!w->has_job.load(std::memory_order_acquire)) {
      std::unique_lock<std::mutex> lk(w->m);
      w->cv.wait(lk, [&] { return w->has_job.load(std::memory_order_acquire) || w->quit; });
      if (w->quit) return;
    }
    w->has_job.store(0, std::memory_order_relaxed);
    w->rc = w->job();
    {
      std::lock_guard<std::mutex> lk(w->m);   // pairs with the caller's wait below
      w->done.store(1, std::memory_order_release);
    }
    w->cv.notify_all();
  }
}

// Runs job(i) on worker i for every device and waits for all; first failure wins.
static int multi_run(b200_ctx *ctx, const std::function<int(int)> &job) {
  b200_multi *mc = ctx->multi;
  for (int i = 0; i < mc->n; ++i) {
    MultiWorker *w = mc->worker[i];
    {
      std::lock_guard<std::mutex> lk(w->m);
      w->job = [&job, i] { return job(i); };
      w->done.store(0, std::memory_order_relaxed);
      w->has_job.store(1, std::memory_order_release);
    }
    w->cv.notify_all();
  }
  int rc = B200_OK;
  for (int i = 0; i < mc->n; ++i) {
    MultiWorker *w = mc->worker[i];
    for (int spins = 0; spins < MULTI_SPIN && !w->done.load(std::memory_order_acquire); ++spins) {}
    if (!w->done.load(std::memory_order_acquire)) {
      std::unique_lock<std::mutex> lk(w->m);
      w->cv.wait(lk, [&] { return w->done.load(std::memory_order_acquire) != 0; });
    }
    if (w->rc != B200_OK && rc == B200_OK) {
      rc = w->rc;
      ctx->err = "device " + std::to_string(i) + ": " + mc->child[i]->err;
    }
  }
  return rc;
}

// Row bands for the next frame of `kind` (0 RT, 1 RAST): equal rows at first, afterwards the
// edges that would have equalised the previous frame's measured cost (piecewise-constant cost
// per row inside each of its bands), on multiples of `align` rows.
void multi_band_edges(const std::vector<int> &prev_edges, const std::vector<float> &prev_cost, int H, int n, int align,
                      std::vector<int> &out, double tolerance = 1.06) {
  out.assign(n + 1, 0);
  out[n] = H;
  bool usable = (int)prev_edges.size() == n + 1 && (int)prev_cost.size() == n && prev_edges[n] == H;
  double total = 0;
  if (usable)
    for (int i = 0; i < n; ++i) {
      if (!(prev_cost[i] > 0.f) || prev_edges[i + 1] <= prev_edges[i]) usable = false;
      total += prev_cost[i];
    }
  if (!usable) {
    for (int i = 1; i < n; ++i) out[i] = (int)((long long)H * i / n);
  } else {
    // Hysteresis: a split within 6 % of balance stays as it is (a rasteriser band whose shape
    // changes cannot be pipelined from its predecessor, and timing noise must not move edges).
    float worst = 0.f;
    for (int i = 0; i < n; ++i) worst = prev_cost[i] > worst ? prev_cost[i] : worst;
    if (worst * n <= tolerance * total) { out = prev_edges; return; }
    int band = 0;
    double before = 0;   // cost of the bands in front of `band`
    for (int k = 1; k < n; ++k) {
      const double want = total * k / n;
      while (band < n - 1 && before + prev_cost[band] < want) before += prev_cost[band++];
      const double rows = prev_edges[band + 1] - prev_edges[band];
      const double y = prev_edges[band] + (want - before) / prev_cost[band] * rows;
      // damped: a frame's cost also carries what does not scale with its rows (allocations of a
      // new band shape, per-frame grids), so the edges move 60 % of the way
      out[k] = (int)(prev_edges[k] + 0.6 * (y - prev_edges[k]) + 0.5);
    }
  }
  for (int k = 1; k < n; ++k) {
    if (align > 1) out[k] = (out[k] + align / 2) / align * align;
    if (out[k] < out[k - 1]) out[k] = out[k - 1];
    if (out[k] > H) out[k] = H;
  }
}

static void multi_note_cost(b200_multi *mc, int kind, const std::vector<int> &edges, int H) {
  mc->edges[kind] = edges;
  mc->edges_h[kind] = H;
  mc->cost[kind].assign(mc->n, 0.f);
  for (int i = 0; i < mc->n; ++i) mc->cost[kind][i] = mc->child[i]->stats.gpu_ms;
}

static void multi_sum_stats(b200_ctx *ctx) {
  b200_multi *mc = ctx->multi;
  b200_stats s{};
  for (int i = 0; i < mc->n; ++i) {
    const b200_stats &c = mc->child[i]->stats;
    s.primary_rays += c.primary_rays; s.shadow_rays += c.shadow_rays; s.prim_tests += c.prim_tests;
    s.exact_evals += c.exact_evals; s.kernel_launches += c.kernel_launches; s.fragments += c.fragments;
    s.bin_entries += c.bin_entries; s.respeculated += c.respeculated;
    s.gpu_ms = c.gpu_ms > s.gpu_ms ? c.gpu_ms : s.gpu_ms;
  }
  ctx->stats = s;
}

extern "C" {

int b200_init_multi(int n_gpus, b200_ctx **out) {
  if (!out) return B200_EINVAL;
  *out = nullptr;
  int have = 0;
  if (cudaGetDeviceCount(&have) != cudaSuccess || have <= 0) return B200_ENODEV;
  if (n_gpus <= 0) n_gpus = have;
  if (n_gpus > have) return B200_EINVAL;
  if (n_gpus == 1) return b200_init(0, out);   // one device: an ordinary context, no threads in between
  if (const char *e = getenv("B200_MULTI_SPIN")) MULTI_SPIN = atoi(e);
  b200_ctx *ctx = new b200_ctx();
  b200_multi *mc = new b200_multi();
  ctx->multi = mc;
  ctx->device = 0;
  mc->n = n_gpus;
  mc->barrier.n = n_gpus;
  mc->phase_rc.assign(n_gpus, B200_OK);
  int rc = B200_OK;
  for (int i = 0; i < n_gpus && rc == B200_OK; ++i) {
    b200_ctx *c = nullptr;
    rc = b200_init(i, &c);
    if (rc == B200_OK) {
      mc->child.push_back(c);
      b200_set_option(c, B200_OPT_RAST_BAND_CULL, 1);   // every device's geometry stage keeps its band's triangles only
    }
  }
  // peer access between every pair (NVLink / NVSwitch): the rasteriser's scene all-gather
  mc->peer_ok = rc == B200_OK ? 1 : 0;
  for (int i = 0; i < n_gpus && rc == B200_OK; ++i) {
    cudaSetDevice(i);
    cudaEvent_t ev = nullptr;
    if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) { rc = B200_ECUDA; break; }
    mc->pushed.push_back(ev);
    for (int j = 0; j < n_gpus; ++j) {
      if (j == i) continue;
      int can = 0;
      cudaDeviceCanAccessPeer(&can, i, j);
      if (!can) { mc->peer_ok = 0; continue; }
      const cudaError_t e = cudaDeviceEnablePeerAccess(j, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) mc->peer_ok = 0;
      cudaGetLastError();
    }
  }
  if (rc == B200_OK)
    for (int i = 0; i < n_gpus; ++i) {
      MultiWorker *w = new MultiWorker();
      w->th = std::thread(worker_main, w, i);
      mc->worker.push_back(w);
    }
  if (rc != B200_OK) { b200_destroy(ctx); return rc; }
  cudaSetDevice(0);
  *out = ctx;
  return B200_OK;
}

int b200_device_count(const b200_ctx *ctx) { return !ctx ? 0 : (ctx->multi ? ctx->multi->n : 1); }

}  // extern "C"

void multi_destroy(b200_ctx *ctx) {
  b200_multi *mc = ctx->multi;
  for (MultiWorker *w : mc->worker) {
    { std::lock_guard<std::mutex> lk(w->m); w->quit = true; }
    w->cv.notify_all();
    w->th.join();
    delete w;
  }
  for (size_t i = 0; i < mc->pushed.size(); ++i) { cudaSetDevice((int)i); cudaEventDestroy(mc->pushed[i]); }
  for (b200_ctx *c : mc->child) b200_destroy(c);
  delete mc;
  ctx->multi = nullptr;
}

int multi_synchronize(b200_ctx *ctx) {
  return multi_run(ctx, [ctx](int i) { return b200_synchronize(ctx->multi->child[i]); });
}

int multi_set_option(b200_ctx *ctx, int option, int value) {
  int rc = B200_OK;
  for (b200_ctx *c : ctx->multi->child) {
    const int r = b200_set_option(c, option, value);
    if (r != B200_OK && rc == B200_OK) { rc = r; ctx->err = c->err; }
  }
  return rc;
}

// ---- raytracer ------------------------------------------------------------------------
int multi_raytrace(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres, int n_spheres,
                   const camera_t *cam, const light_t *lights, int n_lights, int row_begin, int row_end,
                   float *rgb_out, float *depth_out, int32_t *index_out, uint32_t *argb_out) {
  b200_multi *mc = ctx->multi;
  if (!cam || cam->width <= 0 || cam->height <= 0) return ctx_fail(ctx, B200_EINVAL, "bad camera");
  if (row_begin < 0 || row_end > cam->height || row_begin > row_end) return ctx_fail(ctx, B200_EINVAL, "bad row band");
  const int rows = row_end - row_begin, n = mc->n;
  std::vector<int> edges;
  // Large scenes run their blocks from a plan made of the previous frame's block costs, which every device keeps
  // for the rows IT rendered (rt_plan_kernel): the frame after a band moved is dearer on the rows it gained, and
  // balancing on that cost sent the edges back and forth (8 GPUs, 100 800 triangles: costs +-50 % from frame to
  // frame, never settled).  So the bands move only on the evidence of a frame that ran on the same bands as its
  // predecessor -- every other frame while they are still converging.
  const bool have = mc->edges_h[0] == rows && (int)mc->edges[0].size() == n + 1;
  if (have && !mc->settled[0]) edges = mc->edges[0];
  else multi_band_edges(have ? mc->edges[0] : std::vector<int>(), mc->cost[0], rows, n, 16, edges);
  mc->settled[0] = have && edges == mc->edges[0];
  const size_t W = (size_t)cam->width;
  const int rc = multi_run(ctx, [&](int i) -> int {
    const int a = row_begin + edges[i], b = row_begin + edges[i + 1];
    b200_ctx *c = mc->child[i];
    c->stats = b200_stats{};
    if (b <= a) return B200_OK;
    const size_t off = (size_t)(a - row_begin) * W;
    if (argb_out)
      return draw_raytrace_band(c, tris, n_tris, spheres, n_spheres, cam, lights, n_lights, a, b, argb_out + off);
    return render_raytrace_band(c, tris, n_tris, spheres, n_spheres, cam, lights, n_lights, a, b,
                                rgb_out ? rgb_out + 3 * off : nullptr, depth_out ? depth_out + off : nullptr,
                                index_out ? index_out + off : nullptr);
  });
  if (rc != B200_OK) return rc;
  multi_note_cost(mc, 0, edges, rows);
  multi_sum_stats(ctx);
  return B200_OK;
}

// Batched views: whole views go to whole devices -- device i renders the contiguous run [k_i, k_i+1) of the views
// with the single-device views path and returns it straight into its slice of the caller's buffers.  No bands.
int multi_raytrace_views(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres, int n_spheres,
                         const camera_t *cams, int n_views, const light_t *lights, int n_lights, float *rgb_out,
                         float *depth_out, int32_t *index_out, uint32_t *argb_out) {
  b200_multi *mc = ctx->multi;
  if (int rc = check_views(ctx, cams, n_views, lights, n_lights)) return rc;
  const size_t npix = (size_t)cams[0].width * cams[0].height;
  const int n = mc->n;
  const int rc = multi_run(ctx, [&](int i) -> int {
    const int a = (int)((long long)n_views * i / n), b = (int)((long long)n_views * (i + 1) / n);
    b200_ctx *c = mc->child[i];
    c->stats = b200_stats{};
    if (b <= a) return B200_OK;
    const size_t off = (size_t)a * npix;
    if (argb_out)
      return draw_raytrace_views(c, tris, n_tris, spheres, n_spheres, cams + a, b - a, lights, n_lights, argb_out + off);
    return render_raytrace_views(c, tris, n_tris, spheres, n_spheres, cams + a, b - a, lights, n_lights,
                                 rgb_out ? rgb_out + 3 * off : nullptr, depth_out ? depth_out + off : nullptr,
                                 index_out ? index_out + off : nullptr);
  });
  if (rc != B200_OK) return rc;
  multi_sum_stats(ctx);
  return B200_OK;
}

// Ray queries: device i answers the contiguous run [k_i, k_i+1) of the rays with the single-device entry and returns
// it straight into its slice of the caller's output, as multi_raytrace_views does with views.
int multi_rays(b200_ctx *ctx, const rt_triangle *tris, int n_tris, const rt_sphere *spheres, int n_spheres,
               const rt_ray *rays, const float *max_distance, int n_rays, rt_intersection *out, uint8_t *occ_out,
               bool occlusion) {
  b200_multi *mc = ctx->multi;
  if (int rc = check_rays(ctx, tris, n_tris, spheres, n_spheres, rays, max_distance, n_rays,
                          occlusion ? (const void *)occ_out : (const void *)out, occlusion))
    return rc;
  if (n_rays == 0) return B200_OK;
  const int n = mc->n;
  const int rc = multi_run(ctx, [&](int i) -> int {
    const int a = (int)((long long)n_rays * i / n), b = (int)((long long)n_rays * (i + 1) / n);
    b200_ctx *c = mc->child[i];
    c->stats = b200_stats{};
    if (b <= a) return B200_OK;
    if (occlusion) return rt_occluded(c, tris, n_tris, spheres, n_spheres, rays + a, max_distance + a, b - a, occ_out + a);
    return rt_closest_hits(c, tris, n_tris, spheres, n_spheres, rays + a, b - a, out + a);
  });
  if (rc != B200_OK) return rc;
  multi_sum_stats(ctx);
  return B200_OK;
}

// ---- rasteriser -------------------------------------------------------------------------
// Every device keeps its own copy of the images (each over its own PCIe link).
int multi_rast_set_textures(b200_ctx *ctx, const rast_textures_t *tex) {
  return multi_run(ctx, [&](int i) -> int { return rast_set_textures(ctx->multi->child[i], tex); });
}

int rast_band_resident(b200_ctx *ctx, const camera_t *cam, const rast_light_t *light, int row_begin, int row_end,
                       float *rgb_out, float *depth_out, int32_t *index_out, uint32_t *argb_out);   // api.cu

int multi_raster(b200_ctx *ctx, const rast_triangle *room, int n_room, const rast_triangle *boxes, int n_boxes,
                 const camera_t *cam, const rast_light_t *light, int row_begin, int row_end, float *rgb_out,
                 float *depth_out, int32_t *index_out, uint32_t *argb_out) {
  b200_multi *mc = ctx->multi;
  if (!cam || cam->width <= 0 || cam->height <= 0) return ctx_fail(ctx, B200_EINVAL, "bad camera");
  if (!light) return ctx_fail(ctx, B200_EINVAL, "null light");
  if (n_room < 0 || n_boxes < 0 || (n_room > 0 && !room) || (n_boxes > 0 && !boxes)) return ctx_fail(ctx, B200_EINVAL, "bad scene arguments");
  if (row_begin < 0 || row_end > cam->height || row_begin > row_end) return ctx_fail(ctx, B200_EINVAL, "bad row band");
  const int rows = row_end - row_begin, n = mc->n;
  std::vector<int> edges;
  // As for the raytracer, the bands move only on the evidence of a frame that ran on the bands of its predecessor:
  // the frame after a move cannot be pipelined (two host waits, sometimes reallocations -- a 75 ms frame was seen
  // on 8 GPUs when all devices grew their buffers at once), and balancing on its cost kept the edges moving.  The
  // tolerance is wider than the raytracer's: a band costs 0.10 - 0.12 ms, of which timing noise is a tenth.
  const bool have = mc->edges_h[1] == rows && (int)mc->edges[1].size() == n + 1;
  if (have && !mc->settled[1]) edges = mc->edges[1];
  else multi_band_edges(have ? mc->edges[1] : std::vector<int>(), mc->cost[1], rows, n, 8, edges, 1.12);
  mc->settled[1] = have && edges == mc->edges[1];
  const bool colour = mc->child[0]->opt_rast_colour != 0;
  if (colour) edges.assign(n + 1, rows), edges[0] = 0;   // colour modes number the fragments of the whole frame: one device draws it
  const size_t W = (size_t)cam->width;
  // slices of the room list: device i brings [s_i, s_i+1) over its own PCIe link
  const bool gather = mc->peer_ok && n > 1 && (size_t)n_room * sizeof(rast_triangle) >= ((size_t)1 << 20);
  const int rc = multi_run(ctx, [&](int i) -> int {
    b200_ctx *c = mc->child[i];
    c->stats = b200_stats{};
    int rc_i = B200_OK;
    if (!gather) {
      rc_i = rast_upload_scene(c, room, n_room, boxes, n_boxes);
    } else {
      // phase 1: every device's scene buffer exists at its final size
      rc_i = b200_synchronize(c);   // settles a pipelined frame still in flight (it may be rendered again: on ITS scene)
      if (rc_i == B200_OK) rc_i = ensure(c, c->rast_world, sizeof(rast_triangle) * ((size_t)n_room + (size_t)n_boxes + 1));
      mc->phase_rc[i] = rc_i;
      mc->barrier.wait();
      bool all_ok = true;
      for (int j = 0; j < n; ++j) all_ok = all_ok && mc->phase_rc[j] == B200_OK;
      // phase 2: own slice from the host, then on to every peer (NVLink); boxes are small: from the host
      if (all_ok) {
        const size_t s0 = (size_t)n_room * i / n, s1 = (size_t)n_room * (i + 1) / n;
        rast_triangle *mine = (rast_triangle *)c->rast_world.p;
        cudaError_t e = cudaSuccess;
        if (s1 > s0) e = cudaMemcpyAsync(mine + s0, room + s0, (s1 - s0) * sizeof(rast_triangle), cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess && n_boxes)
          e = cudaMemcpyAsync(mine + n_room, boxes, (size_t)n_boxes * sizeof(rast_triangle), cudaMemcpyHostToDevice, c->stream);
        for (int d = 1; d < n && e == cudaSuccess && s1 > s0; ++d) {
          const int j = (i + d) % n;   // staggered: at any moment every device receives from one peer
          e = cudaMemcpyPeerAsync((rast_triangle *)mc->child[j]->rast_world.p + s0, j, mine + s0, i,
                                  (s1 - s0) * sizeof(rast_triangle), c->stream);
        }
        if (e == cudaSuccess) e = cudaEventRecord(mc->pushed[i], c->stream);
        if (e != cudaSuccess) rc_i = ctx_fail(c, B200_ECUDA, "scene all-gather", e);
      }
      mc->phase_rc[i] = all_ok ? rc_i : B200_ECUDA;
      mc->barrier.wait();
      for (int j = 0; j < n; ++j) all_ok = all_ok && mc->phase_rc[j] == B200_OK;
      if (!all_ok) return rc_i != B200_OK ? rc_i : B200_ECUDA;
      // phase 3: the frame starts when every peer's slice has landed here
      for (int j = 0; j < n; ++j)
        if (j != i && cudaStreamWaitEvent(c->stream, mc->pushed[j], 0) != cudaSuccess) return ctx_fail(c, B200_ECUDA, "cudaStreamWaitEvent");
      c->rast_n_room = n_room;
      c->rast_n_boxes = n_boxes;
      c->rast_has_shadow = n_boxes > 0;
    }
    if (rc_i != B200_OK) return rc_i;
    const int a = row_begin + edges[i], b = row_begin + edges[i + 1];
    if (b <= a) return b200_synchronize(c);
    const size_t off = (size_t)(a - row_begin) * W;
    return rast_band_resident(c, cam, light, a, b, rgb_out ? rgb_out + 3 * off : nullptr, depth_out ? depth_out + off : nullptr,
                              index_out ? index_out + off : nullptr, argb_out ? argb_out + off : nullptr);
  });
  if (rc != B200_OK) return rc;
  if (!colour) multi_note_cost(mc, 1, edges, rows);
  multi_sum_stats(ctx);
  return B200_OK;
}

// Band edges and per-device cost (ms) of the last frame of `kind` (0 RT, 1 RAST): diagnostics.
extern "C" int b200_debug_multi_bands(b200_ctx *ctx, int kind, int *edges_out, float *cost_out, int cap) {
  if (!ctx || !ctx->multi || kind < 0 || kind > 1) return B200_EINVAL;
  const b200_multi *mc = ctx->multi;
  const int n = (int)mc->cost[kind].size();
  for (int i = 0; i < n && i < cap; ++i) { edges_out[i] = mc->edges[kind][i + 1]; cost_out[i] = mc->cost[kind][i]; }
  return n;
}

// The band-split rule itself, callable without a device (host logic; CPU tests).
extern "C" int b200_debug_band_edges(const int *prev_edges, const float *prev_cost, int n_prev, int H, int n, int align, int *out) {
  if (!out || n <= 0 || H < 0) return B200_EINVAL;
  std::vector<int> pe, o;
  std::vector<float> pc;
  if (prev_edges && prev_cost && n_prev == n) { pe.assign(prev_edges, prev_edges + n + 1); pc.assign(prev_cost, prev_cost + n); }
  multi_band_edges(pe, pc, H, n, align, o);
  for (int i = 0; i <= n; ++i) out[i] = o[i];
  return B200_OK;
}
