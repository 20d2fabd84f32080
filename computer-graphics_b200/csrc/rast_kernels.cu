// Rasteriser hot path on sm_100a: replaces the triangle loop and post pass of
// rasteriser/Source/skeleton.cpp Draw :243-307 (DrawPolygon :420-431,
// VertexShader :510-522, ComputePolygonRows :433-498, Interpolate :524-551,
// DrawPolygonRows :500-508, PixelShader :559-672, calculateIllumination
// :674-688, surroundingShadowSum :1725-1733, antiAliasing :1736-1753).
//
// The reference draws triangles strictly in list order into global buffers; the
// result at a pixel is a fold over that pixel's fragments in triangle order:
//   opaque  : accepted when zinv >= depth  => winner = max zinv, LATEST on ties
//   shadow  : sets the pixel's flag when zinv > depth *as it stands then*
// Pixels are independent, so the fold is done per pixel by one thread, over the
// pixel's screen tile's triangle list in ascending index order.  Only the
// depth test runs per fragment; shading is deferred to the single winning
// fragment (the reference overwrites the colours of every earlier one).
//
// Coverage is the reference's float edge walk, reproduced exactly but in closed
// form: along an edge one of x / y moves by exactly +-1 per sample, so per
// (edge, row) the samples that land in the row form one run whose two ends are
// found directly (rast_row_record); the reference's min-x / max-x "last equal
// sample wins" rule is then replayed on at most six samples.
//
// Kernels per frame:
//   rast_short_kernel   per triangle of a list of at most 2048: setup record, row records
//                       and the bits of the tiles it touches, in one launch
//   rast_setup_kernel   per triangle of a longer list: VertexShader, row range,
//                       row-table space (and, above 8192 triangles, the owners of its rows)
//   rast_spread_kernel  per triangle fan-out: owners of its row slots, tile counts,
//                       tile lists (atomics)
//   rast_scan_kernel    exclusive scan of tile counts
//   rast_rows_kernel    per row slot: left/right span ends + steps
//   rast_fill_kernel    per tile: sort list, depth/shadow fold, deferred shading
//   rast_resolve_kernel per 32x8 pixels (rast_fast.cuh): shading of the winners, shadow
//                       softening + 5-tap AA + "HDR" mean (:283-307)
//   rast_post_kernel    the same post pass from the six intermediate buffers
#include "common.cuh"
#include <limits.h>
#include <stdlib.h>
#include <vector>
#include "rast_tex.cuh"

constexpr int RAST_LIST_CAP = 2048;   // tile list entries sorted in shared memory
constexpr int RAST_BATCH = 32;        // triangles per shared-memory row batch

struct RastVtx {
  int x, y;
  float zinv, px, py;
};

struct RastSetup {
  RastVtx v[3];
  int ymin;          // smallest vertex y (row 0 of the reference's row table)
  int row0;          // first stored row (clamped to the band being rendered)
  int nrows;         // stored rows (0: nothing to draw)
  unsigned row_off;  // index of the first stored row in the row arrays
  int flags;         // bit0: shadow-volume triangle (colour.x < 0)
  // Interpolate's per-edge steps for edge e = v[e] -> v[(e+1)%3] with
  // N = max(|dx|,|dy|)+1 samples (:533-538): they depend on the edge only
  float sx[3], sy[3], sz[3], spx[3], spy[3];
  int tri;           // scatter path: list index of this (big) triangle; setup records are indexed by big-list position
  float pad[4];
};
// 40 words: rast_setup_kernel's shared-memory staging (record stride 41, conflict-free) and rast_short_kernel's
// word stream (lane k: words k and k + 32) are laid out for that size
static_assert(sizeof(RastSetup) == 160, "RastSetup is 160 bytes");

struct RastParams {
  int W, H;
  int fb0, fb1;      // rows the fill pass must produce (band + post-pass halo)
  int row0, row1;    // rows the post pass writes
  int ts_log2;       // screen-tile size (log2)
  int tiles_x, tiles_y, ty0;  // tile grid; ty0 = first tile row of the band
  float focal;
  float light[4];
  float power[3];
  float indirect[3];   // indirectLightPowerPerArea as it stands when Draw is entered
  // PixelShader leaves the global at 0.2 (:585), so only the first shaded fragment of a Draw sees
  // the entry value: (triangle << 32 | pixel) of that fragment, or null when the entry value is 0.2
  const unsigned long long *first_frag;
  const rast_triangle *src;
  int n_tris;
  RastSetup *setup;
  float4 *rowsA;     // lx, rx (bit-cast ints), left zinv, zinv step (ordered path only)
  float4 *rowsB;     // left px*zinv, its step, left py*zinv, its step
  unsigned row_cap;
  unsigned long long *keys;   // fast path: per-pixel (zinv bits, triangle + 1)
  int *rowsL;        // fast path: left x of every stored row (big triangles; rowsB likewise)
  float4 *srowsB;    // fast path, small triangles: row records at triangle * S2_ROWS + y mod S2_ROWS
  int *srowsL;
  int2 *trimeta;     // fast path: per triangle, index of its first stored row and that row's y
  // scatter of one geometry chunk: the list range [*range_lo, *range_hi) (null: the whole list)
  const unsigned long long *range_lo, *range_hi;
  const int *orig;   // band-culled list: index of every triangle in the complete list (null: the list is complete)
  int *big_list;     // fast path: triangles too large for rast_scatter2_kernel's shared-memory row table
  unsigned big_cap;
  int *row_owner;    // per slot of the row tables: the triangle (fast path: big-list position) that owns it
  unsigned n_rows;   // row slots claimed
  // pipelined mode: the list length / row count are not known on the host yet; n_tris and
  // n_rows above are then launch bounds and the kernels clamp to these device values
  const unsigned long long *n_tris_dev, *n_rows_dev;
  int spread_in_setup;   // long lists: rast_setup_kernel names the owners of its rows itself (no rast_spread_kernel<0>)
  unsigned *tile_count, *tile_off, *tile_cursor;
  // short lists (n_tris <= RAST_BITS_MAX_TRIS): a tile's list is a bit per triangle -- no count /
  // scan / append passes and nothing to sort, the bits come out in list order
  unsigned *tile_bits;
  int bits_words;    // words per tile (0: the list representation above)
  int *bins, *bins_tmp;
  unsigned bin_cap;
  float *depth, *screen, *low, *high;
  int *shadow, *index;
  // ordered path, fused (the default): the fold leaves one word per pixel in `keys` (depth bits << 32 |
  // winner + 1) and a shadow flag per pixel; rast_resolve_kernel<true> shades and post-processes from those
  int fused;
  unsigned char *shadow8;
  float *out_rgb;
  float *out_depth;
  int *out_index;
  uint32_t *out_argb;
  int tex_on;        // rast_set_textures: the triangles' texture / index fields are honoured (ordered path only)
  RastTex tex;
  // Colour modes 1 / 2 (randColourSelect, :647-662; B200_OPT_RAST_COLOUR_MODE): every ACCEPTED fragment draws three
  // rand() values, in the serial order of the reference's loops (triangle, row, x).  The fold counts the accepted
  // fragments ([17]), a second fold emits their keys (triangle << 24 | y << 12 | x), the sorted keys give every
  // winner its ordinal and colour_rgb[ordinal] is the colour vector the host drew for it.
  int colour_mode;
  unsigned long long *colour_emit;          // emit pass: where the keys go (cursor: counters[18]); null otherwise
  const unsigned long long *colour_sorted;  // resolve: the sorted keys
  unsigned long long colour_n;
  const float *colour_rgb;                  // 3 floats per ordinal
  unsigned long long *counters;  // [3] bin entries, [4] rows, [5] overflow flag, [9] first shaded fragment, [10] big triangles, [11] their rows (counting pass), second cache line: [16] fragments (updated while [4] is read), [24] list length (read while [4] is updated)
};

__device__ __forceinline__ int rast_count_tris(const RastParams &p) {
  return p.n_tris_dev ? (int)min((unsigned long long)p.n_tris, *p.n_tris_dev) : p.n_tris;
}
__device__ __forceinline__ unsigned rast_count_rows(const RastParams &p) {
  return p.n_rows_dev ? (unsigned)min((unsigned long long)p.n_rows, *p.n_rows_dev) : p.n_rows;
}

// ---- VertexShader (:510-522) ---------------------------------------------------------
__device__ __forceinline__ bool rast_vertex(const float *v, float focal, int W, int H, RastVtx &o) {
  const float x = xadd(xmul(focal, xdiv(v[0], v[2])), (float)(W / 2));
  const float y = xadd(xmul(focal, xdiv(v[1], v[2])), (float)(H / 2));
  // static_cast<int> of a value outside int range (or NaN) is undefined in the reference; such
  // triangles are dropped.  Everything inside converts and is drawn as the reference draws it:
  // the far plane's (w1 - w0) divisor (:1615) can put a clipped vertex of finite scene input
  // tens of millions of pixels off screen (5e7 at W = 32768, tests/test_rast_clip_gpu.py)
  if (!(fabsf(x) < 2147483648.0f) || !(fabsf(y) < 2147483648.0f)) return false;
  o.x = (int)x;
  o.y = (int)y;
  o.zinv = xdiv(1.0f, v[2]);
  o.px = v[0];
  o.py = v[1];
  return true;
}

// Every lane brings a range of `n` work items described by four ints; ranges of up to
// 32 items are walked by their own lane, longer ones (a triangle covering thousands
// of tiles or rows) are spread over the whole warp.  All 32 lanes must call this.
template <typename F>
__device__ __forceinline__ void warp_spread(int n, int a, int b, int c, int d, F body) {
  const int lane = threadIdx.x & 31;
  if (n <= 32) for (int k = 0; k < n; ++k) body(k, a, b, c, d);
  unsigned big = __ballot_sync(0xffffffffu, n > 32);
  while (big) {
    const int src = __ffs(big) - 1;
    big &= big - 1;
    const int ns = __shfl_sync(0xffffffffu, n, src);
    const int as = __shfl_sync(0xffffffffu, a, src), bs = __shfl_sync(0xffffffffu, b, src);
    const int cs = __shfl_sync(0xffffffffu, c, src), ds = __shfl_sync(0xffffffffu, d, src);
    for (int k = lane; k < ns; k += 32) body(k, as, bs, cs, ds);
  }
}

// VertexShader of the three vertices and Interpolate's per-edge steps (:531-538) of one clipped
// triangle (tr: v0[4] v1[4] v2[4] normal[4] color[3] as floats).  false: a vertex does not
// convert to int (the triangle is dropped).
__device__ __forceinline__ bool rast_tri_setup(const float *tr, float focal, int W, int H, RastSetup &s) {
  float v[3][3];
#pragma unroll
  for (int k = 0; k < 3; ++k) { v[0][k] = tr[k]; v[1][k] = tr[4 + k]; v[2][k] = tr[8 + k]; }
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 3; ++k) ok = rast_vertex(v[k], focal, W, H, s.v[k]) && ok;
  s.flags = tr[16] < 0 ? 1 : 0;
#pragma unroll
  for (int e = 0; e < 3; ++e) {                                  // Interpolate :531-538, per edge
    const RastVtx &a = s.v[e], &b = s.v[(e + 1) % 3];
    const float den = (float)max(max(abs(a.x - b.x), abs(a.y - b.y)), 1);
    const float apx = xmul(a.px, a.zinv), apy = xmul(a.py, a.zinv);
    const float bpx = xmul(b.px, b.zinv), bpy = xmul(b.py, b.zinv);
    s.sx[e] = xdiv_pos((float)(b.x - a.x), den);
    s.sy[e] = xdiv_pos((float)(b.y - a.y), den);
    s.sz[e] = xdiv_pos(xsub(b.zinv, a.zinv), den);
    s.spx[e] = xdiv_pos(xsub(bpx, apx), den);
    s.spy[e] = xdiv_pos(xsub(bpy, apy), den);
  }
  return ok;
}

constexpr int RAST_BITS_MAX_TRIS = 2048;
constexpr int SETUP_THREADS = 256;
constexpr int TRI_WORDS = sizeof(rast_triangle) / 4, SETUP_WORDS = sizeof(RastSetup) / 4;

__global__ void __launch_bounds__(SETUP_THREADS) rast_setup_kernel(const __grid_constant__ RastParams p) {
  // The 84-byte triangles and the 160-byte setup records are staged through shared
  // memory so that global memory only sees fully coalesced word streams.
  __shared__ uint32_t stage[SETUP_THREADS * (SETUP_WORDS + 1)];   // +1: conflict-free record stride
  const int t0 = blockIdx.x * SETUP_THREADS;
  const int t = t0 + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const int n_tris = rast_count_tris(p);
  if (t0 >= n_tris) return;   // pipelined launches are sized by a bound on the list length
  const int n_here = min(SETUP_THREADS, n_tris - t0);
  {
    const uint32_t *src = reinterpret_cast<const uint32_t *>(p.src + t0);
    for (int i = threadIdx.x; i < n_here * TRI_WORDS; i += SETUP_THREADS) stage[i] = __ldg(src + i);
  }
  __syncthreads();
  int nrows = 0;
  RastSetup s;
  s.flags = 0; s.ymin = 0; s.row0 = 0; s.nrows = 0; s.row_off = 0; s.tri = t;
  int xmin = 0, xmax = -1;
  if (t < n_tris) {
    const float *tr = reinterpret_cast<const float *>(stage) + threadIdx.x * TRI_WORDS;   // v0[4] v1[4] v2[4] normal[4] color[3]
    const bool ok = rast_tri_setup(tr, p.focal, p.W, p.H, s);
    if (ok) {
      const int ymin = min(s.v[0].y, min(s.v[1].y, s.v[2].y));
      const int ymax = max(s.v[0].y, max(s.v[1].y, s.v[2].y));
      xmin = min(s.v[0].x, min(s.v[1].x, s.v[2].x)) - 1;   // a minor-axis sample can undershoot by one
      xmax = max(s.v[0].x, max(s.v[1].x, s.v[2].x));
      s.ymin = ymin;
      s.row0 = max(ymin, p.fb0);
      const int rlast = min(ymax, p.fb1 - 1);
      nrows = max(0, rlast - s.row0 + 1);
      if (xmax <= 0 || xmin >= p.W || xmax <= xmin) nrows = 0;   // no pixel of [xmin, xmax) on screen
    }
    s.nrows = nrows;
  }
  // row-table space: one atomic per warp
  unsigned incl = (unsigned)nrows;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned n = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += n;
  }
  const unsigned total = __shfl_sync(0xffffffffu, incl, 31);
  unsigned base = 0;
  if (lane == 31 && total) base = (unsigned)atomicAdd(p.counters + 4, (unsigned long long)total);
  base = __shfl_sync(0xffffffffu, base, 31);
  s.row_off = base + incl - (unsigned)nrows;
  if (t < n_tris && s.row_off + (unsigned)nrows > p.row_cap) {
    s.nrows = 0; nrows = 0;
    atomicExch(p.counters + 5, 1ull);
  }
  if (p.spread_in_setup)   // the owner of each of the triangle's row slots, for rast_rows_kernel
    warp_spread(nrows, (int)s.row_off, 0, 0, t, [&](int k, int x0, int, int, int tri) { p.row_owner[(unsigned)x0 + k] = tri; });
  __syncthreads();   // every thread has read its triangle: the buffer now carries the records out
  if (t < n_tris) {
    const uint32_t *w = reinterpret_cast<const uint32_t *>(&s);
#pragma unroll
    for (int k = 0; k < SETUP_WORDS; ++k) stage[threadIdx.x * (SETUP_WORDS + 1) + k] = w[k];
  }
  __syncthreads();
  {
    uint32_t *dst = reinterpret_cast<uint32_t *>(p.setup + t0);
    for (int i = threadIdx.x; i < n_here * SETUP_WORDS; i += SETUP_THREADS)
      dst[i] = stage[(i / SETUP_WORDS) * (SETUP_WORDS + 1) + i % SETUP_WORDS];
  }
}

// ---- closed-form edge walk -------------------------------------------------------------
struct RastEdge {
  int ax, ay, n;       // start pixel, sample count
  float sx, sy, den;
};

__device__ __forceinline__ int edge_px(const RastEdge &e, int i) {
  return (int)floorf(xadd((float)e.ax, xmul(e.sx, (float)i)));   // :541
}
__device__ __forceinline__ int edge_py(const RastEdge &e, int i) {
  return (int)floorf(xadd((float)e.ay, xmul(e.sy, (float)i)));   // :542
}

// Smallest i in [0, n] with (up ? y(i) >= Y : y(i) <= Y); y(i) is monotone in i.
__device__ __forceinline__ int edge_first(const RastEdge &e, int Y, bool up) {
  // An estimate from the real-number condition; the loops below make it exact in the
  // reference's float arithmetic.  up: a + s*i >= Y  <=>  i >= (Y - a)/s.
  // down (s < 0): floor(a + s*i) <= Y  <=>  a + s*i < Y + 1  <=>  i > (Y + 1 - a)/s.
  const float est = up ? ceilf(__fdividef((float)(Y - e.ay), e.sy))
                       : floorf(__fdividef((float)(Y + 1 - e.ay), e.sy)) + 1.0f;
  int i = est >= 0.f ? (est <= (float)e.n ? (int)est : e.n) : 0;   // NaN -> 0
  if (up) {
    while (i > 0 && edge_py(e, i - 1) >= Y) --i;
    while (i < e.n && edge_py(e, i) < Y) ++i;
  } else {
    while (i > 0 && edge_py(e, i - 1) <= Y) --i;
    while (i < e.n && edge_py(e, i) > Y) ++i;
  }
  return i;
}

// The samples of edge a->b (Interpolate with N = max(|dx|,|dy|)+1, :472-479) whose
// floor(y) equals Y form one run [i0, i1]; returns false when the run is empty.
__device__ __forceinline__ bool edge_run(const RastSetup &s, int ei, int Y, RastEdge &e, int &i0, int &i1) {
  const RastVtx &a = s.v[ei], &b = s.v[(ei + 1) % 3];
  const int dx = abs(a.x - b.x), dy = abs(a.y - b.y);
  e.ax = a.x; e.ay = a.y;
  e.n = max(dx, dy) + 1;
  e.den = (float)max(e.n - 1, 1);
  e.sx = s.sx[ei];   // :533, computed once per edge by rast_setup_kernel
  e.sy = s.sy[ei];   // :534
  if (dy == 0) {                     // step_y = 0: every sample is in row a.y
    if (Y != a.y) return false;
    i0 = 0; i1 = e.n - 1;
    return true;
  }
  if (dy >= dx) {                    // step_y = +-1 exactly: one sample per row
    const int i = b.y > a.y ? Y - a.y : a.y - Y;
    if (i < 0 || i > e.n - 1) return false;
    i0 = i1 = i;
    return true;
  }
  if (e.n <= 8) {
    // |step_y| < 1, short edge (every edge of a small triangle): look at all samples, branch-free;
    // y(i) is monotone, so the samples with y == Y are the run the searches below would find
    int lo = 8, hi = -1;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const bool in = i < e.n && edge_py(e, i) == Y;
      lo = in ? min(lo, i) : lo;
      hi = in ? i : hi;
    }
    i0 = lo; i1 = hi;
    return hi >= 0;
  }
  const bool up = b.y > a.y;         // |step_y| < 1: a run of samples per row
  i0 = edge_first(e, Y, up);
  i1 = edge_first(e, up ? Y + 1 : Y - 1, up) - 1;
  return i0 <= i1 && i0 < e.n;
}

struct RastEnd { int x, e, i; };

// Row Y of ComputePolygonRows' table (:481-495) and the span steps that
// DrawPolygonRows' Interpolate derives from it (:502-503, :524-538).
template <bool WITH_POS = true>
__device__ __forceinline__ void rast_row_record(const RastSetup &s, int Y, float4 &A, float4 &B) {
  RastEnd L, R;
  L.x = INT_MAX; L.e = -1; L.i = 0;
  R.x = -INT_MAX; R.e = -1; R.i = 0;
#pragma unroll
  for (int e = 0; e < 3; ++e) {
    RastEdge ed;
    int i0, i1;
    if (!edge_run(s, e, Y, ed, i0, i1)) continue;
    const int x0 = edge_px(ed, i0);
    if (x0 <= L.x) { L.x = x0; L.e = e; L.i = i0; }
    if (x0 >= R.x) { R.x = x0; R.e = e; R.i = i0; }
    if (i1 > i0) {
      const int x1 = edge_px(ed, i1);
      if (x1 <= L.x) { L.x = x1; L.e = e; L.i = i1; }
      if (x1 >= R.x) { R.x = x1; R.e = e; R.i = i1; }
    }
  }
  if (L.e < 0) {   // unreachable for a valid triangle: every row receives a sample
    A = make_float4(__int_as_float(0), __int_as_float(0), 0.f, 0.f);
    B = make_float4(0.f, 0.f, 0.f, 0.f);
    return;
  }
  float zinv[2], px[2], py[2];
#pragma unroll
  for (int side = 0; side < 2; ++side) {
    const RastEnd &E = side ? R : L;
    const RastVtx &a = s.v[E.e];
    const float fi = (float)E.i;
    zinv[side] = xadd(a.zinv, xmul(s.sz[E.e], fi));                   // :543 (step_z :535 from setup)
    if (WITH_POS) {
      const float apx = xmul(a.px, a.zinv), apy = xmul(a.py, a.zinv);   // :526-527
      px[side] = xdiv(xadd(apx, xmul(s.spx[E.e], fi)), zinv[side]);     // :547 (steps :537-538 from setup)
      py[side] = xdiv(xadd(apy, xmul(s.spy[E.e], fi)), zinv[side]);     // :548
    }
  }
  const int n = R.x - L.x + 1;
  const float den = (float)max(n - 1, 1);
  A = make_float4(__int_as_float(L.x), __int_as_float(R.x), zinv[0], xdiv_pos(xsub(zinv[1], zinv[0]), den));
  if (WITH_POS) {
    const float lpx = xmul(px[0], zinv[0]), lpy = xmul(py[0], zinv[0]);
    const float rpx = xmul(px[1], zinv[1]), rpy = xmul(py[1], zinv[1]);
    B = make_float4(lpx, xdiv_pos(xsub(rpx, lpx), den), lpy, xdiv_pos(xsub(rpy, lpy), den));
  }
}

// ---- the first shaded fragment of the Draw ---------------------------------------------------
// PixelShader shades with the global indirectLightPowerPerArea and then sets it to 0.2 (:580,
// :585), so the value the caller left in the global reaches exactly one fragment: the first
// one accepted, i.e. (the depth buffer is still clear, :247) the first in-bounds fragment with
// zinv >= 0 of the first opaque triangle that has one, rows top to bottom, x left to right
// (:500-508).  Only launched when the entry value differs from 0.2.  Whole frame, never a band.
__device__ __forceinline__ float rast_indirect(const RastParams &p, int k, int tri, size_t q) {
  constexpr float steady = 0.2f * 1.0f;                                            // :585
  if (!p.first_frag) return steady;
  return (((unsigned long long)(unsigned)tri << 32) | (unsigned long long)q) == *p.first_frag ? p.indirect[k] : steady;
}

__global__ void rast_first_fragment_kernel(const __grid_constant__ RastParams p, unsigned long long *first) {
  const int t = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  if (t >= rast_count_tris(p)) return;
  if (((unsigned long long)(unsigned)t << 32) > *(volatile unsigned long long *)first) return;   // an earlier triangle has one
  const float *tr = reinterpret_cast<const float *>(p.src + t);
  if (!(tr[16] >= 0.0f)) return;                                                   // opaque triangles only (:574)
  RastSetup s;
  if (!rast_tri_setup(tr, p.focal, p.W, p.H, s)) return;
  const int ymin = min(s.v[0].y, min(s.v[1].y, s.v[2].y)), ymax = max(s.v[0].y, max(s.v[1].y, s.v[2].y));
  const int xmin = min(s.v[0].x, min(s.v[1].x, s.v[2].x)) - 1, xmax = max(s.v[0].x, max(s.v[1].x, s.v[2].x));
  if (xmax <= 0 || xmin >= p.W || xmax <= xmin) return;
  s.ymin = ymin;
  // textures: a hole of a metal-grill / woven-wood triangle is accepted but not shaded (:603, :625) and leaves
  // the depth buffer clear (:619, :643), so the search goes on behind it
  const int texture = p.tex_on ? __float_as_int(tr[19]) : 0, index = __float_as_int(tr[20]);
  const bool holes = texture == 2 || texture == 3;
  for (int y = max(ymin, 0); y <= min(ymax, p.H - 1); ++y) {
    float4 A, B;
    if (holes) rast_row_record<true>(s, y, A, B);
    else rast_row_record<false>(s, y, A, B);
    const int lx = __float_as_int(A.x), rx = __float_as_int(A.y);
    for (int x = max(lx, 0); x < min(rx, p.W); ++x) {
      const float fi = (float)(x - lx);
      const float zinv = xadd(A.z, xmul(A.w, fi));
      if (zinv >= 0.0f) {
        if (holes && rast_tex_hole(p.tex, texture, index, xdiv(xadd(B.x, xmul(B.y, fi)), zinv),
                                   xdiv(xadd(B.z, xmul(B.w, fi)), zinv), xdiv(1.0f, zinv)))
          continue;
        atomicMin(first, ((unsigned long long)(unsigned)t << 32) | (unsigned long long)((size_t)y * p.W + x));
        return;
      }
    }
  }
}

// One thread per row slot: the owner table names its triangle, so tall triangles
// spread over many threads.
__global__ void rast_rows_kernel(const __grid_constant__ RastParams p) {
  const unsigned slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= rast_count_rows(p)) return;
  const int t = p.row_owner[slot];
  if ((unsigned)t >= (unsigned)p.n_tris) return;   // slot of a triangle dropped on overflow (stale owner)
  const RastSetup &s = p.setup[t];
  const int r = (int)(slot - s.row_off);
  if (r < 0 || r >= s.nrows) return;
  float4 A, B;
  rast_row_record(s, s.row0 + r, A, B);
  p.rowsA[slot] = A;
  p.rowsB[slot] = B;
}

// ---- short lists: everything between the clipped list and the fold in one launch ----------------
// A list of at most RAST_BITS_MAX_TRIS triangles (the reference's own scene: ~300 clipped triangles, most of them
// shadow-volume sides that span the screen) went through four dependent launches of a few microseconds of work
// each -- rast_setup_kernel, two rast_spread_kernel, rast_rows_kernel: 38 of the 114 us of a 900 x 720 frame.
// Here one block takes a triangle: every thread derives the setup record (VertexShader, the per-edge steps: the
// same values in every thread), then the threads share out the row records (rast_row_record) and the bits of the
// screen tiles the bounding box touches.  Row-table space is not claimed but fixed -- triangle t owns rows
// [t * band, (t + 1) * band) of the table (at most 2048 x band rows) -- so nothing in the block waits.
// (One block per (triangle, 128 rows) instead of a loop over the rows: measured slower, 22 700 mostly empty
// blocks at 4K.)
constexpr int SHORT_THREADS = 256;
__global__ void __launch_bounds__(SHORT_THREADS) rast_short_kernel(const __grid_constant__ RastParams p) {
  const int t = (int)blockIdx.x;
  if (t >= rast_count_tris(p)) return;   // pipelined launches are sized by a bound on the list length
  float trl[19];                         // v0[4] v1[4] v2[4] normal[4] color[3]
  {
    const float *tr = reinterpret_cast<const float *>(p.src + t);
#pragma unroll
    for (int k = 0; k < 19; ++k) trl[k] = __ldg(tr + k);
  }
  RastSetup s;
  const bool ok = rast_tri_setup(trl, p.focal, p.W, p.H, s);
  int nrows = 0, xmin = 0, xmax = -1, row0 = 0, ymin = 0;
  if (ok) {
    ymin = min(s.v[0].y, min(s.v[1].y, s.v[2].y));
    const int ymax = max(s.v[0].y, max(s.v[1].y, s.v[2].y));
    xmin = min(s.v[0].x, min(s.v[1].x, s.v[2].x)) - 1;   // a minor-axis sample can undershoot by one
    xmax = max(s.v[0].x, max(s.v[1].x, s.v[2].x));
    row0 = max(ymin, p.fb0);
    const int rlast = min(ymax, p.fb1 - 1);
    nrows = max(0, rlast - row0 + 1);
    if (xmax <= 0 || xmin >= p.W || xmax <= xmin) nrows = 0;   // no pixel of [xmin, xmax) on screen
  }
  s.ymin = ymin; s.row0 = row0; s.nrows = nrows;
  s.row_off = (unsigned)t * (unsigned)(p.fb1 - p.fb0) + (unsigned)(row0 - p.fb0);
  s.tri = t;
  s.pad[0] = s.pad[1] = s.pad[2] = s.pad[3] = 0.f;
  for (int r = threadIdx.x; r < nrows; r += SHORT_THREADS) {
    float4 A, B;
    rast_row_record(s, row0 + r, A, B);
    p.rowsA[s.row_off + r] = A;
    p.rowsB[s.row_off + r] = B;
  }
  if (threadIdx.x < 32) {   // the 160-byte record leaves as one coalesced word stream (lane k: words k and k + 32)
    const uint32_t *w = reinterpret_cast<const uint32_t *>(&s);
    uint32_t *dst = reinterpret_cast<uint32_t *>(p.setup + t);
#pragma unroll
    for (int k = 0; k < SETUP_WORDS; ++k)
      if ((k & 31) == (int)threadIdx.x) dst[k] = w[k];
  }
  if (threadIdx.x == 0 && nrows > 0)   // statistics, and what a later frame of another shape sizes its launches from
    atomicAdd(p.counters + 4, (unsigned long long)nrows);
  if (nrows > 0) {
    const int ts = p.ts_log2;
    const int a = max(0, xmin) >> ts;                               // first tile column
    const int w = (min(p.W - 1, xmax - 1) >> ts) - a + 1;           // tile columns
    const int c = row0 >> ts;                                       // first tile row
    const int n = w * (((row0 + nrows - 1) >> ts) - c + 1);
    for (int k = threadIdx.x; k < n; k += SHORT_THREADS) {
      const size_t tile = (size_t)(c + k / w - p.ty0) * p.tiles_x + a + k % w;
      atomicOr(p.tile_bits + tile * p.bits_words + (t >> 5), 1u << (t & 31));
    }
  }
}

// ---- tile lists ---------------------------------------------------------------------------
__global__ void rast_scan_kernel(const __grid_constant__ RastParams p, int n_tiles) {
  __shared__ unsigned warp_excl[32];
  __shared__ unsigned chunk_total;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  unsigned carry = 0;   // identical in every thread
  for (int base = 0; base < n_tiles; base += blockDim.x) {
    const int i = base + threadIdx.x;
    const unsigned v = i < n_tiles ? p.tile_count[i] : 0u;
    unsigned incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned n = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += n;
    }
    if (lane == 31) warp_excl[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      const unsigned w = lane < nw ? warp_excl[lane] : 0u;
      unsigned wi = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned n = __shfl_up_sync(0xffffffffu, wi, o);
        if (lane >= o) wi += n;
      }
      warp_excl[lane] = wi - w;
      if (lane == 31) chunk_total = wi;
    }
    __syncthreads();
    if (i < n_tiles) { p.tile_off[i] = carry + warp_excl[warp] + incl - v; p.tile_cursor[i] = 0; }
    carry += chunk_total;
    __syncthreads();
  }
  if (threadIdx.x == 0) { p.tile_off[n_tiles] = carry; p.counters[3] = carry; }
}

// Per-triangle fan-out work: WHAT = 0 names the triangle as the owner of its row slots
// (row_owner, for rast_rows_kernel), 1 counts the screen tiles its bounding box touches,
// 2 appends it to those tiles' lists.  Two launch shapes: one thread per triangle (long lists;
// outliers are spread over the warp) or one block per triangle (short lists of big
// triangles, e.g. the Cornell box with its shadow volumes at 4K).
template <int WHAT>
__global__ void rast_spread_kernel(const __grid_constant__ RastParams p, int block_per_tri) {
  const int t = block_per_tri ? (int)blockIdx.x : (int)(blockIdx.x * blockDim.x + threadIdx.x);
  int n = 0, a = 0, b = 1, c = 0;
  if (t < rast_count_tris(p)) {
    const RastSetup &s = p.setup[t];
    if (WHAT == 0) {
      n = s.nrows;
      a = (int)s.row_off;
    } else if (s.nrows > 0) {
      const int ts = p.ts_log2;
      const int xmin = min(s.v[0].x, min(s.v[1].x, s.v[2].x)) - 1;
      const int xmax = max(s.v[0].x, max(s.v[1].x, s.v[2].x));
      a = max(0, xmin) >> ts;                                   // first tile column
      b = (min(p.W - 1, xmax - 1) >> ts) - a + 1;               // tile columns
      c = s.row0 >> ts;                                         // first tile row
      n = b * (((s.row0 + s.nrows - 1) >> ts) - c + 1);
    }
  }
  auto body = [&](int k, int x0, int w, int y0, int tri) {
    if (WHAT == 0) { p.row_owner[(unsigned)x0 + k] = tri; return; }
    const size_t tile = (size_t)(y0 + k / w - p.ty0) * p.tiles_x + x0 + k % w;
    if (WHAT == 1) { atomicAdd(p.tile_count + tile, 1u); return; }
    const unsigned pos = atomicAdd(p.tile_cursor + tile, 1u);
    const unsigned at = p.tile_off[tile] + pos;
    if (at < p.bin_cap) p.bins[at] = tri;
  };
  if (block_per_tri) {
    for (int k = threadIdx.x; k < n; k += blockDim.x) body(k, a, b, c, t);
  } else {
    warp_spread(n, a, b, c, t, body);
  }
}

template <int WHAT>
static void rast_spread_launch(b200_ctx *ctx, const RastParams &p) {
  const int n = p.n_tris;
  if (n <= 0) return;
  const int per_block = n <= 8192;
  const dim3 grid(per_block ? n : (n + 255) / 256);
  rast_spread_kernel<WHAT><<<grid, 256, 0, ctx->stream>>>(p, per_block);
  ctx->stats.kernel_launches++;
  tl_mark(ctx, "rast_spread_kernel");
}

// ---- calculateIllumination (:674-688) without the final "+ indirect" -----------------------
__device__ __forceinline__ void rast_illum_D(const RastParams &p, float x, float y, float z, float nx, float ny,
                                             float nz, float *D) {
  const float rx = xsub(p.light[0], x), ry = xsub(p.light[1], y), rz = xsub(p.light[2], z);
  const double r2d = __dadd_rn(__dadd_rn(__dmul_rn((double)rx, (double)rx), __dmul_rn((double)ry, (double)ry)),
                               __dmul_rn((double)rz, (double)rz));
  const float r_mag = __double2float_rn(r2d);                                       // :677
  const float vp = xadd(xadd(xmul(rx, nx), xmul(ry, ny)), xmul(rz, nz));           // :681
  const float m = vp < 0.0f ? 0.0f : vp;                                            // glm::max
  const float den = __double2float_rn(__dmul_rn((double)4.0f * 3.14159265358979323846, (double)r_mag));  // :682
#pragma unroll
  for (int k = 0; k < 3; ++k) D[k] = xdiv(xmul(p.power[k], m), den);
}

// ---- PixelShader's colour writes for the fragment of triangle t at pixel (gx, gy), position (px, py, pz):
// screenBuffer / lowLightBuffer / highLightBuffer (:578-586; TEX: :588-645, see rast_tex.cuh) ----
template <bool TEX>
__device__ __forceinline__ void rast_shade(const RastParams &p, int t, int gx, int gy, float px, float py, float pz,
                                           float *out, int stride) {   // out[(3 * b + c) * stride]: buffer b (screen, low, high), channel c
  const float *tr = reinterpret_cast<const float *>(p.src + t);   // normal at words 12..14, colour at 16..18, texture 19, index 20
  float colour[3], normal[3];
  float occlusion = 1.0f;
  int texture = 0;
  float D[3];
  if (TEX && p.colour_mode) {
    // :647-662: randColour / nightVision * calculateIllumination, screenBuffer only; the global indirect light
    // is not reset in these modes, so every fragment sees the entry value
    const unsigned long long key = ((unsigned long long)(unsigned)t << 24) | ((unsigned long long)gy << 12) | (unsigned long long)gx;
    unsigned long long lo_i = 0, hi_i = p.colour_n;
    while (lo_i < hi_i) {
      const unsigned long long mid = (lo_i + hi_i) >> 1;
      if (__ldg(p.colour_sorted + mid) < key) lo_i = mid + 1; else hi_i = mid;
    }
    if (lo_i >= p.colour_n) lo_i = p.colour_n - 1;   // (every winner was accepted, so its key is there)
    rast_illum_D(p, px, py, pz, __ldg(tr + 12), __ldg(tr + 13), __ldg(tr + 14), D);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      out[c * stride] = xmul(__ldg(p.colour_rgb + 3 * lo_i + c), xadd(D[c], p.indirect[c]));
      out[(3 + c) * stride] = 0.f;
      out[(6 + c) * stride] = 0.f;
    }
    return;
  }
  if (TEX) {
#pragma unroll
    for (int c = 0; c < 3; ++c) { colour[c] = __ldg(tr + 16 + c); normal[c] = __ldg(tr + 12 + c); }
    texture = __float_as_int(__ldg(tr + 19));
    if (texture != 0) rast_tex_material(p.tex, texture, __float_as_int(__ldg(tr + 20)), px, py, pz, gx, gy, colour, normal, occlusion);
    rast_illum_D(p, px, py, pz, normal[0], normal[1], normal[2], D);
  } else {
    rast_illum_D(p, px, py, pz, __ldg(tr + 12), __ldg(tr + 13), __ldg(tr + 14), D);
  }
  const size_t q = (size_t)gy * p.W + gx;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float cc = TEX ? colour[c] : __ldg(tr + 16 + c);
    const float a = xadd(D[c], rast_indirect(p, c, t, q)), b = xadd(D[c], 0.0f), h = xadd(D[c], 0.4f);   // :580-584
    if (TEX && texture == 3) {   // :634-638: textureColour * (illumination * occlusion)
      out[c * stride] = xmul(cc, xmul(a, occlusion));
      out[(3 + c) * stride] = xmul(cc, xmul(b, occlusion));
      out[(6 + c) * stride] = xmul(cc, xmul(h, occlusion));
    } else {
      out[c * stride] = xmul(cc, a);
      out[(3 + c) * stride] = xmul(cc, b);
      out[(6 + c) * stride] = xmul(cc, h);
    }
  }
}

// In-place ascending sort of a tile's list in global memory when it does not fit
// in shared memory: LSD radix sort, one bit per pass (a stable split), by the
// whole block.  Only pathological scenes (> RAST_LIST_CAP triangles over one
// tile) come here.
__device__ void rast_sort_global(int *a, int *tmp, int n, int max_key, unsigned *scratch) {
  const int T = blockDim.x;
  int bits = 1;
  while ((1 << bits) <= max_key && bits < 31) ++bits;
  int *src = a, *dst = tmp;
  for (int b = 0; b < bits; ++b) {
    // count zeros
    unsigned z = 0;
    for (int i = threadIdx.x; i < n; i += T) z += ((src[i] >> b) & 1) ? 0u : 1u;
    if (threadIdx.x == 0) scratch[0] = 0;
    __syncthreads();
    atomicAdd(&scratch[0], z);
    __syncthreads();
    const unsigned n_zero = scratch[0];
    __syncthreads();
    unsigned run0 = 0, run1 = 0;   // elements placed so far in each half
    for (int base = 0; base < n; base += T) {
      const int i = base + threadIdx.x;
      const int key = i < n ? src[i] : 0;
      const unsigned one = i < n ? (unsigned)((key >> b) & 1) : 0u;
      const unsigned zero = i < n ? 1u - one : 0u;
      // block-wide exclusive scan of `zero` through shared scratch[1..T]
      scratch[1 + threadIdx.x] = zero;
      __syncthreads();
      for (int o = 1; o < T; o <<= 1) {
        const unsigned add = threadIdx.x >= o ? scratch[1 + threadIdx.x - o] : 0u;
        __syncthreads();
        scratch[1 + threadIdx.x] += add;
        __syncthreads();
      }
      const unsigned incl = scratch[1 + threadIdx.x];
      const unsigned chunk_zero = scratch[T];
      const int in_chunk = min(T, n - base);
      if (i < n) {
        if (zero) dst[run0 + incl - 1] = key;
        else dst[n_zero + run1 + (threadIdx.x - (incl))] = key;
      }
      run0 += chunk_zero;
      run1 += (unsigned)in_chunk - chunk_zero;
      __syncthreads();
    }
    int *sw = src; src = dst; dst = sw;
    __threadfence_block();
    __syncthreads();
  }
  if (src != a) {
    for (int i = threadIdx.x; i < n; i += T) a[i] = src[i];
    __syncthreads();
  }
}

// ---- per-tile fold + deferred shading -------------------------------------------------------
template <int TS_LOG2, bool TEX>
__global__ void __launch_bounds__(1 << (2 * TS_LOG2)) rast_fill_kernel(const __grid_constant__ RastParams p) {
  constexpr int TS = 1 << TS_LOG2, NT = TS * TS, NW = NT / 32;
  __shared__ int list[RAST_LIST_CAP];
  __shared__ float4 recA[RAST_BATCH][TS];
  __shared__ int recFlags[RAST_BATCH];
  // TEX: texture and index of the staged triangles (the index in full: the reference leaves one uninitialised,
  // TestModelH.h:254-257), and where their row records are (row_off - row0): a metal-grill / woven-wood fragment
  // that passes the depth test needs its position for the opacity map
  __shared__ int recTex[TEX ? RAST_BATCH : 1], recIdx[TEX ? RAST_BATCH : 1];
  __shared__ unsigned recRowBase[TEX ? RAST_BATCH : 1];
  __shared__ unsigned triRows[RAST_BATCH];   // per staged triangle: the tile rows in which its span meets the tile's columns
  __shared__ unsigned rowTris[TS];           // the transpose: per tile row, the staged triangles a pixel of that row has to look at
  __shared__ unsigned scratch[NT + 2];

  const int tile_x = blockIdx.x, tile_y = p.ty0 + blockIdx.y;
  const size_t tile = (size_t)blockIdx.y * p.tiles_x + tile_x;
  unsigned off = 0;
  int cnt = 0;
  if (!p.bits_words) {
    off = p.tile_off[tile];
    cnt = (int)min(p.tile_off[tile + 1] - off, p.bin_cap > off ? p.bin_cap - off : 0u);
  }
  const int lx_ = threadIdx.x & (TS - 1), ly_ = threadIdx.x >> TS_LOG2;
  const int x = (tile_x << TS_LOG2) + lx_, y = (tile_y << TS_LOG2) + ly_;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  // ---- the tile's triangle list in ascending order ----
  const int *sorted;
  if (p.bits_words) {
    // bit per triangle: thread i expands word i after an exclusive prefix of the word populations
    // (bits_words <= 64: two warps' worth, scanned through shared memory)
    const int nwords = p.bits_words;
    unsigned word = 0;
    if ((int)threadIdx.x < nwords) word = __ldg(p.tile_bits + tile * nwords + threadIdx.x);
    if (warp < 2) {                       // bits_words <= 64: the first two warps scan the word populations
      const int pc = __popc(word);
      int incl = pc;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
      }
      if (lane == 31) scratch[warp] = (unsigned)incl;
      // warp 1 needs warp 0's total: both publish, the block barrier below orders the reads
      scratch[2 + threadIdx.x] = (unsigned)(incl - pc);
    }
    __syncthreads();
    if (warp < 2) {
      int at = (int)scratch[2 + threadIdx.x] + (warp == 1 ? (int)scratch[0] : 0);
      for (unsigned w = word; w; w &= w - 1) list[at++] = (int)threadIdx.x * 32 + (__ffs(w) - 1);
    }
    cnt = (int)(scratch[0] + scratch[1]);
    __syncthreads();
    sorted = list;
  } else if (cnt <= RAST_LIST_CAP) {
    int m = 1;
    while (m < cnt) m <<= 1;
    for (int i = threadIdx.x; i < m; i += NT) list[i] = i < cnt ? p.bins[off + i] : INT_MAX;
    __syncthreads();
    for (int k = 2; k <= m; k <<= 1)            // bitonic sort
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int i = threadIdx.x; i < m; i += NT) {
          const int q = i ^ j;
          if (q > i) {
            const int a = list[i], b = list[q];
            const bool asc = (i & k) == 0;
            if ((a > b) == asc) { list[i] = b; list[q] = a; }
          }
        }
        __syncthreads();
      }
    sorted = list;
  } else {
    rast_sort_global(p.bins + off, p.bins_tmp + off, cnt, p.n_tris, scratch);
    sorted = p.bins + off;
  }

  // ---- fold the fragments of this pixel in triangle order ----
  float depth = 0.f;       // depthBuffer cleared to 0 (:247)
  int win = -1;
  int shadow = 0;
  unsigned n_frag = 0, n_acc = 0;
  const bool on_screen = x < p.W && y < p.H;
  for (int b0 = 0; b0 < cnt; b0 += RAST_BATCH) {
    const int nb = min(RAST_BATCH, cnt - b0);
    __syncthreads();
    // stage row records: warp w takes triangles w, w+NW, ...; lane = tile row
    for (int b = warp; b < nb; b += NW) {
      const int t = sorted[b0 + b];
      const RastSetup *s = p.setup + t;
      const int row0 = s->row0, nrows = s->nrows;
      if (lane == 0) recFlags[b] = s->flags;
      if (TEX && lane == 0) {
        recTex[b] = p.src[t].texture;
        recIdx[b] = p.src[t].index;
        recRowBase[b] = s->row_off - (unsigned)row0;
      }
      bool meets = false;
      if (lane < TS) {
        const int yy = (tile_y << TS_LOG2) + lane;
        const int r = yy - row0;
        float4 A = make_float4(__int_as_float(0), __int_as_float(0), 0.f, 0.f);
        if (r >= 0 && r < nrows) A = p.rowsA[s->row_off + r];
        recA[b][lane] = A;
        // fragments of this row are x = lx .. rx-1: any of them in the tile's columns?
        const int lx = __float_as_int(A.x), rx = __float_as_int(A.y), tx0 = tile_x << TS_LOG2;
        meets = rx > lx && rx > tx0 && lx < tx0 + TS;
      }
      const unsigned m = __ballot_sync(0xffffffffu, meets);
      if (lane == 0) triRows[b] = m;
    }
    __syncthreads();
    // The lists come from bounding boxes: most (triangle, tile row) pairs of a long thin triangle --
    // every shadow-volume side -- hold no fragment of this tile.  Transposed, each row walks only
    // the triangles that do reach it (the fold was ~1000 instructions per pixel on the Cornell box).
    if (threadIdx.x < TS) {
      unsigned mask = 0;
      for (int b = 0; b < nb; ++b) mask |= ((triRows[b] >> threadIdx.x) & 1u) << b;
      rowTris[threadIdx.x] = mask;
    }
    __syncthreads();
    if (on_screen) {
      for (unsigned mine = rowTris[ly_]; mine; mine &= mine - 1) {
        const int b = __ffs(mine) - 1;
        const float4 A = recA[b][ly_];
        const int lx = __float_as_int(A.x), rx = __float_as_int(A.y);
        // fragments x = lx .. rx-1 (right end excluded, :504); (:573) bounds hold by construction
        if (x >= lx && x < rx) {
          ++n_frag;
          const float zinv = xadd(A.z, xmul(A.w, (float)(x - lx)));   // :543
          if (recFlags[b] & 1) {
            if (zinv > depth) shadow = 1;                            // :668-670
          } else if (zinv >= depth) {                                // :574
            bool hole = false;
            if (TEX) {
              const int texture = p.colour_mode ? 0 : recTex[b];   // the colour modes never look at it (:575)
              if (texture == 2 || texture == 3) {                    // :603, :625: the opacity map decides
                const float4 B = __ldg(p.rowsB + (recRowBase[b] + (unsigned)y));
                const float fi = (float)(x - lx);
                const float pz = xdiv(1.0f, zinv);                              // :546
                const float px = xdiv(xadd(B.x, xmul(B.y, fi)), zinv);          // :547
                const float py = xdiv(xadd(B.z, xmul(B.w, fi)), zinv);          // :548
                hole = rast_tex_hole(p.tex, texture, recIdx[b], px, py, pz);
              }
            }
            if (hole) {
              depth = 0.f;                                           // :619 / :643, then :665; the colours stay
            } else {
              depth = zinv;                                          // :665
              win = sorted[b0 + b];
            }
            if (TEX && p.colour_mode && y >= p.fb0 && y < p.fb1) {
              ++n_acc;
              if (p.colour_emit) {
                const unsigned m = __activemask();
                const int leader = __ffs(m) - 1;
                unsigned long long base = 0;
                if (lane == leader) base = atomicAdd(p.counters + 18, (unsigned long long)__popc(m));
                base = __shfl_sync(m, base, leader);
                const unsigned long long at = base + __popc(m & ((1u << lane) - 1));
                if (at < p.colour_n)
                  p.colour_emit[at] = ((unsigned long long)(unsigned)win << 24) | ((unsigned long long)y << 12) | (unsigned long long)x;
              }
            }
          }
        }
      }
    }
  }

  if (TEX && p.colour_emit) return;   // emit pass of a colour-mode frame: the keys are out, the winners are already stored
  if (TEX && p.colour_mode) {
    unsigned long long na = n_acc;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) na += __shfl_xor_sync(0xffffffffu, na, o);
    if (lane == 0 && na) atomicAdd(p.counters + 17, na);   // (colour-mode frames are always fused: shading needs the ordinals)
  }

  // ---- deferred PixelShader of the winning fragment (:575-586) ----
  if (on_screen && y >= p.fb0 && y < p.fb1 && p.fused) {
    const size_t q = (size_t)y * p.W + x;
    p.keys[q] = ((unsigned long long)__float_as_uint(depth) << 32) | (unsigned)(win + 1);
    p.shadow8[q] = (unsigned char)shadow;
  } else if (on_screen && y >= p.fb0 && y < p.fb1) {
    const size_t q = (size_t)y * p.W + x;
    float sc[3] = {0.f, 0.f, 0.f}, lo[3] = {0.f, 0.f, 0.f}, hi[3] = {0.f, 0.f, 0.f};
    if (win >= 0) {
      const RastSetup *s = p.setup + win;
      const unsigned r = s->row_off + (unsigned)(y - s->row0);
      const float4 A = p.rowsA[r], B = p.rowsB[r];
      const float fi = (float)(x - __float_as_int(A.x));
      const float zinv = xadd(A.z, xmul(A.w, fi));
      const float pz = xdiv(1.0f, zinv);                              // :546
      const float px = xdiv(xadd(B.x, xmul(B.y, fi)), zinv);          // :547
      const float py = xdiv(xadd(B.z, xmul(B.w, fi)), zinv);          // :548
      float o[9];
      rast_shade<TEX>(p, win, x, y, px, py, pz, o, 1);
#pragma unroll
      for (int k = 0; k < 3; ++k) { sc[k] = o[k]; lo[k] = o[3 + k]; hi[k] = o[6 + k]; }
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) { p.screen[3 * q + k] = sc[k]; p.low[3 * q + k] = lo[k]; p.high[3 * q + k] = hi[k]; }
    p.depth[q] = depth;
    p.shadow[q] = shadow;
    p.index[q] = win;
  }
  unsigned long long nf = (on_screen && y >= p.fb0 && y < p.fb1) ? n_frag : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) nf += __shfl_xor_sync(0xffffffffu, nf, o);
  if (lane == 0 && nf) atomicAdd(p.counters + 16, nf);
}

// ---- post pass (:283-307) --------------------------------------------------------------------
// The reference darkens screenBuffer in place while scanning row-major, so the
// 5-tap cross at (y,x) sees darkened (y,x), (y-1,x), (y,x-1) and original
// (y+1,x), (y,x+1).  The amount depends only on the final shadow mask, so every
// pixel can be evaluated independently.
__device__ __forceinline__ float rast_sub(const RastParams &p, int y, int x) {
  if (y < 1 || y > p.H - 2 || x < 1 || x > p.W - 2) return 0.f;   // never visited by the loop
  const int *s = p.shadow;
  const size_t W = p.W;
  if (s[y * W + x] != 1) return 0.f;
  // surroundingShadowSum (:1725-1733): [y+1][x-1] counted twice, [y+1][x+1] never
  const int sum = s[y * W + x] + s[(y - 1) * W + x] + s[(y - 1) * W + x - 1] + s[(y - 1) * W + x + 1] +
                  s[(y + 1) * W + x - 1] + s[(y + 1) * W + x] + s[(y + 1) * W + x - 1] + s[y * W + x - 1] +
                  s[y * W + x + 1];
  const float f = xdiv((float)sum, 9.0f);
  const double d = (double)f;
  return d < 0.6 ? 0.05f : d < 0.7 ? 0.08f : d < 0.8 ? 0.1f : d < 0.9 ? 0.12f : 0.3f;
}

__global__ void rast_post_kernel(const __grid_constant__ RastParams p) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = p.row0 + blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= p.W || y >= p.row1) return;
  const size_t W = p.W, q = (size_t)y * W + x;
  float out[3] = {0.f, 0.f, 0.f};
  const bool interior = y >= 1 && y <= p.H - 2 && x >= 1 && x <= p.W - 2;
  if (interior) {
    const float s0 = rast_sub(p, y, x), s1 = rast_sub(p, y - 1, x), s2 = rast_sub(p, y, x - 1);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float *S = p.screen + k, *L = p.low + k, *Hh = p.high + k;
      // the reference only subtracts when the flag is set; x - 0 == x keeps that exact
      const float c0 = s0 != 0.f ? xsub(S[3 * q], s0) : S[3 * q];
      const float c1 = s1 != 0.f ? xsub(S[3 * (q - W)], s1) : S[3 * (q - W)];
      const float c2 = s2 != 0.f ? xsub(S[3 * (q - 1)], s2) : S[3 * (q - 1)];
      float a = xadd(c0, c1);
      a = xadd(a, S[3 * (q + W)]);
      a = xadd(a, c2);
      a = xadd(a, S[3 * (q + 1)]);
      a = xdiv_const<5>(a);
      float b = xadd(L[3 * q], L[3 * (q - W)]);
      b = xadd(b, L[3 * (q + W)]);
      b = xadd(b, L[3 * (q - 1)]);
      b = xadd(b, L[3 * (q + 1)]);
      b = xdiv_const<5>(b);
      float c = xadd(Hh[3 * q], Hh[3 * (q - W)]);
      c = xadd(c, Hh[3 * (q + W)]);
      c = xadd(c, Hh[3 * (q - 1)]);
      c = xadd(c, Hh[3 * (q + 1)]);
      c = xdiv_const<5>(c);
      out[k] = xdiv_const<3>(xadd(xadd(a, b), c));   // :1750
    }
  }
  if (p.out_rgb) { p.out_rgb[3 * q] = out[0]; p.out_rgb[3 * q + 1] = out[1]; p.out_rgb[3 * q + 2] = out[2]; }
  if (p.out_argb) p.out_argb[q] = interior ? put_pixel_argb(out[0], out[1], out[2]) : 0u;   // border: memset 0 (:244)
  if (p.out_depth) p.out_depth[q] = p.depth[q];
  if (p.out_index) p.out_index[q] = p.index[q];
}

#include "rast_fast.cuh"

// ---- host side ---------------------------------------------------------------------------------
// glm::inverse(R) as findU / findV compute it per fragment (glm 0.9.7.2 detail/type_mat4x4.inl:37-92; separately
// rounded products and differences: the reference build has no FMA), and the reference's `yaw != 0` (:1761):
// R is the identity exactly when yaw is 0 (:387-396).
static void rast_tex_view(const float *m_, float *out, int *use_rinv) {
  auto M = [&](int c, int r) -> float { return m_[4 * c + r]; };
  auto sub2 = [](float a, float b, float c, float d) -> float {   // a * b - c * d, three roundings
    volatile float x = a * b, y = c * d;
    return x - y;
  };
  const float Coef00 = sub2(M(2, 2), M(3, 3), M(3, 2), M(2, 3)), Coef02 = sub2(M(1, 2), M(3, 3), M(3, 2), M(1, 3)),
              Coef03 = sub2(M(1, 2), M(2, 3), M(2, 2), M(1, 3)), Coef04 = sub2(M(2, 1), M(3, 3), M(3, 1), M(2, 3)),
              Coef06 = sub2(M(1, 1), M(3, 3), M(3, 1), M(1, 3)), Coef07 = sub2(M(1, 1), M(2, 3), M(2, 1), M(1, 3)),
              Coef08 = sub2(M(2, 1), M(3, 2), M(3, 1), M(2, 2)), Coef10 = sub2(M(1, 1), M(3, 2), M(3, 1), M(1, 2)),
              Coef11 = sub2(M(1, 1), M(2, 2), M(2, 1), M(1, 2)), Coef12 = sub2(M(2, 0), M(3, 3), M(3, 0), M(2, 3)),
              Coef14 = sub2(M(1, 0), M(3, 3), M(3, 0), M(1, 3)), Coef15 = sub2(M(1, 0), M(2, 3), M(2, 0), M(1, 3)),
              Coef16 = sub2(M(2, 0), M(3, 2), M(3, 0), M(2, 2)), Coef18 = sub2(M(1, 0), M(3, 2), M(3, 0), M(1, 2)),
              Coef19 = sub2(M(1, 0), M(2, 2), M(2, 0), M(1, 2)), Coef20 = sub2(M(2, 0), M(3, 1), M(3, 0), M(2, 1)),
              Coef22 = sub2(M(1, 0), M(3, 1), M(3, 0), M(1, 1)), Coef23 = sub2(M(1, 0), M(2, 1), M(2, 0), M(1, 1));
  const float Fac0[4] = {Coef00, Coef00, Coef02, Coef03}, Fac1[4] = {Coef04, Coef04, Coef06, Coef07},
              Fac2[4] = {Coef08, Coef08, Coef10, Coef11}, Fac3[4] = {Coef12, Coef12, Coef14, Coef15},
              Fac4[4] = {Coef16, Coef16, Coef18, Coef19}, Fac5[4] = {Coef20, Coef20, Coef22, Coef23};
  const float Vec0[4] = {M(1, 0), M(0, 0), M(0, 0), M(0, 0)}, Vec1[4] = {M(1, 1), M(0, 1), M(0, 1), M(0, 1)},
              Vec2[4] = {M(1, 2), M(0, 2), M(0, 2), M(0, 2)}, Vec3[4] = {M(1, 3), M(0, 3), M(0, 3), M(0, 3)};
  const float SignA[4] = {+1, -1, +1, -1}, SignB[4] = {-1, +1, -1, +1};
  auto inv3 = [&](const float *a, const float *fa, const float *b, const float *fb, const float *c, const float *fc, int k) -> float {
    volatile float t = sub2(a[k], fa[k], b[k], fb[k]), u = c[k] * fc[k];   // (a * fa - b * fb) + c * fc
    return t + u;
  };
  float Inv[16];
  for (int k = 0; k < 4; ++k) {
    Inv[0 + k] = inv3(Vec1, Fac0, Vec2, Fac1, Vec3, Fac2, k) * SignA[k];
    Inv[4 + k] = inv3(Vec0, Fac0, Vec2, Fac3, Vec3, Fac4, k) * SignB[k];
    Inv[8 + k] = inv3(Vec0, Fac1, Vec1, Fac3, Vec3, Fac5, k) * SignA[k];
    Inv[12 + k] = inv3(Vec0, Fac2, Vec1, Fac4, Vec2, Fac5, k) * SignB[k];
  }
  volatile float d0 = M(0, 0) * Inv[0], d1 = M(0, 1) * Inv[4], d2 = M(0, 2) * Inv[8], d3 = M(0, 3) * Inv[12];
  volatile float s01 = d0 + d1, s23 = d2 + d3;
  const float det = s01 + s23;
  const float one_over = 1.0f / det;
  for (int k = 0; k < 16; ++k) out[k] = Inv[k] * one_over;
  *use_rinv = 0;
  for (int c = 0; c < 4; ++c)
    for (int r = 0; r < 4; ++r)
      if (m_[4 * c + r] != (c == r ? 1.0f : 0.0f)) *use_rinv = 1;
}

// host logic, callable without a device (CPU tests compare it with the oracle's restatement)
extern "C" int b200_debug_rast_inverse(const float *R16, float *out16, int *use_rinv) {
  if (!R16 || !out16 || !use_rinv) return B200_EINVAL;
  rast_tex_view(R16, out16, use_rinv);
  return B200_OK;
}

// The back end of a frame of n triangles: scatter / resolve (rast_fast.cuh) or ordered screen tiles.  rast_frame
// asks before the geometry stage (n: the list bound a pipelined geometry stage writes under) and acts on the answer
// there; rast_launch asks again for the list it is given.
bool rast_scatter_path(const b200_ctx *ctx, long long n) {
  return ctx->opt_rast_path == 2 || (ctx->opt_rast_path == 0 && !ctx->rast_has_shadow && !ctx->rast_tex_on &&
                                     !ctx->opt_rast_colour && n < RAST_FAST_MAX_TRIS);
}

// rast_fill_kernel at the frame's tile size (TEX: the variant that knows about textures / colour modes)
template <bool TEX>
static int rast_fill_launch(b200_ctx *ctx, const RastParams &p, const char *name) {
  const dim3 grid(p.tiles_x, p.tiles_y);
  switch (p.ts_log2) {
    case 3: rast_fill_kernel<3, TEX><<<grid, 64, 0, ctx->stream>>>(p); break;
    case 4: rast_fill_kernel<4, TEX><<<grid, 256, 0, ctx->stream>>>(p); break;
    default: rast_fill_kernel<5, TEX><<<grid, 1024, 0, ctx->stream>>>(p); break;
  }
  ctx->stats.kernel_launches++;
  tl_mark(ctx, name);
  CU_CHECK(ctx, cudaGetLastError());
  return B200_OK;
}

// ---- scatter / resolve (rast_fast.cuh); p: the frame as rast_launch set it up ----
static int rast_launch_scatter(b200_ctx *ctx, RastParams &p, bool spec) {
  const int W = p.W, n = p.n_tris, row0 = p.row0, row1 = p.row1;
  const size_t npix = (size_t)W * p.H;
  ctx->rast_w = 0; ctx->rast_h = 0;   // no intermediate buffers in this path
  if (int rc = ensure(ctx, ctx->rast_keys, npix * sizeof(unsigned long long))) return rc;
  p.keys = (unsigned long long *)ctx->rast_keys.p;
  if (int rc = ensure(ctx, ctx->rast_trimeta, sizeof(int2) * (size_t)(n ? n : 1))) return rc;
  p.trimeta = (int2 *)ctx->rast_trimeta.p;
  p.orig = ctx->rast_culled ? (const int *)ctx->rast_orig.p : nullptr;
  // small triangles: S2_ROWS record places each, addressed by the key (only the rows drawn are touched)
  if (int rc = ensure(ctx, ctx->rast_srowsB, sizeof(float4) * S2_ROWS * (size_t)(n ? n : 1))) return rc;
  if (int rc = ensure(ctx, ctx->rast_srowsL, sizeof(int) * S2_ROWS * (size_t)(n ? n : 1))) return rc;
  p.srowsB = (float4 *)ctx->rast_srowsB.p;
  p.srowsL = (int *)ctx->rast_srowsL.p;
  const int s2_blocks = (n + S2_THREADS - 1) / S2_THREADS;
  size_t n_rows = 0, big_cap = 0;   // rows of the big triangles, entries of the big list
  if (spec) {
    // sizes guessed from the last verified frame; the kernels flag any overflow.  A frame whose
    // predecessor had no big triangle does not launch the big-triangle kernels at all.
    n_rows = (size_t)rast_spec_cap(ctx->rast_spec.rows);
    big_cap = ctx->rast_spec.big ? (size_t)rast_spec_cap(ctx->rast_spec.big) : 0;
  } else if (n > 0) {
    // exact sizes from a counting pass: [10] big triangles, [11] their rows
    unsigned long long *hc = (unsigned long long *)ctx->pinned;
    rast_scatter2_kernel<true><<<s2_blocks, S2_THREADS, 0, ctx->stream>>>(p);
    ctx->stats.kernel_launches++;
    tl_mark(ctx, "rast_scatter2_kernel<count>");
    CU_CHECK(ctx, cudaGetLastError());
    CU_CHECK(ctx, cudaMemcpyAsync(hc, ctx->counters.p, 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CU_CHECK(ctx, cudaMemsetAsync(p.counters + 10, 0, 2 * sizeof(unsigned long long), ctx->stream));
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    if (hc[11] > 0xfffffff0ull) return ctx_fail(ctx, B200_ENOMEM, "row table budget exceeded");
    n_rows = (size_t)hc[11];
    big_cap = (size_t)hc[10];
  }
  p.n_rows = (unsigned)(n_rows > 0xffffffffull ? 0xffffffffull : n_rows);
  if (n_rows < 1) n_rows = 1;
  if (big_cap > 0x7fffffffull) big_cap = 0x7fffffffull;
  if (int rc = ensure(ctx, ctx->rast_rowsA, sizeof(int) * n_rows)) return rc;
  if (int rc = ensure(ctx, ctx->rast_rowsB, sizeof(float4) * n_rows)) return rc;
  if (int rc = ensure(ctx, ctx->rast_setup, sizeof(RastSetup) * (big_cap ? big_cap : 1))) return rc;
  if (int rc = ensure(ctx, ctx->rast_big, sizeof(int) * (big_cap ? big_cap : 1))) return rc;
  if (int rc = ensure(ctx, ctx->rast_row_owner, sizeof(int) * n_rows)) return rc;
  p.rowsL = (int *)ctx->rast_rowsA.p;
  p.rowsB = (float4 *)ctx->rast_rowsB.p;
  p.row_cap = (unsigned)(n_rows > 0xffffffffull ? 0xffffffffull : n_rows);
  p.setup = (RastSetup *)ctx->rast_setup.p;
  p.big_list = (int *)ctx->rast_big.p;
  p.big_cap = (unsigned)big_cap;
  p.row_owner = (int *)ctx->rast_row_owner.p;
  // cleared right before the scatter so that the 64-bit keys (66 MB at 4K, less than the L2)
  // are still cache-resident when the atomics arrive
  if (!ctx->rast_keys_cleared) {   // (a pipelined whole-Draw frame: already done by its geometry kernel)
    CU_CHECK(ctx, cudaMemsetAsync(p.keys + (size_t)p.fb0 * W, 0, (size_t)(p.fb1 - p.fb0) * W * sizeof(unsigned long long), ctx->stream));
    tl_mark(ctx, "memset keys");
  }
  ctx->rast_keys_cleared = 0;
  if (n > 0) {
    if (spec && ctx->rast_geom_chunks > 1) {
      // chunk k of the list is scattered on the second stream as soon as the geometry kernel's
      // k-th launch is done, while chunk k + 1 of the scene is still on the link; the frame goes on
      // when all are in
      for (int c = 0; c < ctx->rast_geom_chunks; ++c) {
        RastParams pc = p;
        pc.range_lo = c ? p.counters + 12 + (c - 1) : nullptr;
        pc.range_hi = p.counters + 12 + c;
        const int bound = ctx->rast_geom_chunk_tris[c] + ctx->rast_geom_chunk_tris[c] / 32 + 1024;   // + 3 %: clipping can add triangles
        CU_CHECK(ctx, cudaStreamWaitEvent(ctx->aux_stream, ctx->ev_chunk[c], 0));
        rast_scatter2_kernel<false><<<(bound + S2_THREADS - 1) / S2_THREADS, S2_THREADS, 0, ctx->aux_stream>>>(pc);
        ctx->stats.kernel_launches++;
      }
      CU_CHECK(ctx, cudaEventRecord(ctx->ev_join, ctx->aux_stream));
      CU_CHECK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
    } else {
      rast_scatter2_kernel<false><<<s2_blocks, S2_THREADS, 0, ctx->stream>>>(p);
      ctx->stats.kernel_launches++;
    }
    tl_mark(ctx, "rast_scatter2_kernel");
    if (big_cap > 0) {
      rast_setup_big_kernel<<<(int)((big_cap + 127) / 128), 128, 0, ctx->stream>>>(p);
      ctx->stats.kernel_launches++;
      tl_mark(ctx, "rast_setup_big_kernel");
      if (p.n_rows > 0) {
        rast_scatter_kernel<<<(int)(((size_t)p.n_rows + 255) / 256), 256, 0, ctx->stream>>>(p);
        ctx->stats.kernel_launches++;
        tl_mark(ctx, "rast_scatter_kernel");
      }
    }
    CU_CHECK(ctx, cudaGetLastError());
  }
  // host-pointer entries: resolve in slices, each slice's packed rows leave for the host
  // while the next one is resolved (band_slice_done is a no-op otherwise)
  const int k = (ctx->slice_host && (size_t)(row1 - row0) * W >= B200_SLICE_MIN_PIXELS) ? B200_SLICES : 1;
  for (int i = 0; i < k; ++i) {
    p.row0 = band_slice_edge(row0, row1 - row0, i, k, RS_H);
    p.row1 = band_slice_edge(row0, row1 - row0, i + 1, k, RS_H);
    if (p.row1 <= p.row0) continue;
    dim3 rg((W + RS_W - 1) / RS_W, (p.row1 - p.row0 + RS_H - 1) / RS_H);
    rast_resolve_kernel<false, false><<<rg, RS_W * RS_H, 0, ctx->stream>>>(p);
    ctx->stats.kernel_launches++;
    tl_mark(ctx, "rast_resolve_kernel");
    CU_CHECK(ctx, cudaGetLastError());
    if (int rc = band_slice_done(ctx, p.row0, p.row1)) return rc;
  }
  return B200_OK;
}

// ---- ordered screen tiles; p: the frame as rast_launch set it up ----
static int rast_launch_ordered(b200_ctx *ctx, RastParams &p, bool spec) {
  const int W = p.W, H = p.H, n = p.n_tris, row0 = p.row0, row1 = p.row1, colour = p.colour_mode;
  const int n_tiles = p.tiles_x * p.tiles_y;
  const size_t npix = (size_t)W * H;
  const bool texk = p.tex_on || colour;           // the kernel variants that know about textures / colour modes
  const bool bits = n <= RAST_BITS_MAX_TRIS;      // short list: bit-per-triangle tile lists
  unsigned long long *hc = (unsigned long long *)ctx->pinned;
  p.spread_in_setup = n > 8192 ? 1 : 0;   // short lists of big triangles: one block per triangle spreads better
  if (int rc = ensure(ctx, ctx->rast_setup, sizeof(RastSetup) * (size_t)(n ? n : 1))) return rc;
  p.setup = (RastSetup *)ctx->rast_setup.p;
  // row slots: a short list (rast_short_kernel) gives every triangle a band's worth; a long one claims what its
  // triangles reach, at worst the whole band each (pipelined: what the last verified frame claimed, + 3 %)
  size_t row_cap = spec && !bits ? (size_t)rast_spec_cap(ctx->rast_spec.rows) : (size_t)(n ? n : 1) * (size_t)(p.fb1 - p.fb0);
  const size_t row_budget = (size_t)64 << 20;   // 64 Mi rows = 2 GiB of row records
  if (row_cap > row_budget) row_cap = row_budget;
  if (int rc = ensure(ctx, ctx->rast_row_owner, sizeof(int) * row_cap)) return rc;
  p.row_owner = (int *)ctx->rast_row_owner.p;
  if (int rc = ensure(ctx, ctx->rast_rowsA, sizeof(float4) * row_cap)) return rc;
  if (int rc = ensure(ctx, ctx->rast_rowsB, sizeof(float4) * row_cap)) return rc;
  if (int rc = ensure(ctx, ctx->rast_tile_count, sizeof(unsigned) * (size_t)(n_tiles + 1) * 3)) return rc;
  // Automatic strategy: fused -- the fold leaves 9 bytes per pixel and the resolve kernel does the
  // rest.  B200_OPT_RAST_PATH = 1 keeps the reference's six intermediate buffers (raster_read_buffers).
  const bool fused = ctx->opt_rast_path == 0 || colour;
  p.fused = fused ? 1 : 0;
  if (fused) {
    if (int rc = ensure(ctx, ctx->rast_keys, npix * sizeof(unsigned long long))) return rc;
    if (int rc = ensure(ctx, ctx->rast_shadow8, npix)) return rc;
    p.keys = (unsigned long long *)ctx->rast_keys.p;
    p.shadow8 = (unsigned char *)ctx->rast_shadow8.p;
    ctx->rast_w = 0; ctx->rast_h = 0;
  } else {
    if (int rc = ensure(ctx, ctx->rast_screen, npix * 3 * sizeof(float))) return rc;
    if (int rc = ensure(ctx, ctx->rast_low, npix * 3 * sizeof(float))) return rc;
    if (int rc = ensure(ctx, ctx->rast_high, npix * 3 * sizeof(float))) return rc;
    if (int rc = ensure(ctx, ctx->rast_shadow, npix * sizeof(int))) return rc;
    if (int rc = ensure(ctx, ctx->rast_depth, npix * sizeof(float))) return rc;
    if (int rc = ensure(ctx, ctx->rast_index, npix * sizeof(int))) return rc;
    ctx->rast_w = W; ctx->rast_h = H;
  }
  p.rowsA = (float4 *)ctx->rast_rowsA.p;
  p.rowsB = (float4 *)ctx->rast_rowsB.p;
  p.row_cap = (unsigned)(row_cap > 0xffffffffull ? 0xffffffffull : row_cap);
  p.n_rows = p.row_cap;   // a launch bound until the rows claimed are read back (pipelined: clamped on the device)
  p.tile_count = (unsigned *)ctx->rast_tile_count.p;
  p.tile_off = p.tile_count + (n_tiles + 1);
  p.tile_cursor = p.tile_off + (n_tiles + 1);
  p.depth = (float *)ctx->rast_depth.p;
  p.screen = (float *)ctx->rast_screen.p;
  p.low = (float *)ctx->rast_low.p;
  p.high = (float *)ctx->rast_high.p;
  p.shadow = (int *)ctx->rast_shadow.p;
  p.index = (int *)ctx->rast_index.p;

  if (bits) {
    p.bits_words = (n + 31) / 32 > 0 ? (n + 31) / 32 : 1;
    if (int rc = ensure(ctx, ctx->rast_tile_bits, sizeof(unsigned) * (size_t)n_tiles * p.bits_words)) return rc;
    p.tile_bits = (unsigned *)ctx->rast_tile_bits.p;
    CU_CHECK(ctx, cudaMemsetAsync(p.tile_bits, 0, sizeof(unsigned) * (size_t)n_tiles * p.bits_words, ctx->stream));
  } else {
    CU_CHECK(ctx, cudaMemsetAsync(p.tile_count, 0, sizeof(unsigned) * (size_t)(n_tiles + 1), ctx->stream));
  }
  if (n > 0 && bits) {
    // setup, row records and tile bits of a short list
    rast_short_kernel<<<n, SHORT_THREADS, 0, ctx->stream>>>(p);
    ctx->stats.kernel_launches++;
    tl_mark(ctx, "rast_short_kernel");
  } else if (n > 0) {
    rast_setup_kernel<<<(n + SETUP_THREADS - 1) / SETUP_THREADS, SETUP_THREADS, 0, ctx->stream>>>(p);
    ctx->stats.kernel_launches++;
    tl_mark(ctx, "rast_setup_kernel");
    if (!p.spread_in_setup) rast_spread_launch<0>(ctx, p);
    rast_spread_launch<1>(ctx, p);
  }
  if (!bits) {
    rast_scan_kernel<<<1, 1024, 0, ctx->stream>>>(p, n_tiles);
    ctx->stats.kernel_launches++;
    tl_mark(ctx, "rast_scan_kernel");
  }
  CU_CHECK(ctx, cudaGetLastError());
  size_t bin_cap = 0;
  if (spec) {
    // sizes guessed from the last verified frame; the setup / scan kernels flag any overflow
    bin_cap = (size_t)rast_spec_cap(ctx->rast_spec.bins);
    ctx->rast_inflight.cap_bins = bin_cap;
  } else {
    // the bin array is sized from the scanned total: read it back (tiny, one sync)
    CU_CHECK(ctx, cudaMemcpyAsync(hc, ctx->counters.p, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    if (hc[5]) return ctx_fail(ctx, B200_ENOMEM, "row table budget exceeded (triangles too tall for this band)");
    bin_cap = (size_t)hc[3];
    p.n_rows = (unsigned)hc[4];
  }
  if (int rc = ensure(ctx, ctx->rast_bins, sizeof(int) * (bin_cap ? bin_cap : 1))) return rc;
  if (int rc = ensure(ctx, ctx->rast_tmp, sizeof(int) * (bin_cap ? bin_cap : 1))) return rc;
  p.bins = (int *)ctx->rast_bins.p;
  p.bins_tmp = (int *)ctx->rast_tmp.p;
  p.bin_cap = (unsigned)(bin_cap > 0xffffffffull ? 0xffffffffull : bin_cap);
  if (p.n_rows > 0 && n > 0 && !bits) {
    rast_rows_kernel<<<(int)(((size_t)p.n_rows + 255) / 256), 256, 0, ctx->stream>>>(p);
    ctx->stats.kernel_launches++;
    tl_mark(ctx, "rast_rows_kernel");
  }
  if (n > 0 && bin_cap > 0 && !bits) rast_spread_launch<2>(ctx, p);
  if (int rc = texk ? rast_fill_launch<true>(ctx, p, "rast_fill_kernel") : rast_fill_launch<false>(ctx, p, "rast_fill_kernel"))
    return rc;
  if (colour) {
    // the accepted fragments in the reference's serial order: count, emit, sort; then the host draws
    // three rand() values per fragment, exactly as PixelShader would have (:649-651, :657-659)
    CU_CHECK(ctx, cudaMemcpyAsync(hc, ctx->counters.p, 24 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
    const unsigned long long n_acc = hc[17];
    if (n_acc > 0x3fffffffull) return ctx_fail(ctx, B200_ENOMEM, "colour modes 1 / 2: too many accepted fragments");
    const size_t na = (size_t)(n_acc ? n_acc : 1);
    if (int rc = ensure(ctx, ctx->rast_colour_keys, 2 * na * sizeof(unsigned long long))) return rc;
    if (int rc = ensure(ctx, ctx->rast_colour_rgb, 3 * na * sizeof(float))) return rc;
    unsigned long long *keys_a = (unsigned long long *)ctx->rast_colour_keys.p, *keys_b = keys_a + na;
    if (n_acc) {
      RastParams pe = p;
      pe.colour_emit = keys_a;
      pe.colour_n = n_acc;
      if (int rc = rast_fill_launch<true>(ctx, pe, "rast_fill_kernel<emit>")) return rc;
      int tri_bits = 1;
      while (tri_bits < 31 && (1ll << tri_bits) < (long long)n) ++tri_bits;
      if (int rc = rast_colour_sort(ctx, keys_a, keys_b, n_acc, 24 + tri_bits)) return rc;
      std::vector<float> rgb(3 * (size_t)n_acc);
      for (size_t i = 0; i < (size_t)n_acc; ++i) {
        float LO = 0.2f;
        float HI = 0.5f;
        float r0 = LO + static_cast<float>(rand()) / (static_cast<float>(RAND_MAX / HI - LO));   // :649-651
        float r1 = LO + static_cast<float>(rand()) / (static_cast<float>(RAND_MAX / HI - LO));
        float r2 = LO + static_cast<float>(rand()) / (static_cast<float>(RAND_MAX / HI - LO));
        if (colour == 1) { rgb[3 * i] = r0; rgb[3 * i + 1] = r1; rgb[3 * i + 2] = r2; }           // :652
        else { rgb[3 * i] = r0 - 0.2f; rgb[3 * i + 1] = 1.0f; rgb[3 * i + 2] = r2 - 0.2f; }       // :660
      }
      CU_CHECK(ctx, cudaMemcpyAsync(ctx->rast_colour_rgb.p, rgb.data(), rgb.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
      CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));   // `rgb` leaves scope
    }
    p.colour_sorted = keys_b;
    p.colour_n = n_acc;
    p.colour_rgb = (const float *)ctx->rast_colour_rgb.p;
  }
  const int k = (ctx->slice_host && (size_t)(row1 - row0) * W >= B200_SLICE_MIN_PIXELS) ? B200_SLICES : 1;
  for (int i = 0; i < k; ++i) {
    p.row0 = band_slice_edge(row0, row1 - row0, i, k, fused ? RS_H : 8);
    p.row1 = band_slice_edge(row0, row1 - row0, i + 1, k, fused ? RS_H : 8);
    if (p.row1 <= p.row0) continue;
    dim3 pb(32, 8), pg((W + 31) / 32, (p.row1 - p.row0 + 7) / 8);
    const dim3 rg((W + RS_W - 1) / RS_W, (p.row1 - p.row0 + RS_H - 1) / RS_H);
    if (fused && texk) rast_resolve_kernel<true, true><<<rg, RS_W * RS_H, 0, ctx->stream>>>(p);
    else if (fused) rast_resolve_kernel<true, false><<<rg, RS_W * RS_H, 0, ctx->stream>>>(p);
    else rast_post_kernel<<<pg, pb, 0, ctx->stream>>>(p);
    ctx->stats.kernel_launches++;
    tl_mark(ctx, fused ? "rast_resolve_kernel<ordered>" : "rast_post_kernel");
    CU_CHECK(ctx, cudaGetLastError());
    if (int rc = band_slice_done(ctx, p.row0, p.row1)) return rc;
  }
  return B200_OK;
}

int rast_launch(b200_ctx *ctx, const camera_t *cam, const rast_light_t *light, int row0, int row1,
                float *d_rgb, float *d_depth, int32_t *d_index, uint32_t *d_argb, bool spec) {
  // n is the list length, or in a pipelined whole-Draw frame the bound the geometry stage wrote under
  const int W = cam->width, H = cam->height, n = ctx->rast_n_tris;
  const int colour = ctx->opt_rast_colour;
  if (ctx->opt_rast_path == 2 && ctx->rast_has_shadow)
    return ctx_fail(ctx, B200_EINVAL, "the scatter path cannot draw shadow-volume triangles");
  if (ctx->opt_rast_path == 2 && n >= RAST_FAST_MAX_TRIS) return ctx_fail(ctx, B200_EINVAL, "too many triangles for the scatter path");
  if (ctx->opt_rast_path == 2 && (ctx->rast_tex_on || colour))
    return ctx_fail(ctx, B200_EINVAL, "the scatter path cannot draw textures or colour modes (both depend on the order of the fragments)");
  if (colour && (row0 != 0 || row1 != H)) return ctx_fail(ctx, B200_EINVAL, "colour modes 1 / 2 number the fragments of the whole frame: no row bands");
  if (colour && (W > 4096 || H > 4096)) return ctx_fail(ctx, B200_EINVAL, "colour modes 1 / 2: frames up to 4096 x 4096");

  RastParams p;
  memset(&p, 0, sizeof p);
  p.W = W; p.H = H;
  p.row0 = row0; p.row1 = row1;
  p.fb0 = row0 - 2 > 0 ? row0 - 2 : 0;
  p.fb1 = row1 + 2 < H ? row1 + 2 : H;
  p.ts_log2 = ctx->opt_rast_tile_log2;
  const int ts = p.ts_log2, TS = 1 << ts;
  p.tiles_x = (W + TS - 1) >> ts;
  p.ty0 = p.fb0 >> ts;
  p.tiles_y = ((p.fb1 - 1) >> ts) - p.ty0 + 1;
  p.focal = cam->focal;
  memcpy(p.light, light->pos, sizeof p.light);
  memcpy(p.power, light->power, sizeof p.power);
  memcpy(p.indirect, light->indirect, sizeof p.indirect);
  p.src = (const rast_triangle *)ctx->rast_src.p;
  p.n_tris = n;
  p.tex_on = ctx->rast_tex_on && !colour;   // the colour modes never look at the texture fields (:575)
  p.colour_mode = colour;
  if (p.tex_on) {
    p.tex = ctx->rast_tex;
    memcpy(p.tex.cam, cam->pos, sizeof p.tex.cam);
    rast_tex_view(cam->R, p.tex.Rinv, &p.tex.use_rinv);
  }
  p.out_rgb = d_rgb; p.out_depth = d_depth; p.out_index = d_index; p.out_argb = d_argb;
  p.counters = (unsigned long long *)ctx->counters.p;
  if (spec) {   // the list length (whole-Draw frames) and the rows claimed are known on the device only
    p.n_tris_dev = ctx->rast_inflight.whole_draw ? p.counters + 24 : nullptr;
    p.n_rows_dev = p.counters + 4;
  }

  // the entry value of indirectLightPowerPerArea reaches the first shaded fragment only (:585)
  if (n > 0 && !colour && rast_indirect_entry_differs(light)) {
    unsigned long long *first = p.counters + 9;
    CU_CHECK(ctx, cudaMemsetAsync(first, 0xff, sizeof(unsigned long long), ctx->stream));
    rast_first_fragment_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(p, first);
    ctx->stats.kernel_launches++;
    tl_mark(ctx, "rast_first_fragment_kernel");
    p.first_frag = first;
  }

  const bool scatter = rast_scatter_path(ctx, n);
  if (spec) ctx->rast_inflight.fast = scatter ? 1 : 0;
  return scatter ? rast_launch_scatter(ctx, p, spec) : rast_launch_ordered(ctx, p, spec);
}
