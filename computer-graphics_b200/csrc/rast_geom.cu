// Geometry stage of the rasteriser's Draw on sm_100a
// (rasteriser/Source/skeleton.cpp:205-241): toCameraSpace :701-716,
// createShadowVolume :1676-1722, rotation :223-228, toClipSpace :691-699 and the
// six-plane clip :720-1673, order preserving.
//
// The reference clips the whole list plane after plane, each pass mapping a
// triangle to 0, 1 or 2 triangles and keeping list order.  A triangle's
// descendants never interact with another triangle's, so one thread carries one
// pre-clip triangle through all six planes with a small local list (at most 32
// descendants) and the final list is the concatenation in input order: a count
// pass, an exclusive scan, and a write pass.
//
// The reference spells the clip out as 6 planes x 7 hand-copied cases; they all
// instantiate one pattern, written once here, with the reference's two slips in
// the far plane kept (:1607 tests v2.x instead of v2.w; :1615 divides by
// (w1 - w0) instead of (w1 - w2)).
#include "rast_geom.cuh"
#include <limits.h>

struct GeomParams {
  GeomXform x;
  const rast_triangle *room;
  int n_room;
  const rast_triangle *boxes;
  int n_boxes;
  unsigned *counts;     // [n_pre + 1]
  unsigned *offs;       // [n_pre + 1] exclusive scan, total at [n_pre]
  rast_triangle *out;
  unsigned out_cap;
  unsigned long long *flags;   // bit0: a triangle whose texture field cannot be drawn (see tex_on), bit1: a shadow-coloured input triangle
  int tex_on;                  // rast_set_textures: texture 1..3 are drawn; otherwise only 0 is accepted
  // single-pass mode (pipelined frames): chained scan over the blocks
  unsigned *ticket;            // hands out block ids in scheduling order (forward progress of the look-back)
  unsigned long long *desc;    // per block: state << 62 | value; state 1 = block sum, 2 = inclusive prefix
  unsigned long long *total;   // list length
  // single-pass mode on a list bound for the scatter path: the blocks also clear the key buffer
  // (stores issued while their triangles are still on the way; saves a 66 MB memset launch at 4K)
  uint4 *clear;
  size_t clear_n;              // 16-byte units
  // single-pass mode, band culling (B200_OPT_RAST_BAND_CULL): only the triangles whose vertex rows
  // (VertexShader :513, truncated like :516) meet [cull0, cull1) are written, in list order, and
  // orig[] receives their indices in the complete list (what the owner-index output reports)
  int cull, cull0, cull1;
  int *orig;
  // single-pass mode launched in several chunks of blocks (a large scene still arriving from the
  // host: chunk k is transformed, clipped and scattered while chunk k + 1 is on the PCIe link):
  // blocks of the whole list, last block of this launch, where that block leaves the length of the
  // list written so far
  int n_blocks_total, chunk_last_bid;
  unsigned long long *chunk_hi;
};

// MODE 0: count the triangles each pre-clip triangle turns into; MODE 1: write them at the
// offsets a scan of the counts gave (exact sizes: two passes and a host read-back in between);
// MODE 2: one pass -- count, block scan, decoupled look-back over the preceding blocks'
// published sums, write -- into a list whose capacity was guessed (pipelined frames).
constexpr int GEOM_WARP_MAX_PRE = 8192;   // pre-clip triangles up to which a pipelined frame gives every triangle a warp

template <int MODE>
__global__ void __launch_bounds__(128) rast_geom_kernel(const __grid_constant__ GeomParams p) {
  constexpr bool WRITE = MODE != 0;
  constexpr int GT = 128, TW = sizeof(rast_triangle) / 4;
  __shared__ uint32_t stage[GT * TW];   // coalesced word streams in and out of the 84-byte records
  __shared__ unsigned s_bid, s_warp[4], s_prefix, s_prefix_all;
  if (MODE == 2) {
    if (threadIdx.x == 0) s_bid = atomicAdd(p.ticket, 1u);
    __syncthreads();
  }
  const int bid = MODE == 2 ? (int)s_bid : (int)blockIdx.x;
  if (MODE == 2 && p.clear_n) {   // (set for the first chunk's launch only: its block ids start at 0)
    const size_t per = (p.clear_n + gridDim.x - 1) / gridDim.x;
    const size_t a = (size_t)bid * per, b = a + per < p.clear_n ? a + per : p.clear_n;
    for (size_t i = a + threadIdx.x; i < b; i += GT) p.clear[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  const int j0 = bid * GT;
  const int j = j0 + threadIdx.x;
  const int n_pre = p.n_room + 7 * p.n_boxes;
  // a block whose triangles all come from `room` reads them through shared memory
  const bool staged_in = j0 + GT <= p.n_room;
  if (staged_in) {
    const uint32_t *src = reinterpret_cast<const uint32_t *>(p.room + j0);
    for (int i = threadIdx.x; i < GT * TW; i += GT) stage[i] = __ldg(src + i);
    __syncthreads();
  }
  // ---- the pre-clip triangle j (Draw :205-220) ----
  const rast_triangle *srcp;
  int s = 0;
  const int jj = j < n_pre ? j : n_pre - 1;   // tail threads repeat the last triangle, their output is dropped
  if (staged_in) srcp = reinterpret_cast<const rast_triangle *>(stage + threadIdx.x * TW);
  else if (jj < p.n_room) srcp = p.room + jj;
  else { srcp = p.boxes + (jj - p.n_room) / 7; s = (jj - p.n_room) % 7; }
  GTri t;
  float attr[9];   // normal[4], color[3], texture, index (bit-cast)
  geom_preclip(p.x, srcp, s, t, attr);
  // ---- six planes, list order preserved (:236-241) ----
  // Fast path: a triangle inside all six planes comes out unchanged.
  GTri cur[32];
  int n_cur = 1;
  const bool all_in = geom_all_in(p.x, t);
  cur[0] = t;
  if (!all_in) n_cur = clip_six_planes(p.x.W, p.x.H, p.x.focal, cur);
  if (MODE != 1 && j < n_pre) {
    const int texture = __float_as_int(attr[7]);
    if (texture != 0 && (!p.tex_on || texture < 0 || texture > 3)) atomicOr(p.flags, 1ull);
    if (s == 0 && !(attr[4] >= 0.0f)) atomicOr(p.flags, 2ull);
  }
  if (MODE == 0) {
    if (j < n_pre) p.counts[j] = (unsigned)n_cur;
    return;
  }
  // ---- single pass: which descendants are kept, where they go ----
  // kept: bit i set when descendant i is written (all of them unless the band is culled)
  unsigned kept = n_cur >= 32 ? 0xffffffffu : ((1u << n_cur) - 1u);
  if (MODE == 2 && p.cull) {
    kept = 0;
    for (int i = 0; i < n_cur; ++i) {
      int ymin = INT_MAX, ymax = INT_MIN;
      bool ok = true;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const GV &v = cur[i].v[k];
        const float y = xadd(xmul(p.x.focal, xdiv(v.y, v.z)), (float)(p.x.H / 2));   // :513
        ok = ok && fabsf(y) < 2147483648.0f;                // not convertible: the triangle loop drops it (rast_vertex)
        const int yi = ok ? (int)y : 0;                     // :516 static_cast<int>
        ymin = min(ymin, yi); ymax = max(ymax, yi);
      }
      if (ok && ymax >= p.cull0 && ymin < p.cull1) kept |= 1u << i;
    }
  }
  if (j >= n_pre) kept = 0;
  unsigned my_off = 0, my_all = 0;   // first kept output of this thread in the written list / first descendant in the complete list
  const unsigned cnt_all = j < n_pre ? (unsigned)n_cur : 0u, cnt_kept = (unsigned)__popc(kept);
  if (MODE == 2) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned incl = cnt_all | (cnt_kept << 16);   // both counts in one scan: at most 32 each per thread, 4096 per block
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    unsigned before = 0, block_sum = 0;
#pragma unroll
    for (int w = 0; w < 4; ++w) { before += w < warp ? s_warp[w] : 0u; block_sum += s_warp[w]; }
    const unsigned long long block_val = (unsigned long long)(block_sum & 0xffffu) | ((unsigned long long)(block_sum >> 16) << 31);
    if (warp == 0) {
      // Decoupled look-back by the whole warp: lane l inspects the block l places back; the
      // window moves 32 blocks at a time until it contains a block whose inclusive prefix is known.
      // Every block before this one already holds its ticket, so it will publish.  The value carries
      // two sums: complete list (low 31 bits) and written list (next 31 bits).
      const unsigned long long VAL = (1ull << 62) - 1;
      if (lane == 0 && bid > 0) atomicExch(p.desc + bid, (1ull << 62) | block_val);
      unsigned long long prefix = 0;
      for (int base = bid - 1;;) {
        const int k = base - lane;
        const unsigned long long v = k >= 0 ? atomicAdd(p.desc + k, 0ull) : (2ull << 62);   // "block -1": prefix 0
        const unsigned state = (unsigned)(v >> 62);
        const unsigned ready = __ballot_sync(0xffffffffu, state != 0), done = __ballot_sync(0xffffffffu, state == 2);
        const int first = done ? __ffs(done) - 1 : 31;                 // nearest block with an inclusive prefix
        const unsigned need = first == 31 ? 0xffffffffu : ((2u << first) - 1u);
        if ((ready & need) != need) continue;                            // someone in the window has not published yet
        unsigned long long part = lane <= first ? (v & VAL) : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        prefix += part;
        if (done) break;
        base -= 32;
      }
      if (lane == 0) {
        atomicExch(p.desc + bid, (2ull << 62) | (prefix + block_val));
        if (bid == p.n_blocks_total - 1) *p.total = (prefix + block_val) >> 31;   // length of the written list
        if (bid == p.chunk_last_bid && p.chunk_hi) *p.chunk_hi = (prefix + block_val) >> 31;
        s_prefix = (unsigned)(prefix >> 31);
        s_prefix_all = (unsigned)(prefix & 0x7fffffffull);
      }
    }
    __syncthreads();
    const unsigned ex = before + incl - (cnt_all | (cnt_kept << 16));   // exclusive, both halves (no carry: sums < 65536)
    my_off = s_prefix + (ex >> 16);
    my_all = s_prefix_all + (ex & 0xffffu);
  }
  // Common case: no triangle of the block is clipped (at most one output each): the kept records
  // go through shared memory, compacted, and leave as one coalesced stream.
  if (__syncthreads_and(staged_in && n_cur == 1)) {
    const unsigned off0 = MODE == 2 ? s_prefix : p.offs[j0];
    const unsigned slot = MODE == 2 ? my_off - off0 : threadIdx.x;   // position among the block's kept records
    __syncthreads();   // (every thread has read its input record from `stage`)
    if (kept) {
      float *o = reinterpret_cast<float *>(stage) + slot * TW;
      const GTri &g = cur[0];
      o[0] = x86_nan(g.v[0].x); o[1] = x86_nan(g.v[0].y); o[2] = x86_nan(g.v[0].z); o[3] = x86_nan(g.v[0].w);
      o[4] = x86_nan(g.v[1].x); o[5] = x86_nan(g.v[1].y); o[6] = x86_nan(g.v[1].z); o[7] = x86_nan(g.v[1].w);
      o[8] = x86_nan(g.v[2].x); o[9] = x86_nan(g.v[2].y); o[10] = x86_nan(g.v[2].z); o[11] = x86_nan(g.v[2].w);
#pragma unroll
      for (int k = 0; k < 9; ++k) o[12 + k] = attr[k];   // (room triangles: the caller's attributes)
      if (MODE == 2 && p.orig && my_off < p.out_cap) p.orig[my_off] = (int)my_all;
    }
    const unsigned n_out = MODE == 2 ? (s_warp[0] + s_warp[1] + s_warp[2] + s_warp[3]) >> 16 : (unsigned)GT;
    __syncthreads();
    uint32_t *dst = reinterpret_cast<uint32_t *>(p.out + off0);
    if (off0 + n_out <= p.out_cap)
      for (int i = threadIdx.x; i < (int)n_out * TW; i += GT) dst[i] = stage[i];
    return;
  }
  if (j >= n_pre) return;
  unsigned off = MODE == 2 ? my_off : p.offs[j];
  for (int i = 0; i < n_cur; ++i) {
    if (!((kept >> i) & 1u)) continue;
    if (off >= p.out_cap) break;
    rast_triangle *o = p.out + off;
    const GTri &g = cur[i];
    o->v0[0] = x86_nan(g.v[0].x); o->v0[1] = x86_nan(g.v[0].y); o->v0[2] = x86_nan(g.v[0].z); o->v0[3] = x86_nan(g.v[0].w);
    o->v1[0] = x86_nan(g.v[1].x); o->v1[1] = x86_nan(g.v[1].y); o->v1[2] = x86_nan(g.v[1].z); o->v1[3] = x86_nan(g.v[1].w);
    o->v2[0] = x86_nan(g.v[2].x); o->v2[1] = x86_nan(g.v[2].y); o->v2[2] = x86_nan(g.v[2].z); o->v2[3] = x86_nan(g.v[2].w);
#pragma unroll
    for (int k = 0; k < 4; ++k) o->normal[k] = s ? x86_nan(attr[k]) : attr[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) o->color[k] = attr[4 + k];
    o->texture = __float_as_int(attr[7]);
    o->index = __float_as_int(attr[8]);
    if (MODE == 2 && p.orig) p.orig[off] = (int)(my_all + i);
    ++off;
  }
}

// Short lists -- the reference's own scene is 10 room + 20 box triangles = 150 pre-clip triangles, 120 of them
// shadow-volume sides that nearly every plane cuts: with one thread per triangle the frame waited 32 us for the
// longest chain of six planes x up to 32 descendants walked by a single lane out of local memory.  Here one WARP
// takes a pre-clip triangle and lane i holds descendant i in registers: per plane every lane clips its own
// triangle (clip_one, the same code), an exclusive prefix of the 0 / 1 / 2 results gives the places in the
// reference's list order (:236-241: the list is rebuilt plane by plane, each triangle followed by its extra
// triangle), and the descendants change lanes through shared memory.  Blocks chain their counts through the same
// decoupled look-back as rast_geom_kernel<2>.  Pipelined frames without band culling / key clearing / chunks.
constexpr int GW_WARPS = 4;
__global__ void __launch_bounds__(32 * GW_WARPS) rast_geom_warp_kernel(const __grid_constant__ GeomParams p) {
  __shared__ float xch[GW_WARPS][12][32];
  __shared__ unsigned s_bid, s_cnt[GW_WARPS], s_prefix;
  if (threadIdx.x == 0) s_bid = atomicAdd(p.ticket, 1u);
  __syncthreads();
  const int bid = (int)s_bid, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n_pre = p.n_room + 7 * p.n_boxes;
  const int j = bid * GW_WARPS + warp;
  const int jj = j < n_pre ? j : n_pre - 1;   // tail warps repeat the last triangle, their output is dropped
  const rast_triangle *srcp;
  int s = 0;
  if (jj < p.n_room) srcp = p.room + jj;
  else { srcp = p.boxes + (jj - p.n_room) / 7; s = (jj - p.n_room) % 7; }
  GTri mine;
  float attr[9];   // normal[4], color[3], texture, index (bit-cast)
  geom_preclip(p.x, srcp, s, mine, attr);      // every lane the same triangle
  int n_cur = 1;
  if (!geom_all_in(p.x, mine)) {
    const float wfar = xdiv(5.0f, p.x.focal);
    float (*xw)[32] = xch[warp];
    for (int plane = 1; plane <= 6 && n_cur > 0; ++plane) {
      ClipCtx c;
      c.plane = plane; c.W = p.x.W; c.H = p.x.H; c.focal = p.x.focal; c.wfar = wfar;
      GTri o0, o1;
      int m = 0;
      if (lane < n_cur) m = clip_one(c, mine, o0, o1);
      int incl = m;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
      }
      const int total = __shfl_sync(0xffffffffu, incl, 31), at = incl - m;
      __syncwarp();                                   // the previous plane's reads are done
      auto put = [&](const GTri &g, int k) {
        xw[0][k] = g.v[0].x; xw[1][k] = g.v[0].y; xw[2][k] = g.v[0].z; xw[3][k] = g.v[0].w;
        xw[4][k] = g.v[1].x; xw[5][k] = g.v[1].y; xw[6][k] = g.v[1].z; xw[7][k] = g.v[1].w;
        xw[8][k] = g.v[2].x; xw[9][k] = g.v[2].y; xw[10][k] = g.v[2].z; xw[11][k] = g.v[2].w;
      };
      if (m >= 1 && at < 32) put(o0, at);
      if (m == 2 && at + 1 < 32) put(o1, at + 1);
      __syncwarp();
      n_cur = min(total, 32);                         // (five doubling planes: 32 is the reference's own maximum)
      if (lane < n_cur) {
        mine.v[0].x = xw[0][lane]; mine.v[0].y = xw[1][lane]; mine.v[0].z = xw[2][lane]; mine.v[0].w = xw[3][lane];
        mine.v[1].x = xw[4][lane]; mine.v[1].y = xw[5][lane]; mine.v[1].z = xw[6][lane]; mine.v[1].w = xw[7][lane];
        mine.v[2].x = xw[8][lane]; mine.v[2].y = xw[9][lane]; mine.v[2].z = xw[10][lane]; mine.v[2].w = xw[11][lane];
      }
    }
  }
  if (lane == 0 && j < n_pre) {
    const int texture = __float_as_int(attr[7]);
    if (texture != 0 && (!p.tex_on || texture < 0 || texture > 3)) atomicOr(p.flags, 1ull);
    if (s == 0 && !(attr[4] >= 0.0f)) atomicOr(p.flags, 2ull);
  }
  const unsigned cnt = j < n_pre ? (unsigned)n_cur : 0u;
  if (lane == 0) s_cnt[warp] = cnt;
  __syncthreads();
  unsigned before = 0, block_sum = 0;
#pragma unroll
  for (int w = 0; w < GW_WARPS; ++w) { before += w < warp ? s_cnt[w] : 0u; block_sum += s_cnt[w]; }
  if (warp == 0) {
    // decoupled look-back by the whole warp, as in rast_geom_kernel<2> (one sum: nothing is culled here)
    const unsigned long long VAL = (1ull << 62) - 1, block_val = block_sum;
    if (lane == 0 && bid > 0) atomicExch(p.desc + bid, (1ull << 62) | block_val);
    unsigned long long prefix = 0;
    for (int base = bid - 1;;) {
      const int k = base - lane;
      const unsigned long long v = k >= 0 ? atomicAdd(p.desc + k, 0ull) : (2ull << 62);   // "block -1": prefix 0
      const unsigned state = (unsigned)(v >> 62);
      const unsigned ready = __ballot_sync(0xffffffffu, state != 0), done = __ballot_sync(0xffffffffu, state == 2);
      const int first = done ? __ffs(done) - 1 : 31;
      const unsigned need = first == 31 ? 0xffffffffu : ((2u << first) - 1u);
      if ((ready & need) != need) continue;
      unsigned long long part = lane <= first ? (v & VAL) : 0ull;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
      prefix += part;
      if (done) break;
      base -= 32;
    }
    if (lane == 0) {
      atomicExch(p.desc + bid, (2ull << 62) | (prefix + block_val));
      if (bid == p.n_blocks_total - 1) *p.total = prefix + block_val;   // length of the list
      s_prefix = (unsigned)prefix;
    }
  }
  __syncthreads();
  const unsigned off = s_prefix + before + (unsigned)lane;
  if (j < n_pre && lane < n_cur && off < p.out_cap) {
    rast_triangle *o = p.out + off;
    o->v0[0] = x86_nan(mine.v[0].x); o->v0[1] = x86_nan(mine.v[0].y); o->v0[2] = x86_nan(mine.v[0].z); o->v0[3] = x86_nan(mine.v[0].w);
    o->v1[0] = x86_nan(mine.v[1].x); o->v1[1] = x86_nan(mine.v[1].y); o->v1[2] = x86_nan(mine.v[1].z); o->v1[3] = x86_nan(mine.v[1].w);
    o->v2[0] = x86_nan(mine.v[2].x); o->v2[1] = x86_nan(mine.v[2].y); o->v2[2] = x86_nan(mine.v[2].z); o->v2[3] = x86_nan(mine.v[2].w);
#pragma unroll
    for (int k = 0; k < 4; ++k) o->normal[k] = s ? x86_nan(attr[k]) : attr[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) o->color[k] = attr[4 + k];
    o->texture = __float_as_int(attr[7]);
    o->index = __float_as_int(attr[8]);
  }
}

// Exclusive scan of counts[0..n) into offs[0..n], total at offs[n]: per-block
// sums, a one-block scan of those, then per-block scans with their offsets.
constexpr int SCAN_THREADS = 1024, SCAN_ITEMS = 4, SCAN_BLOCK = SCAN_THREADS * SCAN_ITEMS;

// Exclusive prefix of `v` over the block (all SCAN_THREADS threads call); total in *total.
__device__ __forceinline__ unsigned block_excl_scan(unsigned v, unsigned *total) {
  __shared__ unsigned warp_excl[32];
  __shared__ unsigned block_total;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  unsigned incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned m = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += m;
  }
  __syncthreads();   // protects warp_excl / block_total across back-to-back calls
  if (lane == 31) warp_excl[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    const unsigned w = lane < nw ? warp_excl[lane] : 0u;
    unsigned wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned m = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += m;
    }
    warp_excl[lane] = wi - w;
    if (lane == 31) block_total = wi;
  }
  __syncthreads();
  *total = block_total;
  return warp_excl[warp] + incl - v;
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_reduce_kernel(const unsigned *__restrict__ counts, int n,
                                                                   unsigned *__restrict__ block_sums) {
  const int base = blockIdx.x * SCAN_BLOCK + threadIdx.x * SCAN_ITEMS;
  unsigned s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) s += base + k < n ? counts[base + k] : 0u;
  unsigned total;
  block_excl_scan(s, &total);
  if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

// In-place exclusive scan of block_sums[0..nb), grand total at block_sums[nb]; one block.
__global__ void __launch_bounds__(SCAN_THREADS) scan_sums_kernel(unsigned *__restrict__ block_sums, int nb) {
  unsigned carry = 0;
  for (int base = 0; base < nb; base += SCAN_THREADS) {
    const int i = base + threadIdx.x;
    const unsigned v = i < nb ? block_sums[i] : 0u;
    unsigned total;
    const unsigned ex = block_excl_scan(v, &total);
    if (i < nb) block_sums[i] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0) block_sums[nb] = carry;
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_apply_kernel(const unsigned *__restrict__ counts, int n,
                                                                  const unsigned *__restrict__ block_sums, int nb,
                                                                  unsigned *__restrict__ offs,
                                                                  unsigned long long *__restrict__ total_out) {
  const int base = blockIdx.x * SCAN_BLOCK + threadIdx.x * SCAN_ITEMS;
  unsigned v[SCAN_ITEMS], s = 0;
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) { v[k] = base + k < n ? counts[base + k] : 0u; s += v[k]; }
  unsigned total;
  unsigned run = block_sums[blockIdx.x] + block_excl_scan(s, &total);
#pragma unroll
  for (int k = 0; k < SCAN_ITEMS; ++k) {
    if (base + k < n) offs[base + k] = run;
    run += v[k];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    offs[n] = block_sums[nb];
    if (total_out) *total_out = block_sums[nb];
  }
}

// offs[0..n] = exclusive scan of counts[0..n); tmp holds nb + 1 block sums.
int scan_exclusive(b200_ctx *ctx, const unsigned *counts, unsigned *offs, int n, unsigned *tmp,
                   unsigned long long *total_out) {
  const int nb = (n + SCAN_BLOCK - 1) / SCAN_BLOCK;
  scan_reduce_kernel<<<nb, SCAN_THREADS, 0, ctx->stream>>>(counts, n, tmp);
  scan_sums_kernel<<<1, SCAN_THREADS, 0, ctx->stream>>>(tmp, nb);
  scan_apply_kernel<<<nb, SCAN_THREADS, 0, ctx->stream>>>(counts, n, tmp, nb, offs, total_out);
  ctx->stats.kernel_launches += 3;
  tl_mark(ctx, "scan_apply_kernel");
  CU_CHECK(ctx, cudaGetLastError());
  return B200_OK;
}

// Camera / light part of the stage on the host: the per-triangle transform's constants and the
// camera-space rotated light the triangle loop's calculateIllumination reads (:675).
void rast_geom_xform(const camera_t *cam, const rast_light_t *light, GeomXform *x, rast_light_t *light_out) {
  x->W = cam->width; x->H = cam->height; x->focal = cam->focal;
  memcpy(x->cam, cam->pos, sizeof x->cam);
  memcpy(x->R, cam->R, sizeof x->R);
  // lightPos = sceneCoordinatesLightPos - cameraPos, w = 1 (:211-212, :713-716); then R * lightPos (:223)
  volatile float lx = light->pos[0] - cam->pos[0], ly = light->pos[1] - cam->pos[1], lz = light->pos[2] - cam->pos[2];
  x->light_cam[0] = lx; x->light_cam[1] = ly; x->light_cam[2] = lz; x->light_cam[3] = 1.0f;
  *light_out = *light;
  for (int r = 0; r < 4; ++r) {
    volatile float a = cam->R[0 + r] * x->light_cam[0], b = cam->R[4 + r] * x->light_cam[1];
    volatile float c = cam->R[8 + r] * x->light_cam[2], d = cam->R[12 + r] * x->light_cam[3];
    volatile float ab = a + b, cd = c + d;
    light_out->pos[r] = ab + cd;
  }
}

// Host: runs the stage on the uploaded world-space scene; leaves the clipped list
// in ctx->rast_src / ctx->rast_n_tris and the camera-space rotated light in
// light_out (what the triangle loop's calculateIllumination reads, :675).
int rast_geometry(b200_ctx *ctx, const camera_t *cam, const rast_light_t *light, rast_light_t *light_out,
                  bool spec) {
  const int n_room = ctx->rast_n_room, n_boxes = ctx->rast_n_boxes;
  const int n_pre = n_room + 7 * n_boxes;
  GeomParams p;
  memset(&p, 0, sizeof p);
  rast_geom_xform(cam, light, &p.x, light_out);
  p.room = (const rast_triangle *)ctx->rast_world.p;
  p.n_room = n_room;
  p.boxes = p.room + n_room;
  p.n_boxes = n_boxes;
  const int n_scan_blocks = (n_pre + SCAN_BLOCK - 1) / SCAN_BLOCK;
  const int n_blocks = (n_pre + 127) / 128;
  const bool short_list = n_pre <= GEOM_WARP_MAX_PRE;   // pipelined frames: a warp per pre-clip triangle (rast_geom_warp_kernel)
  const int n_blocks_warp = (n_pre + GW_WARPS - 1) / GW_WARPS;
  const int n_desc = short_list && n_blocks_warp > n_blocks ? n_blocks_warp : n_blocks;
  const size_t tmp_words = 2 * (size_t)(n_pre + 1) + n_scan_blocks + 2;          // counts, offsets, scan scratch
  const size_t chain_off = (tmp_words * sizeof(unsigned) + 15) / 16 * 16;        // then: ticket (16 B), block descriptors
  if (int rc = ensure(ctx, ctx->rast_geom_tmp, chain_off + 16 + sizeof(unsigned long long) * (size_t)(n_desc + 1))) return rc;
  p.flags = (unsigned long long *)ctx->counters.p + 7;
  p.tex_on = ctx->rast_tex_on;
  p.counts = (unsigned *)ctx->rast_geom_tmp.p;
  p.offs = p.counts + (n_pre + 1);
  p.ticket = (unsigned *)((char *)ctx->rast_geom_tmp.p + chain_off);
  p.desc = (unsigned long long *)((char *)ctx->rast_geom_tmp.p + chain_off + 16);
  p.total = (unsigned long long *)ctx->counters.p + 24;
  if (spec && n_pre > 0) {
    // pipelined: one pass into a list whose capacity comes from the last verified frame; the
    // list length stays on the device ([24]) and the guess is checked when the frame is waited for
    unsigned long long cap = rast_spec_cap(ctx->rast_spec.tris);
    if (cap > 0x3fffffffull) cap = 0x3fffffffull;
    if (int rc = ensure(ctx, ctx->rast_src, sizeof(rast_triangle) * (size_t)cap)) return rc;
    p.out = (rast_triangle *)ctx->rast_src.p;
    p.out_cap = (unsigned)cap;
    CU_CHECK(ctx, cudaMemsetAsync(p.ticket, 0, 16 + sizeof(unsigned long long) * (size_t)n_desc, ctx->stream));
    ctx->rast_culled = 0;
    if (ctx->rast_cull_on) {
      if (int rc = ensure(ctx, ctx->rast_orig, sizeof(int) * (size_t)cap)) return rc;
      p.cull = 1; p.cull0 = ctx->rast_cull0; p.cull1 = ctx->rast_cull1;
      p.orig = (int *)ctx->rast_orig.p;
      ctx->rast_culled = 1;
    }
    const bool clear = ctx->rast_clear_ptr && ((size_t)ctx->rast_clear_ptr & 15) == 0 && (ctx->rast_clear_bytes & 15) == 0;
    if (clear) ctx->rast_keys_cleared = 1;
    // A scene that is still arriving from the host in chunks (draw_raster_band on a large list): one
    // launch per chunk, each behind its chunk's copy; rast_launch scatters chunk k on the second
    // stream while chunk k + 1 is on the link.
    const int chunks = ctx->rast_geom_chunks;
    if (short_list && !ctx->rast_cull_on && !clear && chunks == 1) {
      p.n_blocks_total = n_blocks_warp;
      rast_geom_warp_kernel<<<n_blocks_warp, 32 * GW_WARPS, 0, ctx->stream>>>(p);
      ctx->stats.kernel_launches++;
      tl_mark(ctx, "rast_geom_warp_kernel");
      CU_CHECK(ctx, cudaGetLastError());
      ctx->rast_n_tris = (int)cap;
      return B200_OK;
    }
    p.n_blocks_total = n_blocks;
    for (int c = 0; c < chunks; ++c) {
      const int b0 = chunks > 1 ? ctx->rast_up_edge[c] / 128 : 0;
      const int b1 = (chunks > 1 && c + 1 < chunks) ? ctx->rast_up_edge[c + 1] / 128 : n_blocks;
      p.clear = (clear && c == 0) ? (uint4 *)ctx->rast_clear_ptr : nullptr;
      p.clear_n = (clear && c == 0) ? ctx->rast_clear_bytes / 16 : 0;
      p.chunk_last_bid = b1 - 1;
      p.chunk_hi = chunks > 1 ? (unsigned long long *)ctx->counters.p + 12 + c : nullptr;
      ctx->rast_geom_chunk_tris[c] = (b1 - b0) * 128;
      if (chunks > 1) CU_CHECK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_up[c], 0));
      if (b1 > b0) rast_geom_kernel<2><<<b1 - b0, 128, 0, ctx->stream>>>(p);
      if (chunks > 1) CU_CHECK(ctx, cudaEventRecord(ctx->ev_chunk[c], ctx->stream));
    }
    ctx->stats.kernel_launches += chunks;
    tl_mark(ctx, "rast_geom_kernel<2>");
    CU_CHECK(ctx, cudaGetLastError());
    ctx->rast_n_tris = (int)cap;
    return B200_OK;
  }
  unsigned total = 0;
  ctx->rast_culled = 0;
  if (n_pre > 0) {
    rast_geom_kernel<0><<<(n_pre + 127) / 128, 128, 0, ctx->stream>>>(p);
    ctx->stats.kernel_launches++;
    tl_mark(ctx, "rast_geom_kernel");
    CU_CHECK(ctx, cudaGetLastError());
    unsigned long long *dc = (unsigned long long *)ctx->counters.p;
    if (int rc = scan_exclusive(ctx, p.counts, p.offs, n_pre, p.offs + (n_pre + 1), dc + 24)) return rc;
    {
      // one small read-back into pinned memory: [7] validation flags, [24] clipped-list length
      unsigned long long *hc = (unsigned long long *)ctx->pinned;
      CU_CHECK(ctx, cudaMemcpyAsync(hc, dc, 32 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
      CU_CHECK(ctx, cudaStreamSynchronize(ctx->stream));
      const unsigned long long flags = hc[7];
      total = (unsigned)hc[24];
      if (flags & 1ull) return ctx_fail(ctx, B200_EINVAL, "texture != 0 needs rast_set_textures and must be 1..3");
      ctx->rast_has_shadow = (n_boxes > 0 || (flags & 2ull)) ? 1 : 0;
    }
  }
  if (int rc = ensure(ctx, ctx->rast_src, sizeof(rast_triangle) * (size_t)(total ? total : 1))) return rc;
  p.out = (rast_triangle *)ctx->rast_src.p;
  p.out_cap = total;
  if (total > 0) {
    rast_geom_kernel<1><<<(n_pre + 127) / 128, 128, 0, ctx->stream>>>(p);
    ctx->stats.kernel_launches++;
    tl_mark(ctx, "rast_geom_kernel");
    CU_CHECK(ctx, cudaGetLastError());
  }
  ctx->rast_n_tris = (int)total;
  return B200_OK;
}
