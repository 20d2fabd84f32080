// Fast path of the rasteriser for lists WITHOUT shadow-volume triangles.
//
// With only opaque triangles the reference's fold (`zinv >= depth`, drawn in
// list order, rasteriser/Source/skeleton.cpp:574,665) is order independent: the
// pixel ends up owned by the fragment with the largest zinv, the LATEST triangle
// on ties.  That is a lexicographic maximum of (zinv, index), so fragments can be
// scattered in any order with one 64-bit atomic max per fragment on
//   key = zinv bits << 32 | (triangle index + 1)          (0 = empty pixel)
// (non-negative floats order like their bit patterns; fragments with zinv < 0 or
// NaN fail `zinv >= depth` against the cleared buffer and are never drawn).
//
//   rast_scatter2_kernel    one thread per triangle, straight from the 84-byte list
//                           (no setup record in HBM): VertexShader, the per-edge steps,
//                           then the reference's own edge walk (ComputePolygonRows
//                           :481-495, sample by sample) into a packed row table in
//                           shared memory.  The (triangle,row) pairs of a warp are then
//                           dealt out evenly over its lanes: row record (span ends and
//                           steps, :502-503), slim copy for the resolve pass, one atomic
//                           max per fragment that can still win.  Triangles too large
//                           for the shared-memory table go to a list for
//   rast_setup_big_kernel + rast_scatter_kernel   per big triangle / per (big triangle,row):
//                           the closed-form row records of rast_kernels.cu.
//   rast_resolve_kernel     per 32x8 pixel tile + 1-pixel halo: the winners are
//                           compacted, each winning fragment is re-derived exactly
//                           from its row record (fragment, three
//                           calculateIllumination) into shared memory, then the 5-tap
//                           AA / HDR mean of the post pass (:283-307; no shadow flags
//                           => nothing is darkened) is taken from shared memory and
//                           the frame written once.
// HBM holds per drawn row 20 bytes (left x, left p*zinv and steps; small triangles: at a place the key
// itself names, big ones: through 8 bytes per triangle); no per-pixel colour buffers and no tile lists.
#pragma once

// Low word of a key: (triangle << 5 | code) + 1.  Triangle order decides ties, as in the reference;
// the code tells the resolve pass where the fragment's row record is WITHOUT another look-up:
// code < S2_ROWS: a small triangle, record at triangle * S2_ROWS + code (code = y mod S2_ROWS: a small
// triangle spans at most S2_ROWS rows, so y mod S2_ROWS is unique within it); RAST_CODE_BIG: a big
// triangle, rows found through trimeta.
constexpr int S2_ROWS = 24;       // a "small" triangle spans at most this many rows
constexpr unsigned RAST_CODE_BIG = 31u;
constexpr int RAST_FAST_MAX_TRIS = 1 << 27;
__device__ __forceinline__ unsigned long long rast_key(float zinv, unsigned low) {
  const unsigned hi = zinv == 0.0f ? 0u : __float_as_uint(zinv);   // -0.0 passes `>= 0` too
  return ((unsigned long long)hi << 32) | (low + 1u);
}

// red.max on a key with an L2 evict-last policy: the 64-bit keys (66 MB at 4K) are what the
// scatter revisits at random, while the triangles it reads and the row records it writes
// stream through once -- the policy keeps the keys resident while those pass.
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void red_max_u64_keep(unsigned long long *addr, unsigned long long v, uint64_t pol) {
  asm volatile("red.relaxed.gpu.global.max.L2::cache_hint.u64 [%0], %1, %2;" ::"l"(addr), "l"(v), "l"(pol) : "memory");
}

// The fragments x0 <= x < x1 of one span (:504, :573): one atomic max per fragment, fire and
// forget.  (A plain read in front of the atomic, to skip fragments that are already beaten, was
// measured: the dependent L2 round trip per fragment made the span loop latency bound -- 49 % of
// the kernel's stall samples -- while the atomics themselves are far from the REDG rate.)
__device__ __forceinline__ void rast_span_scatter(unsigned long long *row, int lx, int x0, int x1, float zl, float zs,
                                                  unsigned low, uint64_t keep) {
  for (int x = x0; x < x1; ++x) {
    const float zinv = xadd(zl, xmul(zs, (float)(x - lx)));   // :543
    if (zinv >= 0.0f) red_max_u64_keep(row + x, rast_key(zinv, low), keep);   // :574 against the cleared buffer
  }
}

constexpr int S2_THREADS = 128;   // triangles per block
constexpr int S2_XSPAN = 60;      // a "small" triangle spans at most S2_ROWS rows and this many columns (edge samples and x offsets fit 6 bits)

// COUNT: only classifies and counts (big triangles [10], their
// rows [11]) so that a frame that cannot size its buffers from a verified predecessor gets exact
// sizes from one cheap extra pass.
template <bool COUNT>
__global__ void __launch_bounds__(S2_THREADS) rast_scatter2_kernel(const __grid_constant__ RastParams p) {
  constexpr int TW = sizeof(rast_triangle) / 4;
  // stage: the block's triangles, read as one coalesced word stream; once every thread holds its
  // triangle in registers the same memory carries the per-edge constants the row tasks need
  __shared__ uint32_t stage[S2_THREADS * TW];
  __shared__ unsigned rowtab[S2_ROWS * S2_THREADS];          // [row][thread]: left | right << 16, each x << 8 | edge << 6 | sample
  __shared__ unsigned short task[S2_THREADS / 32][32 * S2_ROWS];   // per warp: lane | table row << 5 of every row task
  __shared__ int org[2 * S2_THREADS];                        // [0][thread] x origin of the packed offsets, [1][thread] ymin, 
  float *epar = reinterpret_cast<float *>(stage);            // [edge * 6 + k][thread]: a.zinv, sz, a.px*a.zinv, spx, a.py*a.zinv, spy

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // (a launch for one geometry chunk works on the list range that chunk wrote; if the launch turns
  // out too small for it -- clipping added more than 3 % -- the frame is flagged and rendered again)
  const int lo = p.range_lo ? (int)*p.range_lo : 0;
  const int n_tris = p.range_hi ? (int)min((unsigned long long)p.n_tris, *p.range_hi) : rast_count_tris(p);
  if (p.range_hi && blockIdx.x == 0 && threadIdx.x == 0 && (long long)n_tris - lo > (long long)gridDim.x * S2_THREADS)
    atomicExch(p.counters + 5, 1ull);
  const int t0 = lo + blockIdx.x * S2_THREADS, t = t0 + tid;
  if (t0 >= n_tris) return;   // pipelined launches are sized by a bound on the list length
  const int n_here = min(S2_THREADS, n_tris - t0);
  {
    const uint32_t *src = reinterpret_cast<const uint32_t *>(p.src + t0);
    for (int i = tid; i < n_here * TW; i += S2_THREADS) stage[i] = __ldg(src + i);
  }
  __syncthreads();

  RastSetup s;
  int ymin = 0, xorg = 0, row_first = 0, cnt = 0, span_rows = 0;   // cnt: stored rows (band-clamped), small triangles only
  bool big = false;
  if (t < n_tris) {
    const float *tr = reinterpret_cast<const float *>(stage) + tid * TW;
    const bool ok = rast_tri_setup(tr, p.focal, p.W, p.H, s);
    if (ok) {
      ymin = min(s.v[0].y, min(s.v[1].y, s.v[2].y));
      const int ymax = max(s.v[0].y, max(s.v[1].y, s.v[2].y));
      const int vxmin = min(s.v[0].x, min(s.v[1].x, s.v[2].x)), xmax = max(s.v[0].x, max(s.v[1].x, s.v[2].x));
      xorg = vxmin - 1;                                     // a minor-axis sample can undershoot by one
      row_first = max(ymin, p.fb0);
      const int rlast = min(ymax, p.fb1 - 1);
      int nrows = max(0, rlast - row_first + 1);
      if (xmax <= 0 || xorg >= p.W || xmax <= xorg) nrows = 0;   // no pixel of [xorg, xmax) on screen
      span_rows = ymax - ymin + 1;
      big = nrows > 0 && (span_rows > S2_ROWS || xmax - vxmin > S2_XSPAN);
      cnt = big ? 0 : nrows;
      if (COUNT && big) atomicAdd(p.counters + 11, (unsigned long long)nrows);
    }
  }
  __syncthreads();   // every thread has its triangle in registers: `stage` may be overwritten

  // ---- big triangles: to the list of rast_setup_big_kernel (warp-aggregated append) ----
  {
    const unsigned m = __ballot_sync(0xffffffffu, big);
    if (m) {
      unsigned at0 = 0;
      if (lane == 0) at0 = (unsigned)atomicAdd(p.counters + 10, (unsigned long long)__popc(m));
      at0 = __shfl_sync(0xffffffffu, at0, 0);
      if (!COUNT && big) {
        const unsigned at = at0 + __popc(m & ((1u << lane) - 1));
        if (at < p.big_cap) p.big_list[at] = t;
        else atomicExch(p.counters + 5, 1ull);
      }
    }
  }
  if (COUNT) return;
  if (!__any_sync(0xffffffffu, cnt > 0)) return;   // nothing small and visible in this warp (no block barrier below)

  // ---- ComputePolygonRows (:455-495): every sample of the three edges, in order ----
  if (cnt > 0) {
    unsigned *rt = rowtab + tid;
    for (int r = 0; r < span_rows; ++r) rt[r * S2_THREADS] = 0xffffffffu;   // left.x = +INT_MAX, right.x = -INT_MAX
    const int n0 = max(abs(s.v[0].x - s.v[1].x), abs(s.v[0].y - s.v[1].y)) + 1;
    const int n1 = max(abs(s.v[1].x - s.v[2].x), abs(s.v[1].y - s.v[2].y)) + 1;
    const int n2 = max(abs(s.v[2].x - s.v[0].x), abs(s.v[2].y - s.v[0].y)) + 1;
    const int n_all = n0 + n1 + n2;
    float ax = (float)s.v[0].x, ay = (float)s.v[0].y, sx = s.sx[0], sy = s.sy[0];
    int e = 0, i = 0, ne = n0;
    for (int k = 0; k < n_all; ++k) {
      const float fi = (float)i;
      const int x = (int)floorf(xadd(ax, xmul(sx, fi)));   // :541
      const int y = (int)floorf(xadd(ay, xmul(sy, fi)));   // :542
      const int r = y - ymin;
      if (r >= 0 && r < span_rows) {                        // r < 0: the :485 guard
        const unsigned w = rt[r * S2_THREADS];
        const unsigned xr = (unsigned)(x - xorg);
        const unsigned f = (xr << 8) | ((unsigned)e << 6) | (unsigned)i;
        unsigned L = w & 0xffffu, R = w >> 16;
        if (L == 0xffffu || xr <= (L >> 8)) L = f;          // :487 `<=`: the later sample wins ties
        if (R == 0xffffu || xr >= (R >> 8)) R = f;          // :491 `>=`
        rt[r * S2_THREADS] = L | (R << 16);
      }
      if (++i == ne) {
        i = 0; ++e;
        const bool second = e == 1;
        ax = (float)(second ? s.v[1].x : s.v[2].x); ay = (float)(second ? s.v[1].y : s.v[2].y);
        sx = second ? s.sx[1] : s.sx[2]; sy = second ? s.sy[1] : s.sy[2];
        ne = second ? n1 : n2;
      }
    }
    // what the row tasks of OTHER lanes need of this triangle
#pragma unroll
    for (int ed = 0; ed < 3; ++ed) {
      const RastVtx &a = s.v[ed];
      epar[(ed * 6 + 0) * S2_THREADS + tid] = a.zinv;
      epar[(ed * 6 + 1) * S2_THREADS + tid] = s.sz[ed];
      epar[(ed * 6 + 2) * S2_THREADS + tid] = xmul(a.px, a.zinv);   // :526
      epar[(ed * 6 + 3) * S2_THREADS + tid] = s.spx[ed];
      epar[(ed * 6 + 4) * S2_THREADS + tid] = xmul(a.py, a.zinv);   // :527
      epar[(ed * 6 + 5) * S2_THREADS + tid] = s.spy[ed];
    }
    org[tid] = xorg;
    org[S2_THREADS + tid] = ymin;
  }
  // Row tasks: only rows that draw something (right end excluded, :504: a row whose ends
  // coincide -- the top and bottom rows of most small triangles -- has no fragment, and no
  // pixel can ever ask for its record).
  unsigned n_task = 0;
  if (cnt > 0) {
    const unsigned *rt = rowtab + tid;
    const int r_off = row_first - ymin;
    for (int r = 0; r < cnt; ++r) {
      const unsigned w = rt[(r_off + r) * S2_THREADS];
      n_task += (w != 0xffffffffu && (w >> 24) > ((w >> 8) & 0xffu)) ? 1u : 0u;
    }
  }
  unsigned tincl = n_task;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned n = __shfl_up_sync(0xffffffffu, tincl, o);
    if (lane >= o) tincl += n;
  }
  const unsigned n_tasks = __shfl_sync(0xffffffffu, tincl, 31);
  if (cnt > 0) {
    const unsigned *rt = rowtab + tid;
    const int r_off = row_first - ymin;
    unsigned at = tincl - n_task;
    for (int r = 0; r < cnt; ++r) {
      const unsigned w = rt[(r_off + r) * S2_THREADS];
      if (w != 0xffffffffu && (w >> 24) > ((w >> 8) & 0xffu)) task[warp][at++] = (unsigned short)(lane | ((r_off + r) << 5));
    }
  }
  __syncwarp();

  // ---- row tasks, dealt out evenly: DrawPolygonRows (:500-508) ----
  const uint64_t keep = l2_policy_evict_last();
  unsigned long long n_frag = 0;
  for (unsigned k = lane; k < n_tasks; k += 32) {
    const unsigned tk = task[warp][k];
    const int src = warp * 32 + (int)(tk & 31u), r = (int)(tk >> 5);
    const unsigned w = rowtab[r * S2_THREADS + src];
    const unsigned L = w & 0xffffu, R = w >> 16;
    {
      const int xo = org[src], y = org[S2_THREADS + src] + r;
      const int lx = xo + (int)(L >> 8);
      const int rx = xo + (int)(R >> 8);
      float zinv[2], px[2], py[2];
#pragma unroll
      for (int side = 0; side < 2; ++side) {
        const unsigned E = side ? R : L;
        const int ed = (int)((E >> 6) & 3u);
        const float fi = (float)(E & 63u);
        const float *ep = epar + (ed * 6) * S2_THREADS + src;
        zinv[side] = xadd(ep[0], xmul(ep[S2_THREADS], fi));                                  // :543
        px[side] = xdiv(xadd(ep[2 * S2_THREADS], xmul(ep[3 * S2_THREADS], fi)), zinv[side]);   // :547
        py[side] = xdiv(xadd(ep[4 * S2_THREADS], xmul(ep[5 * S2_THREADS], fi)), zinv[side]);   // :548
      }
      const float den = (float)max(rx - lx, 1);                      // Interpolate(left, right, rx - lx + 1) :502-503
      const float zs = xdiv_pos(xsub(zinv[1], zinv[0]), den);        // :535
      const float lpx = xmul(px[0], zinv[0]), lpy = xmul(py[0], zinv[0]);   // :526-527
      const float rpx = xmul(px[1], zinv[1]), rpy = xmul(py[1], zinv[1]);
      const float4 B = make_float4(lpx, xdiv_pos(xsub(rpx, lpx), den), lpy, xdiv_pos(xsub(rpy, lpy), den));
      const int x0 = max(lx, 0), x1 = min(rx, p.W);                  // right end excluded (:504); bounds (:573)
      const unsigned slot = (unsigned)y % (unsigned)S2_ROWS, tri = (unsigned)(t0 + src);
      rast_span_scatter(p.keys + (size_t)y * p.W, lx, x0, x1, zinv[0], zs, (tri << 5) | slot, keep);
      n_frag += x1 > x0 ? (unsigned long long)(x1 - x0) : 0ull;
      const size_t at = (size_t)tri * S2_ROWS + slot;
      __stcs(p.srowsB + at, B);   // for the resolve pass; streaming stores: the keys should stay in L2
      __stcs(p.srowsL + at, lx);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) n_frag += __shfl_xor_sync(0xffffffffu, n_frag, o);
  if (lane == 0 && n_frag) atomicAdd(p.counters + 16, n_frag);
}

// ---- big triangles -----------------------------------------------------------------------
// Setup record, row space and the owners of its row slots (the work items of rast_scatter_kernel)
// of every triangle rast_scatter2_kernel put on the big list.
__global__ void __launch_bounds__(128) rast_setup_big_kernel(const __grid_constant__ RastParams p) {
  const unsigned k = blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const unsigned n_big = (unsigned)min((unsigned long long)p.big_cap, p.counters[10]);
  int nrows = 0, t = 0;
  RastSetup s;
  s.flags = 0; s.ymin = 0; s.row0 = 0; s.nrows = 0; s.row_off = 0; s.tri = 0;
  if (k < n_big) {
    t = p.big_list[k];
    rast_tri_setup(reinterpret_cast<const float *>(p.src + t), p.focal, p.W, p.H, s);   // ok: rast_scatter2_kernel checked
    s.tri = t;
    const int ymin = min(s.v[0].y, min(s.v[1].y, s.v[2].y)), ymax = max(s.v[0].y, max(s.v[1].y, s.v[2].y));
    s.ymin = ymin;
    s.row0 = max(ymin, p.fb0);
    nrows = max(0, min(ymax, p.fb1 - 1) - s.row0 + 1);
    s.nrows = nrows;
  }
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
  if (k < n_big && s.row_off + (unsigned)nrows > p.row_cap) {
    s.nrows = 0; nrows = 0;
    atomicExch(p.counters + 5, 1ull);
  }
  warp_spread(nrows, (int)s.row_off, 0, 0, (int)k, [&](int j, int x0, int, int, int owner) { p.row_owner[(unsigned)x0 + j] = owner; });
  if (k < n_big) {
    p.setup[k] = s;
    if (nrows > 0) p.trimeta[t] = make_int2((int)s.row_off, s.row0);
  }
}

// One thread per row slot of the big triangles: closed-form row record, slim copy for the resolve
// pass, the span's fragments.
__global__ void rast_scatter_kernel(const __grid_constant__ RastParams p) {
  const unsigned slot = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long n_frag = 0;
  if (slot < rast_count_rows(p)) {
    const unsigned k = min((unsigned)p.row_owner[slot], p.big_cap ? p.big_cap - 1 : 0u);   // stale owner after an overflow
    const RastSetup &s = p.setup[k];
    const int r = (int)(slot - s.row_off);
    if (r >= 0 && r < s.nrows) {
      const int y = s.row0 + r;
      float4 A, B;
      rast_row_record<true>(s, y, A, B);
      const int lx = __float_as_int(A.x), rx = __float_as_int(A.y);
      __stcs(p.rowsB + slot, B);
      __stcs(p.rowsL + slot, lx);
      const int x0 = max(lx, 0), x1 = min(rx, p.W);      // right end excluded (:504); bounds (:573)
      rast_span_scatter(p.keys + (size_t)y * p.W, lx, x0, x1, A.z, A.w, ((unsigned)s.tri << 5) | RAST_CODE_BIG, l2_policy_evict_last());
      n_frag = x1 > x0 ? (unsigned long long)(x1 - x0) : 0ull;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) n_frag += __shfl_xor_sync(0xffffffffu, n_frag, o);
  if ((threadIdx.x & 31) == 0 && n_frag) atomicAdd(p.counters + 16, n_frag);
}

constexpr int RS_W = 32, RS_H = 8, RS_HW = RS_W + 2, RS_HH = RS_H + 2, RS_N = RS_HW * RS_HH;   // tile + 1-pixel halo
constexpr int RS_HALO = 2 * RS_HW + 2 * RS_H;                                                   // halo positions
constexpr int RS_FW = RS_W + 4, RS_FH = RS_H + 4;                                               // shadow flags: 2-pixel halo

// ORDERED = false: the scatter path's keys (row record named by the key).  ORDERED = true: the
// ordered-tile path's per-pixel result (rast_fill_kernel with p.fused: depth bits << 32 | winner + 1,
// and a shadow flag per pixel) -- the same pass then also does the shadow softening of the post pass
// (:286-303), so that path keeps no colour buffers in HBM either.
// TEX (ordered path only): the winners' texture / index fields are honoured (rast_tex.cuh); the depth
// word is then not the winner's zinv (holes, :619 / :643), which is recomputed from the row record.
template <bool ORDERED, bool TEX>
__global__ void __launch_bounds__(RS_W * RS_H, 2048 / (RS_W * RS_H)) rast_resolve_kernel(const __grid_constant__ RastParams p) {
  static_assert(ORDERED || !TEX, "textures are drawn by the ordered path");
  __shared__ float col[9][RS_N];            // [screen rgb, low rgb, high rgb][position]: conflict-free taps
  __shared__ float zinv_s[RS_N];            // the winner's zinv (:665); 0 = empty
  __shared__ int owner[RS_N];
  __shared__ unsigned short work[RS_N];
  __shared__ int n_work;
  __shared__ __align__(16) float out_stage[RS_H][3 * RS_W];   // one row of RGB per warp, for 128-bit stores
  __shared__ unsigned char flag[ORDERED ? RS_FH * RS_FW : 1];   // shadowBuffer of the tile + 2-pixel halo

  const int tid = threadIdx.x, lane = tid & 31;
  const int tx = tid % RS_W, ty = tid / RS_W;                                   // a warp is one row of the tile
  const int x0 = blockIdx.x * RS_W - 1, y0 = p.row0 + blockIdx.y * RS_H - 1;   // halo origin

  if (tid == 0) n_work = 0;
  if (ORDERED) {
    for (int i = tid; i < RS_FH * RS_FW; i += RS_W * RS_H) {
      const int gx = x0 - 1 + i % RS_FW, gy = y0 - 1 + i / RS_FW;
      flag[i] = (gx >= 0 && gx < p.W && gy >= p.fb0 && gy < p.fb1) ? p.shadow8[(size_t)gy * p.W + gx] : (unsigned char)0;
    }
  }
  __syncthreads();

  // ---- the winners of the tile (every thread its own pixel) and of the 1-pixel halo (the first 84
  // threads one more); covered positions are appended to the work list, warp-aggregated ----
  auto take = [&](bool active, int hx, int hy) {
    const int pos = hy * RS_HW + hx;
    const int gx = x0 + hx, gy = y0 + hy;
    unsigned long long key = 0;
    if (active && gx >= 0 && gx < p.W && gy >= p.fb0 && gy < p.fb1) key = __ldcs(p.keys + (size_t)gy * p.W + gx);   // read once
    const bool covered = (ORDERED ? (unsigned)(key & 0xffffffffull) : (unsigned)(key != 0)) != 0;
    if (active) {
      owner[pos] = (int)(unsigned)(key & 0xffffffffull) - 1;             // scatter: triangle << 5 | code; ordered: triangle; or -1
      zinv_s[pos] = __uint_as_float((unsigned)(key >> 32));
      if (!covered) {
#pragma unroll
        for (int k = 0; k < 9; ++k) col[k][pos] = 0.f;                          // cleared buffers (:244-249)
      }
    }
    const unsigned m = __ballot_sync(0xffffffffu, covered);
    if (m) {
      int base = 0;
      if (lane == 0) base = atomicAdd(&n_work, __popc(m));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (covered) work[base + __popc(m & ((1u << lane) - 1))] = (unsigned short)pos;
    }
  };
  take(true, tx + 1, ty + 1);
  if (tid < (RS_HALO + 31) / 32 * 32) {   // whole warps
    const int h = tid;
    int hx, hy;
    if (h < RS_HW) { hx = h; hy = 0; }
    else if (h < 2 * RS_HW) { hx = h - RS_HW; hy = RS_HH - 1; }
    else if (h < 2 * RS_HW + RS_H) { hx = 0; hy = h - 2 * RS_HW + 1; }
    else { hx = RS_HW - 1; hy = h - 2 * RS_HW - RS_H + 1; }
    take(h < RS_HALO, h < RS_HALO ? hx : 0, h < RS_HALO ? hy : 0);
  }
  __syncthreads();

  // ---- deferred PixelShader of every winner (:575-586) ----
  const int nw = n_work;
  for (int k = tid; k < nw; k += RS_W * RS_H) {
    const int pos = work[k];
    const int gx = x0 + pos % RS_HW, gy = y0 + pos / RS_HW;
    int t;
    float4 B;
    int lx;
    float zinv_tex = 0.f;
    if (ORDERED) {
      t = owner[pos];
      const RastSetup *su = p.setup + t;
      const unsigned rr = su->row_off + (unsigned)(gy - su->row0);
      B = __ldg(p.rowsB + rr);
      if (TEX) {
        const float4 A = __ldg(p.rowsA + rr);
        lx = __float_as_int(A.x);
        zinv_tex = xadd(A.z, xmul(A.w, (float)(gx - lx)));          // :543 again: a later hole may have cleared the depth
      } else {
        lx = __float_as_int(__ldg(&p.rowsA[rr].x));
      }
    } else {
      const unsigned low = (unsigned)owner[pos], code = low & 31u;
      t = (int)(low >> 5);
      if (code < (unsigned)S2_ROWS) {                                 // small triangle: the record's place is in the key
        const size_t rr = (size_t)t * S2_ROWS + code;
        B = __ldg(p.srowsB + rr);
        lx = __ldg(p.srowsL + rr);
      } else {
        const int2 m = __ldg(p.trimeta + t);
        const unsigned rr = (unsigned)m.x + (unsigned)(gy - m.y);
        B = __ldg(p.rowsB + rr);
        lx = __ldg(p.rowsL + rr);
      }
    }
    const float fi = (float)(gx - lx);
    const float zinv = TEX ? zinv_tex : zinv_s[pos];                // as the scatter / fold computed it (:543)
    const float pz = xdiv(1.0f, zinv);                              // :546
    const float px = xdiv(xadd(B.x, xmul(B.y, fi)), zinv);          // :547
    const float py = xdiv(xadd(B.z, xmul(B.w, fi)), zinv);          // :548
    rast_shade<TEX>(p, t, gx, gy, px, py, pz, &col[0][pos], RS_N);  // :575-586 (TEX: :588-645)
  }
  __syncthreads();

  // ---- post pass on the core pixels (:283-307, antiAliasing :1736-1753) ----
  const int x = x0 + 1 + tx, y = y0 + 1 + ty;
  if (y >= p.row1) return;                                           // warp-uniform: a warp is one row
  const bool in_x = x < p.W;
  const int c0 = (ty + 1) * RS_HW + (tx + 1);
  const size_t q = (size_t)y * p.W + x;
  float out[3] = {0.f, 0.f, 0.f};
  const bool interior = y >= 1 && y <= p.H - 2 && x >= 1 && x <= p.W - 2;
  // The reference darkens screenBuffer in place while scanning row-major (:286-303): the cross at
  // (y,x) sees darkened (y,x), (y-1,x), (y,x-1) and original (y+1,x), (y,x+1); the amount depends on
  // the final shadow mask only (surroundingShadowSum :1725-1733: [y+1][x-1] twice, [y+1][x+1] never).
  float s0 = 0.f, s1 = 0.f, s2 = 0.f;
  if (ORDERED) {
    auto sub = [&](int yy, int xx) -> float {   // (yy, xx) relative to the pixel: flags of pixel (y + yy, x + xx)
      const int gy = y + yy, gx = x + xx;
      if (gy < 1 || gy > p.H - 2 || gx < 1 || gx > p.W - 2) return 0.f;   // never visited by the loop
      const unsigned char *f = flag + (ty + 2 + yy) * RS_FW + (tx + 2 + xx);
      if (f[0] != 1) return 0.f;
      const int sum = f[0] + f[-RS_FW] + f[-RS_FW - 1] + f[-RS_FW + 1] + f[RS_FW - 1] + f[RS_FW] + f[RS_FW - 1] + f[-1] + f[1];
      const double d = (double)xdiv((float)sum, 9.0f);
      return d < 0.6 ? 0.05f : d < 0.7 ? 0.08f : d < 0.8 ? 0.1f : d < 0.9 ? 0.12f : 0.3f;
    };
    s0 = sub(0, 0); s1 = sub(-1, 0); s2 = sub(0, -1);
  }
  // five empty, undarkened taps average to +0 exactly: nothing to compute (most pixels of a sparse scene)
  const bool any = (owner[c0] & owner[c0 - RS_HW] & owner[c0 + RS_HW] & owner[c0 - 1] & owner[c0 + 1]) >= 0 ||
                   s0 != 0.f || s1 != 0.f || s2 != 0.f;
  if (in_x && interior && any) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float acc[3];
#pragma unroll
      for (int b = 0; b < 3; ++b) {
        const float *cb = col[3 * b + c];
        float v0 = cb[c0], v1 = cb[c0 - RS_HW], v2 = cb[c0 - 1];
        if (ORDERED && b == 0) {   // the reference only subtracts where the flag is set; x - 0 == x keeps that exact
          if (s0 != 0.f) v0 = xsub(v0, s0);
          if (s1 != 0.f) v1 = xsub(v1, s1);
          if (s2 != 0.f) v2 = xsub(v2, s2);
        }
        float a = xadd(v0, v1);
        a = xadd(a, cb[c0 + RS_HW]);
        a = xadd(a, v2);
        a = xadd(a, cb[c0 + 1]);
        acc[b] = xdiv_const<5>(a);
      }
      out[c] = xdiv_const<3>(xadd(xadd(acc[0], acc[1]), acc[2]));     // :1750
    }
  }
  if (p.out_rgb) {
    const int xs = x0 + 1;                                           // first pixel of the warp's row segment
    if (xs + RS_W <= p.W && (p.W & 3) == 0) {
      // 32 pixels x 3 floats = 24 x 128-bit stores per warp instead of 96 scalar ones
      float *st = out_stage[ty];
      st[3 * tx] = out[0]; st[3 * tx + 1] = out[1]; st[3 * tx + 2] = out[2];
      __syncwarp();
      if (lane < 3 * RS_W / 4)
        reinterpret_cast<float4 *>(p.out_rgb + 3 * ((size_t)y * p.W + xs))[lane] = reinterpret_cast<const float4 *>(st)[lane];
    } else if (in_x) {
      p.out_rgb[3 * q] = out[0]; p.out_rgb[3 * q + 1] = out[1]; p.out_rgb[3 * q + 2] = out[2];
    }
  }
  if (!in_x) return;
  if (p.out_argb) p.out_argb[q] = interior ? put_pixel_argb(out[0], out[1], out[2]) : 0u;
  if (p.out_depth) p.out_depth[q] = zinv_s[c0];
  if (p.out_index) {
    const int t = ORDERED ? owner[c0] : owner[c0] >> 5;              // -1 >> 5 = -1
    p.out_index[q] = (t >= 0 && p.orig) ? __ldg(p.orig + t) : t;
  }
}
