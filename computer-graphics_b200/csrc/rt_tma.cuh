// mbarrier / TMA bulk-copy primitives, the double-buffered tile ring every raytracer scene walk streams its records
// through (rt_filtered_kernel.cuh, rt_lattice_kernel.cuh, rt_rays.cu), its streaming loop (rt_rays.cu), and warp
// reductions (also rt_grid.cuh).
#pragma once
#include <stdint.h>

// ---- mbarrier / TMA bulk-copy primitives (sm_90+/sm_100a PTX) ------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
// 1-D bulk copy global -> shared, completion signalled on the mbarrier.
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ---- the tile ring ------------------------------------------------------------------
// Two shared-memory buffers of TILE records (48 bytes each), refilled by 1-D TMA bulk copies while the threads work on
// the other one.  A ring belongs to a block (block scope: __syncthreads before a refill) or to one warp (warp scope:
// __syncwarp).  One thread of its scope, the issuer, issues every copy.
//
// A refill overwrites, through the async proxy, a buffer the threads have just read through the generic proxy.  The
// barrier orders those reads before the issuer's copy; the PTX memory model also asks for a cross-proxy fence between
// them, which rt_ring_stream's issuer runs before every copy into a buffer that has been read (rt_ring_fence).
constexpr int RT_REC_F4 = 3;   // float4s per record

// One tile of work: up to TILE consecutive records of a list.
struct RtItem {
  const float4 *rec;
  const int *idx;    // null: record i is triangle base + i; else idx[i] is (copied into the ring with the records)
  int base, cnt;
};

struct RtRing {
  float4 *buf[2];    // TILE records each (a tile is a select of the two: an offset from one base spilled more)
  int *smem_idx;     // 2 x TILE triangle indices, for lists with an index (RtItem::idx)
  uint64_t *bars;    // one mbarrier per buffer
  uint32_t phase_bits;
  int issued;        // tiles waited on so far: the next copy goes to buffer issued & 1
};

// Sets up the mbarriers of n rings (bars[2 n]).  One thread runs it, before a block barrier.
__device__ __forceinline__ void rt_ring_init(uint64_t *bars, int n) {
  for (int i = 0; i < 2 * n; ++i) mbar_init(&bars[i], 1);
  mbar_fence_init();
}

template <int TILE>
__device__ __forceinline__ RtRing rt_ring(float4 *smem, int *smem_idx, uint64_t *bars) {
  RtRing r;
  r.buf[0] = smem; r.buf[1] = smem + TILE * RT_REC_F4; r.smem_idx = smem_idx; r.bars = bars; r.phase_bits = 0; r.issued = 0;
  return r;
}

// Orders the scope's generic-proxy reads of a buffer, made before the barrier the issuer has just passed, before the
// async-proxy write of the copy that refills it.
__device__ __forceinline__ void rt_ring_fence() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

template <int TILE>
__device__ __forceinline__ void rt_ring_issue(RtRing &ring, const RtItem &it) {
  const int buf = ring.issued & 1;
  const uint32_t rec_bytes = (uint32_t)it.cnt * 48u, idx_bytes = it.idx ? (((uint32_t)it.cnt + 3u) & ~3u) * 4u : 0u;
  mbar_expect_tx(&ring.bars[buf], rec_bytes + idx_bytes);
  tma_bulk_g2s(ring.buf[0] + (size_t)buf * TILE * RT_REC_F4, it.rec, rec_bytes, &ring.bars[buf]);
  if (it.idx) tma_bulk_g2s(ring.smem_idx + buf * TILE, it.idx, idx_bytes, &ring.bars[buf]);
}

// Streams the tiles next(RtItem &) -> bool hands out through the ring, each one prefetched while the one before it is
// worked on: body(T, Tidx, base, cnt) -> bool gets the tile's records T[0 .. 3 cnt) of item base and, for an item
// with an index list (RtItem::idx), its triangle indices Tidx[0 .. cnt).  Every thread of the scope calls it with the same items.  body returning false ends
// the walk (uniformly over the scope); the tile still in flight is waited for first, so that no copy outlives it.
// The caller's barrier must separate this walk from an earlier one on the same ring: the first copy refills the buffer
// the earlier walk read last but one.
template <bool WARP_SCOPE, int TILE, class Next, class Body>
__device__ __forceinline__ void rt_ring_stream(RtRing &ring, bool issuer, Next &&next, Body &&body) {
  RtItem item;
  bool have = next(item);
  if (issuer && have) {
    if (ring.issued > 0) rt_ring_fence();   // an earlier walk read the buffer
    rt_ring_issue<TILE>(ring, item);
  }
  while (have) {
    const int buf = ring.issued & 1;
    ++ring.issued;
    if (WARP_SCOPE) __syncwarp(); else __syncthreads();   // every thread is done with the other buffer: refill it
    RtItem next_item;
    const bool have_next = next(next_item);
    if (issuer && have_next) {
      rt_ring_fence();
      rt_ring_issue<TILE>(ring, next_item);
    }
    mbar_wait(&ring.bars[buf], (ring.phase_bits >> buf) & 1u);
    ring.phase_bits ^= 1u << buf;
    // (the current item is read, and replaced by the next, before the body: with both live through it the
    // lattice kernel spilled more)
    const int *Tidx = ring.smem_idx + buf * TILE;
    const int base = item.base, cnt = item.cnt;
    item = next_item;
    have = have_next;
    if (!body(buf ? ring.buf[1] : ring.buf[0], Tidx, base, cnt)) {
      if (have) {   // drain before leaving
        mbar_wait(&ring.bars[buf ^ 1], (ring.phase_bits >> (buf ^ 1)) & 1u);
        ring.phase_bits ^= 1u << (buf ^ 1);
        ++ring.issued;
      }
      return;
    }
  }
}

// ---- warp helpers -------------------------------------------------------------------
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
