// Raytracer ray queries on sm_100a: ClosestIntersection (raytracer/Source/skeleton.cpp:263-363) for rays the
// caller supplies, the shadow test of DirectLight, `ClosestIntersection(...) && distance < r_mag` (:394-397), and
// DirectLight itself for hits the caller supplies.
//
//   rt_rays_kernel<ANY>        one thread per ray, rays in the caller's order.  Every warp streams the scene's
//                              48-byte RtGeom records through its own tile ring (rt_ring_stream in rt_tma.cuh, at
//                              warp scope), culls each tile against the box of its 32 rays and runs the
//                              reference arithmetic (rt_exact_triangle, ascending index) on the survivors, then the
//                              spheres (rt_exact_spheres).  ANY = occlusion query: a ray stops at the first pair the
//                              reference accepts below its limit, a warp leaves when its 32 rays are decided.
//   rt_rays_bruteforce_kernel  B200_OPT_RT_BRUTEFORCE = 1: the per-ray exact loop over every pair
//                              (rt_closest_bruteforce), no cull and no early exit (the on-device cross-check).
//   rt_direct_light_kernel     DirectLight (:366-415) for caller-supplied hits, one thread per (hit, light) pair: the
//                              shadow ray walks the scene like rt_rays_kernel<true> (rt_rays_walk), then the Lambert
//                              term.  rt_direct_light_bruteforce_kernel is its B200_OPT_RT_BRUTEFORCE = 1 twin.
//
// There is no spatial index: a call costs rays x triangles, minus what the cull removes.  Large scenes stream every
// record like small ones.  DESIGN.md section 3.4 has the exactness argument of the early exit and the soundness
// argument of the cull.
#include "rt_common.cuh"   // rt_count, rt_closest_bruteforce
#include "rt_exact.cuh"
#include "rt_tma.cuh"

constexpr int RT_RAYS_THREADS = 128;   // 4 warps, each with its own ring
constexpr int RT_RAYS_TILE = 64;       // records per tile
constexpr int RT_RAYS_WARPS = RT_RAYS_THREADS / 32;
// "Tame" values: finite and at most this large in magnitude.  With tame rays and records every determinant the
// reference forms is far from overflow (6 monomials of at most (2e11)^3), see the early-exit argument below.
constexpr float RT_RAYS_TAME = 1e11f;

struct RtRaysParams {
  const float4 *geom;            // ctx->rt_geom: v0, e1, e2 per triangle
  const rt_sphere *sph;
  int n_tris, n_sph;
  const rt_ray *rays;
  const float *max_distance;     // ANY only
  int n;
  rt_intersection *hits;         // closest query
  uint8_t *occluded;             // occlusion query
  unsigned long long *counters;  // [1] exact evaluations, [2] nonzero: some record is not tame (rt_rays_scene_kernel)
};

__device__ __forceinline__ bool rt_tame(float x) { return fabsf(x) <= RT_RAYS_TAME; }   // false for NaN and inf

// Whether every triangle record is tame (the early exit needs it; see rt_rays_kernel).
__global__ void rt_rays_scene_kernel(const float4 *__restrict__ geom, int n, unsigned long long *counters) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  bool wild = false;
  if (i < n) {
    const float4 g0 = geom[3 * i], g1 = geom[3 * i + 1], g2 = geom[3 * i + 2];
    wild = !(rt_tame(g0.x) && rt_tame(g0.y) && rt_tame(g0.z) && rt_tame(g0.w) && rt_tame(g1.x) && rt_tame(g1.y) &&
             rt_tame(g1.z) && rt_tame(g1.w) && rt_tame(g2.x));
  }
  if (__any_sync(0xffffffffu, wild) && (threadIdx.x & 31) == 0) atomicOr(counters + 2, 1ull);
}

// position.w = start.w + 0.0f (:326 / :345).  For a NaN start.w the reference's x86 (SSE) addition returns that NaN,
// quietened, payload kept; the GPU's FADD would return its canonical NaN instead.
__device__ __forceinline__ float rt_pos_w(float sw) {
  return sw != sw ? __uint_as_float(__float_as_uint(sw) | 0x00400000u) : xadd(sw, 0.0f);
}

// ---- directed-rounding interval arithmetic (the cull's enclosures) ---------------------------------------
struct Iv { float lo, hi; };
__device__ __forceinline__ Iv iv_add(Iv a, Iv b) { return {__fadd_rd(a.lo, b.lo), __fadd_ru(a.hi, b.hi)}; }
__device__ __forceinline__ Iv iv_sub(Iv a, Iv b) { return {__fsub_rd(a.lo, b.hi), __fsub_ru(a.hi, b.lo)}; }
__device__ __forceinline__ Iv iv_neg(Iv a) { return {-a.hi, -a.lo}; }
__device__ __forceinline__ Iv iv_mulp(Iv a, float p) {   // interval x point
  return p >= 0.0f ? Iv{__fmul_rd(a.lo, p), __fmul_ru(a.hi, p)} : Iv{__fmul_rd(a.hi, p), __fmul_ru(a.lo, p)};
}
__device__ __forceinline__ Iv iv_mul(Iv a, Iv b) {
  return {fminf(fminf(__fmul_rd(a.lo, b.lo), __fmul_rd(a.lo, b.hi)), fminf(__fmul_rd(a.hi, b.lo), __fmul_rd(a.hi, b.hi))),
          fmaxf(fmaxf(__fmul_ru(a.lo, b.lo), __fmul_ru(a.lo, b.hi)), fmaxf(__fmul_ru(a.hi, b.lo), __fmul_ru(a.hi, b.hi)))};
}
__device__ __forceinline__ Iv iv_pp(float a, float b, float c, float d) {   // a*b - c*d of points
  return {__fsub_rd(__fmul_rd(a, b), __fmul_ru(c, d)), __fsub_ru(__fmul_ru(a, b), __fmul_rd(c, d))};
}
__device__ __forceinline__ Iv iv_dot(const Iv *a, const Iv *b) {
  return iv_add(iv_add(iv_mul(a[0], b[0]), iv_mul(a[1], b[1])), iv_mul(a[2], b[2]));
}
__device__ __forceinline__ float iv_mag(Iv a) { return fmaxf(fabsf(a.lo), fabsf(a.hi)); }

// The warp's bundle: boxes of its rays' starts and directions.
struct RtBundle {
  float slo[3], shi[3], dlo[3], dhi[3];
  float dA;        // max |d| component
  bool t_cull;     // every direction has |d|inf >= 1e-6 (the distance < 0 test may be culled)
};

// True when the reference provably rejects record (g0, g1, g2) for EVERY ray of the bundle: the rounded u < 0,
// v < 0, u + v > 1 or distance < 0 of rt_exact_triangle, with the sign of D proven.  All values tame (the caller
// checks the bundle, here the record).  Soundness: DESIGN.md 3.4.
__device__ __forceinline__ bool rt_rays_cull(const RtBundle &B, float4 g0, float4 g1, float4 g2) {
  const float v0[3] = {g0.x, g0.y, g0.z}, e1[3] = {g0.w, g1.x, g1.y}, e2[3] = {g1.z, g1.w, g2.x};
  if (!(rt_tame(v0[0]) && rt_tame(v0[1]) && rt_tame(v0[2]) && rt_tame(e1[0]) && rt_tame(e1[1]) && rt_tame(e1[2]) &&
        rt_tame(e2[0]) && rt_tame(e2[1]) && rt_tame(e2[2])))
    return false;
  // s = start - v0 is rounded to nearest by the reference (:296); RN is monotone, so [RD(lo - v0), RU(hi - v0)]
  // holds every s the rays of the bundle form
  Iv s[3], d[3];
  float sA = 0.f;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    s[k] = {__fsub_rd(B.slo[k], v0[k]), __fsub_ru(B.shi[k], v0[k])};
    d[k] = {B.dlo[k], B.dhi[k]};
    sA = fmaxf(sA, iv_mag(s[k]));
  }
  const float a1 = fmaxf(fabsf(e1[0]), fmaxf(fabsf(e1[1]), fabsf(e1[2])));
  const float a2 = fmaxf(fabsf(e2[0]), fmaxf(fabsf(e2[1]), fabsf(e2[2])));
  // E: bound of |xdet3 - det| for D, Du, Dv and Dt: 6 monomials, 5 roundings each (30 u |a||b||c|, taken as 64 u),
  // plus underflow (at most 14 x 2^-150 per operation, amplified by at most 4e11)
  const float dA = B.dA;
  float E = __fmul_ru(__fmul_ru(dA, a1), a2);
  E = __fadd_ru(E, __fmul_ru(__fmul_ru(dA, sA), __fadd_ru(a1, a2)));
  E = __fadd_ru(E, __fmul_ru(__fmul_ru(sA, a1), a2));
  E = __fadd_ru(__fmul_ru(E, 64.0f * 5.9604645e-8f), 1e-29f);
  // N = e1 x e2 (the reference's D = -d.N, Dt = s.N)
  const Iv N[3] = {iv_pp(e1[1], e2[2], e1[2], e2[1]), iv_pp(e1[2], e2[0], e1[0], e2[2]), iv_pp(e1[0], e2[1], e1[1], e2[0])};
  const Iv D = iv_neg(iv_dot(d, N));
  float sg;
  if (D.lo > E) sg = 1.0f;
  else if (D.hi < -E) sg = -1.0f;
  else return false;                   // the sign of D is not proven: nothing is culled
  const float Dmax = __fadd_ru(iv_mag(D), E);   // >= |D as the reference rounds it|
  auto sgn = [&](Iv a) { return sg > 0.0f ? a : iv_neg(a); };
  // Du = -d.(s x e2), Dv = -d.(e1 x s)
  const Iv sxe2[3] = {iv_sub(iv_mulp(s[1], e2[2]), iv_mulp(s[2], e2[1])), iv_sub(iv_mulp(s[2], e2[0]), iv_mulp(s[0], e2[2])),
                      iv_sub(iv_mulp(s[0], e2[1]), iv_mulp(s[1], e2[0]))};
  const Iv Du = sgn(iv_neg(iv_dot(d, sxe2)));
  // u < 0: sigma Du_ref < 0 and |u| normal (-0 would pass u >= 0)
  if (Du.hi < -E && __fsub_rd(-Du.hi, E) > __fmul_ru(Dmax, 1e-30f)) return true;
  const Iv e1xs[3] = {iv_sub(iv_mulp(s[2], e1[1]), iv_mulp(s[1], e1[2])), iv_sub(iv_mulp(s[0], e1[2]), iv_mulp(s[2], e1[0])),
                      iv_sub(iv_mulp(s[1], e1[0]), iv_mulp(s[0], e1[1]))};
  const Iv Dv = sgn(iv_neg(iv_dot(d, e1xs)));
  if (Dv.hi < -E && __fsub_rd(-Dv.hi, E) > __fmul_ru(Dmax, 1e-30f)) return true;
  // u + v > 1: sigma (D - Du - Dv) below -(3E + |D| 2^-22)
  const Iv W = iv_sub(iv_sub(sgn(D), Du), Dv);
  if (W.hi < -__fadd_ru(__fmul_ru(3.0f, E), __fmul_ru(Dmax, 2.3841858e-7f))) return true;
  // distance < 0: t = Dt / D negative with |t| >= 1e-20, and |d| >= 1e-6 keeps t * len away from -0
  if (B.t_cull) {
    const Iv Dt = sgn(iv_dot(s, N));
    if (Dt.hi < -E && __fsub_rd(-Dt.hi, E) > __fmul_ru(Dmax, 1e-20f)) return true;
  }
  return false;
}

// The shared memory of the kernels that walk the scene: one ring of triangle records per warp.  Set up once per block by
// rt_rays_smem_init, whose barrier is the only block barrier of those kernels: from there on every warp runs on its own.
struct RtRaysSmem {
  float4 tiles[RT_RAYS_WARPS][2][RT_RAYS_TILE * RT_REC_F4];
  uint64_t bars[RT_RAYS_WARPS][2];
};

__device__ __forceinline__ void rt_rays_smem_init(RtRaysSmem &s) {
  if (threadIdx.x == 0) rt_ring_init(&s.bars[0][0], RT_RAYS_WARPS);
  __syncthreads();
}

// ClosestIntersection(start s, dir d) for one ray per thread, every thread of the block taking part, over the scene
// of p (the kernel parameters' geom, n_tris, sph, n_sph and counters): the triangle records streamed through the
// warp's ring, culled against the box of the warp's active rays, the survivors run in ascending index order, then the
// spheres.  `active` = false: the thread traces nothing.  ANY: returns DirectLight's shadow test
// `ClosestIntersection(...) && distance < maxd`, and stops at the first pair accepted below maxd when the ray and the
// scene are tame (counters[2] == 0, rt_rays_scene_kernel).  Otherwise fills `best` and returns false.  Adds the exact
// evaluations to counters[1].
template <bool ANY, class Params>
__device__ __forceinline__ bool rt_rays_walk(RtRaysSmem &S, const Params &p, float sx, float sy, float sz, float dx, float dy,
                                             float dz, float maxd, bool active, RtHit &best) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  best.t = 0.f; best.dist = FLT_MAX; best.idx = 0;
  bool occ = false;
  const float len = xsqrt(xdot3(dx, dy, dz, dx, dy, dz));   // glm::length(dir3), :307
  const float dinf = fmaxf(fabsf(dx), fmaxf(fabsf(dy), fabsf(dz)));
  // Early exit (ANY) needs a tame ray (1e-18 <= |d|inf, so len > 0) and a tame scene: then no pair can leave a NaN
  // distance behind, and the reference's final distance is the minimum over the pairs it accepts.
  const bool ray_tame = rt_tame(sx) && rt_tame(sy) && rt_tame(sz) && dinf <= RT_RAYS_TAME && dinf >= 1e-18f;
  const bool may_exit = ANY && ray_tame && p.counters[2] == 0;
  unsigned long long n_exact = 0;

  // the bundle box of the warp's active rays; the cull runs only when all of them are tame
  RtBundle B;
  const bool cull = __all_sync(0xffffffffu, !active || ray_tame);
  {
    const float s3[3] = {sx, sy, sz}, d3[3] = {dx, dy, dz};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      B.slo[k] = warp_min(active ? s3[k] : INFINITY); B.shi[k] = warp_max(active ? s3[k] : -INFINITY);
      B.dlo[k] = warp_min(active ? d3[k] : INFINITY); B.dhi[k] = warp_max(active ? d3[k] : -INFINITY);
    }
    B.dA = fmaxf(fmaxf(fmaxf(-B.dlo[0], B.dhi[0]), fmaxf(-B.dlo[1], B.dhi[1])), fmaxf(-B.dlo[2], B.dhi[2]));
    B.t_cull = warp_min(active ? dinf : INFINITY) >= 1e-6f;
  }

  bool warp_busy = __any_sync(0xffffffffu, active);
  RtRing ring = rt_ring<RT_RAYS_TILE>(&S.tiles[warp][0][0], nullptr, S.bars[warp]);
  const int n_tiles = warp_busy ? (p.n_tris + RT_RAYS_TILE - 1) / RT_RAYS_TILE : 0;
  int k = 0;
  auto next = [&](RtItem &it) {   // the scene's records in order
    if (k >= n_tiles) return false;
    it.rec = p.geom + (size_t)k * RT_RAYS_TILE * RT_REC_F4; it.idx = nullptr;
    it.base = k * RT_RAYS_TILE; it.cnt = min(RT_RAYS_TILE, p.n_tris - it.base);
    ++k;
    return true;
  };
  rt_ring_stream<true, RT_RAYS_TILE>(ring, lane == 0, next, [&](const float4 *T, const int *, int base, int cnt) {
    for (int r0 = 0; r0 < cnt && warp_busy; r0 += 32) {
      // cull: one record per lane against the whole bundle
      bool keep = false;
      if (r0 + lane < cnt) {
        keep = true;
        if (cull) {
          const float4 *q = T + (size_t)(r0 + lane) * 3;
          keep = !rt_rays_cull(B, q[0], q[1], q[2]);
        }
      }
      unsigned mask = __ballot_sync(0xffffffffu, keep);
      while (mask) {
        const int j = __ffs(mask) - 1;
        mask &= mask - 1;
        if (active) {
          const float4 *q = T + (size_t)(r0 + j) * 3;
          rt_exact_triangle(sx, sy, sz, dx, dy, dz, len, q[0], q[1], q[2], base + r0 + j, best);
          ++n_exact;
          // an accepted pair (best.dist < FLT_MAX) below the limit; a limit of +inf must not count the start value
          if (ANY && may_exit && best.dist < FLT_MAX && best.dist < maxd) { occ = true; active = false; }
        }
      }
      if (ANY) warp_busy = __any_sync(0xffffffffu, active);
    }
    return !ANY || warp_busy;   // only the occlusion query leaves early
  });
  if (active) rt_exact_spheres(p.sph, p.n_sph, sx, sy, sz, dx, dy, dz, best);   // :341-355
  rt_count(p.counters + 1, n_exact);
  return ANY && (occ || (active && best.dist < FLT_MAX && best.dist < maxd));   // :395-397
}

template <bool ANY>
__global__ void __launch_bounds__(RT_RAYS_THREADS) rt_rays_kernel(const __grid_constant__ RtRaysParams p) {
  __shared__ __align__(128) RtRaysSmem S;
  rt_rays_smem_init(S);
  const int i = blockIdx.x * RT_RAYS_THREADS + threadIdx.x;
  const bool live = i < p.n;
  float sx = 0.f, sy = 0.f, sz = 0.f, sw = 0.f, dx = 0.f, dy = 0.f, dz = 0.f, maxd = 0.f;
  if (live) {
    const rt_ray *r = p.rays + i;   // (4-byte alignment is all a caller's device pointer promises)
    sx = __ldg(&r->start[0]); sy = __ldg(&r->start[1]); sz = __ldg(&r->start[2]); sw = __ldg(&r->start[3]);
    dx = __ldg(&r->dir[0]); dy = __ldg(&r->dir[1]); dz = __ldg(&r->dir[2]);
    if (ANY) maxd = p.max_distance[i];
  }
  RtHit best;
  // ANY: a NaN or non-positive limit answers 0 without a test
  const bool occ = rt_rays_walk<ANY>(S, p, sx, sy, sz, dx, dy, dz, maxd, live && (!ANY || maxd > 0.0f), best);
  if (!live) return;
  if (ANY) {
    p.occluded[i] = occ ? 1 : 0;
  } else {
    rt_intersection o;
    o.distance = best.dist;
    if (best.dist < FLT_MAX) {
      // position = start + vec4(t * dir3, 0)   (:326 / :345)
      o.position[0] = xadd(sx, xmul(best.t, dx)); o.position[1] = xadd(sy, xmul(best.t, dy));
      o.position[2] = xadd(sz, xmul(best.t, dz)); o.position[3] = rt_pos_w(sw);
      o.triangle_index = best.idx >= 0 ? best.idx : -1;
      o.sphere_index = best.idx >= 0 ? -1 : -1 - best.idx;
    } else {
      o.position[0] = o.position[1] = o.position[2] = o.position[3] = 0.f;
      o.triangle_index = o.sphere_index = -1;
    }
    p.hits[i] = o;
  }
}

template <bool ANY>
__global__ void __launch_bounds__(128) rt_rays_bruteforce_kernel(const __grid_constant__ RtRaysParams p, const __grid_constant__ RtKParams k) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < p.n) {
    const rt_ray r = p.rays[i];
    const float sx = r.start[0], sy = r.start[1], sz = r.start[2], dx = r.dir[0], dy = r.dir[1], dz = r.dir[2];
    const RtHit best = rt_closest_bruteforce(k, sx, sy, sz, dx, dy, dz);
    const bool hit = best.dist < FLT_MAX;
    if (ANY) {
      p.occluded[i] = (hit && best.dist < p.max_distance[i]) ? 1 : 0;
    } else {
      rt_intersection o;
      o.distance = best.dist;
      if (hit) {
        o.position[0] = xadd(sx, xmul(best.t, dx)); o.position[1] = xadd(sy, xmul(best.t, dy));
        o.position[2] = xadd(sz, xmul(best.t, dz)); o.position[3] = rt_pos_w(r.start[3]);
        o.triangle_index = best.idx >= 0 ? best.idx : -1;
        o.sphere_index = best.idx >= 0 ? -1 : -1 - best.idx;
      } else {
        o.position[0] = o.position[1] = o.position[2] = o.position[3] = 0.f;
        o.triangle_index = o.sphere_index = -1;
      }
      p.hits[i] = o;
    }
  }
  rt_count(p.counters + 1, i < p.n ? (unsigned long long)p.n_tris : 0ull);
}

// ---- DirectLight (skeleton.cpp:366-415) for caller-supplied hits: one thread per (hit, light) pair ---------------
struct RtDirectParams {
  const float4 *geom;            // ctx->rt_geom: v0, e1, e2 per triangle
  const rt_triangle *src;        // colour and normal
  const rt_sphere *sph;
  int n_tris, n_sph;
  const rt_intersection *hits;
  int n, n_lights;
  float lights[B200_MAX_LIGHTS][7];   // pos[4], colour[3]
  float *power;                  // [(i * n_lights + l) * 3 + c]
  unsigned long long *counters;  // [0] shadow rays, [1] exact evaluations, [2] nonzero: some record is not tame
};

// What DirectLight forms before its shadow test (:370-394) for entry i and light L.  `named` = false: the entry
// names no primitive (a miss record, an index out of range) and the pair is not traced.
struct RtShadowRay {
  bool named;
  float cr, cg, cb, nx, ny, nz;   // colour and normal (rt_surface2)
  float rx, ry, rz, r_mag;    // r = light - p (:370), r_mag (:371)
  float ox, oy, oz;           // the start p + 1e-5 n (:394)
};

__device__ __forceinline__ RtShadowRay rt_shadow_ray(const RtDirectParams &p, int i, const float *L) {
  RtShadowRay s;
  s.named = false;
  float col[3] = {0.f, 0.f, 0.f};
  s.nx = s.ny = s.nz = 0.f;
  float px = 0.f, py = 0.f, pz = 0.f;
  int idx = 0;
  if (i < p.n) {
    const rt_intersection *h = p.hits + i;   // (4-byte alignment is all a caller's device pointer promises)
    const int ti = __ldg(&h->triangle_index), si = __ldg(&h->sphere_index);
    // `if (triangleIndex != -1)` (:377): that triangle, otherwise that sphere
    s.named = ti != -1 ? (ti >= 0 && ti < p.n_tris) : (si >= 0 && si < p.n_sph);
    idx = ti != -1 ? ti : -1 - si;
    px = __ldg(&h->position[0]); py = __ldg(&h->position[1]); pz = __ldg(&h->position[2]);
  }
  if (s.named) rt_surface2(p.src, p.sph, idx, px, py, pz, col, s.nx, s.ny, s.nz);
  s.cr = col[0]; s.cg = col[1]; s.cb = col[2];
  s.rx = xsub(L[0], px); s.ry = xsub(L[1], py); s.rz = xsub(L[2], pz);
  s.r_mag = rt_exact_rmag(s.rx, s.ry, s.rz);
  s.ox = xadd(px, xmul(s.nx, 0.00001f)); s.oy = xadd(py, xmul(s.ny, 0.00001f)); s.oz = xadd(pz, xmul(s.nz, 0.00001f));
  return s;
}

// The Lambert term of a clear shadow ray (:400-412), 0 for an occluded or unnamed pair.  Every NaN is stored as the
// x86 indefinite NaN (x86_nan): from NaN-free inputs each one begins as an invalid operation (DESIGN.md 3.4).  Not
// inlined, and it forms the pair's inputs again: nothing of them stays live through the walk.
__device__ __noinline__ void rt_store_power(const RtDirectParams &p, int i, int l, bool occ) {
  const float *L = p.lights[l];
  const RtShadowRay s = rt_shadow_ray(p, i, L);
  float pw[3] = {0.f, 0.f, 0.f};
  const float col[3] = {s.cr, s.cg, s.cb};
  if (s.named && !occ) rt_exact_lambert(s.rx, s.ry, s.rz, s.r_mag, s.nx, s.ny, s.nz, col, L + 4, pw);
  float *o = p.power + ((size_t)i * p.n_lights + l) * 3;
  o[0] = x86_nan(pw[0]); o[1] = x86_nan(pw[1]); o[2] = x86_nan(pw[2]);
}

// blockIdx.y = the light: the 32 shadow rays of a warp share their end point and start on neighbouring hits, which
// is what the cull of rt_rays_walk needs.
__global__ void __launch_bounds__(RT_RAYS_THREADS) rt_direct_light_kernel(const __grid_constant__ RtDirectParams p) {
  __shared__ __align__(128) RtRaysSmem S;
  rt_rays_smem_init(S);
  const int i = blockIdx.x * RT_RAYS_THREADS + threadIdx.x, l = blockIdx.y;
  const float *L = p.lights[l];
  const RtShadowRay s = rt_shadow_ray(p, i, L);
  RtHit best;
  // a NaN or zero r_mag: no distance lies below it (:395), nothing to test
  const bool occ = rt_rays_walk<true>(S, p, s.ox, s.oy, s.oz, s.rx, s.ry, s.rz, s.r_mag, s.named && s.r_mag > 0.0f, best);
  rt_count(p.counters + 0, s.named ? 1ull : 0ull);
  if (i < p.n) rt_store_power(p, i, l, occ);
}

__global__ void __launch_bounds__(128) rt_direct_light_bruteforce_kernel(const __grid_constant__ RtDirectParams p,
                                                                         const __grid_constant__ RtKParams k) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, l = blockIdx.y;
  const float *L = p.lights[l];
  const RtShadowRay s = rt_shadow_ray(p, i, L);
  bool occ = false;
  if (s.named) {
    const RtHit best = rt_closest_bruteforce(k, s.ox, s.oy, s.oz, s.rx, s.ry, s.rz);
    occ = best.dist < FLT_MAX && best.dist < s.r_mag;   // :394-397
  }
  rt_count(p.counters + 0, s.named ? 1ull : 0ull);
  rt_count(p.counters + 1, s.named ? (unsigned long long)p.n_tris : 0ull);
  if (i < p.n) rt_store_power(p, i, l, occ);
}

// The scene flag the occlusion walk's early exit reads (counters[2]).
static int rt_launch_scene_flag(b200_ctx *ctx, const float4 *geom, int n_tris, unsigned long long *counters) {
  if (n_tris == 0) return B200_OK;
  rt_rays_scene_kernel<<<(n_tris + 255) / 256, 256, 0, ctx->stream>>>(geom, n_tris, counters);
  tl_mark(ctx, "rt_rays_scene_kernel");
  ctx->stats.kernel_launches++;
  CU_CHECK(ctx, cudaGetLastError());
  return B200_OK;
}

// Enqueues one query on ctx->stream: d_hits (closest) or d_occ with d_max (occlusion); n > 0.
int rt_launch_rays(b200_ctx *ctx, const rt_ray *d_rays, const float *d_max, int n, rt_intersection *d_hits, uint8_t *d_occ) {
  RtRaysParams p;
  memset(&p, 0, sizeof p);
  p.geom = (const float4 *)ctx->rt_geom.p;
  p.sph = (const rt_sphere *)ctx->rt_spheres.p;
  p.n_tris = ctx->rt_n_tris; p.n_sph = ctx->rt_n_spheres;
  p.rays = d_rays; p.max_distance = d_max; p.n = n;
  p.hits = d_hits; p.occluded = d_occ;
  p.counters = (unsigned long long *)ctx->counters.p;
  const bool any = d_occ != nullptr;
  if (ctx->opt_rt_bruteforce) {
    RtKParams k;   // the scene fields rt_closest_bruteforce reads
    memset(&k, 0, sizeof k);
    k.geom = p.geom; k.sph = p.sph; k.n_tris = p.n_tris; k.n_sph = p.n_sph;
    const unsigned blocks = (unsigned)((n + 127) / 128);
    if (any) rt_rays_bruteforce_kernel<true><<<blocks, 128, 0, ctx->stream>>>(p, k);
    else rt_rays_bruteforce_kernel<false><<<blocks, 128, 0, ctx->stream>>>(p, k);
    tl_mark(ctx, "rt_rays_bruteforce_kernel");
    ctx->stats.kernel_launches++;
    CU_CHECK(ctx, cudaGetLastError());
    return B200_OK;
  }
  if (any) if (int rc = rt_launch_scene_flag(ctx, p.geom, p.n_tris, p.counters)) return rc;
  const unsigned blocks = (unsigned)((n + RT_RAYS_THREADS - 1) / RT_RAYS_THREADS);
  if (any) rt_rays_kernel<true><<<blocks, RT_RAYS_THREADS, 0, ctx->stream>>>(p);
  else rt_rays_kernel<false><<<blocks, RT_RAYS_THREADS, 0, ctx->stream>>>(p);
  tl_mark(ctx, "rt_rays_kernel");
  ctx->stats.kernel_launches++;
  CU_CHECK(ctx, cudaGetLastError());
  return B200_OK;
}

int rt_launch_direct_light(b200_ctx *ctx, const rt_intersection *d_hits, int n, const light_t *lights, int n_lights,
                           float *d_power) {
  RtDirectParams p;
  memset(&p, 0, sizeof p);
  p.geom = (const float4 *)ctx->rt_geom.p;
  p.src = (const rt_triangle *)ctx->rt_src.p;
  p.sph = (const rt_sphere *)ctx->rt_spheres.p;
  p.n_tris = ctx->rt_n_tris; p.n_sph = ctx->rt_n_spheres;
  p.hits = d_hits; p.n = n; p.n_lights = n_lights;
  for (int l = 0; l < n_lights; ++l) {
    memcpy(&p.lights[l][0], lights[l].pos, 4 * sizeof(float));
    memcpy(&p.lights[l][4], lights[l].colour, 3 * sizeof(float));
  }
  p.power = d_power;
  p.counters = (unsigned long long *)ctx->counters.p;
  const dim3 grid((unsigned)((n + RT_RAYS_THREADS - 1) / RT_RAYS_THREADS), (unsigned)n_lights);
  if (ctx->opt_rt_bruteforce) {
    RtKParams k;   // the scene fields rt_closest_bruteforce reads
    memset(&k, 0, sizeof k);
    k.geom = p.geom; k.sph = p.sph; k.n_tris = p.n_tris; k.n_sph = p.n_sph;
    rt_direct_light_bruteforce_kernel<<<grid, RT_RAYS_THREADS, 0, ctx->stream>>>(p, k);
    tl_mark(ctx, "rt_direct_light_bruteforce_kernel");
    ctx->stats.kernel_launches++;
    CU_CHECK(ctx, cudaGetLastError());
    return B200_OK;
  }
  if (int rc = rt_launch_scene_flag(ctx, p.geom, p.n_tris, p.counters)) return rc;
  rt_direct_light_kernel<<<grid, RT_RAYS_THREADS, 0, ctx->stream>>>(p);
  tl_mark(ctx, "rt_direct_light_kernel");
  ctx->stats.kernel_launches++;
  CU_CHECK(ctx, cudaGetLastError());
  return B200_OK;
}
