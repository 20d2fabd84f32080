// Production raytracer kernel: brute force over every (ray, triangle) pair, but
// almost every pair is decided by a conservative edge-function filter; the
// reference arithmetic (rt_exact.cuh) runs only where its outcome can matter.
// The frame is bit-identical to rt_bruteforce_kernel and to the reference.
//
// Why this is legitimate.  ClosestIntersection (raytracer/Source/skeleton.cpp:
// 263-363) keeps the hit with the smallest `distance`, lowest index on ties; a
// triangle that fails `check` (:328) or `distance < 0` (:311) never changes its
// state.  So any pair that PROVABLY fails one of those tests in the reference's
// own float arithmetic can be skipped, and any pair that PROVABLY passes `check`
// needs only the t/distance part.  All primary rays share the camera origin and
// all shadow rays of one light end at that light, so per (origin, triangle) the
// three Cramer numerators are linear in the ray direction d:
//     sigma*Du = d.PU   sigma*Dv = d.PV   sigma*(D-Du-Dv) = d.PW      (planes)
// with sigma the sign that t >= 0 forces on det(A).  A pair is a definite miss
// when one of the three is below -E, a definite inside when all are above +E,
// where E bounds (reference rounding error + filter rounding error); see
// rt_prep_planes_kernel for the bound.  Pairs in the +-E band run the reference
// arithmetic unchanged.
//
// Hierarchy (per warp = 8x4 pixel patch, 9 samples per pixel):
//   L0  each LANE tests a different triangle's planes against the bounding box
//       of the whole warp's ray bundle; __ballot_sync gives the survivors
//       (warp vote early-out: 32 triangles x 288 rays per ~20 instructions);
//   L1  for each survivor, each lane tests its pixel's 9-ray bundle box;
//   L2  per ray: the three plane values decide miss / inside / ambiguous;
//   EX  reference arithmetic for what is left (about two per ray).
// Plane records are streamed through shared memory in tiles by 1-D TMA bulk
// copies (cp.async.bulk + mbarrier), double buffered.
#pragma once
#include "rt_common.cuh"
#include "rt_exact.cuh"
#include "rt_tma.cuh"

constexpr int RT_TILE = 256;      // triangles per shared-memory tile
constexpr int RT_THREADS = 256;   // 8 warps: a 16x16 pixel block
constexpr int RT_REC_F4 = 3;      // float4s per plane record (48 bytes)
// direction grids (rt_grid.cuh)
constexpr int RT_GRID_G = 64;              // light cube map: cells per face edge
constexpr int RT_GRID_FACE = RT_GRID_G * RT_GRID_G;
constexpr int RT_WTILE = 64;               // records per tile of a warp's private ring (grid kernels)
constexpr int RT_GRID_MAX_CELLS = 96;      // shadow phase: distinct cells one warp (8x4 pixels, 288 rays) may walk, else it streams the scene
constexpr int RT_GRID_TABLE_LOG2 = 8;      // hash set used to collect them
constexpr int RT_SEEN_LOG2 = 8, RT_SEEN = 1 << RT_SEEN_LOG2;   // per-warp set of triangles already met in this light phase

// ---- per-frame plane records ------------------------------------------------------
// origin 0 = camera (directions (dx, dy, f): the z term is folded into a constant)
// origin 1+l = light l (directions g = hit - light, general 3-D)   (batched views: see RtPrepViews)
//   q0 = (Ux, Uy, Uz|cU, Vx)  q1 = (Vy, Vz|cV, Wx, Wy)  q2 = (Wz|cW, E, T0, T1)
// camera: E absolute (max |d| folded in), T0 = lower bound of |Dt|, T1 = E + 0.5*max(|Px|+|Py|)
// light : E per unit |g|_inf, T0/T1 = reject / definite thresholds of d.PN (t >= 0 test)
struct RtPrepParams {
  const float4 *geom;
  int n_tris;
  float cam[3];
  float focal;
  float dmax;        // upper bound of |d|_inf over the frame's primary rays
  float world_S;     // upper bound of |start - v0|_inf for any ray start in the scene
  float n_scale;     // max(1, max |normal component|): the shadow-ray start is hit + 1e-5 * normal (:394)
  int n_lights;
  float lights[B200_MAX_LIGHTS][3];
  float4 *planes;    // [(1 + n_lights)][n_tiles * RT_TILE][3]
  size_t origin_stride_f4;
  float *dt_cam;     // [n_tris] det(start - v0, e1, e2) for start = camera, in the reference's own arithmetic
  // [n_lights][n_tris] for a shadow ray that starts on the triangle (a hit point p): the sign of the
  // reference's D = det(-(L - p), e1, e2) times an upper bound of |D| below 1e30, or 0 where not known.
  // Null for frames that go to the grid kernels, which do not use it.
  float *self_D;
};

// Batched views (one launch renders up to RT_VIEWS_MAX whole frames of one scene and one set of lights):
// origin v < n_views is view v's camera, origin n_views + l is light l.  Each view has its own camera
// records and dt_cam[v][n_tris]; the light records and self_D are shared.  Kernel parameters, indexed by
// blockIdx.y (preparation) / blockIdx.z (render).
constexpr int RT_VIEWS_MAX = 64;
struct RtPrepViews {
  int n_views;
  float cam_inf;                 // max over the views of |cam|inf: C of the self_D bound (see below)
  float cam[RT_VIEWS_MAX][4];    // position, focal
  float dmax[RT_VIEWS_MAX];
};
struct RtViewsParams {
  int n_views;
  struct { float cam[3]; float focal; float R[16]; } view[RT_VIEWS_MAX];
};

template <bool VIEWS>
__device__ __forceinline__ void rt_prep_planes_body(const RtPrepParams &p, const RtPrepViews *pv) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int o = blockIdx.y;  // origin
  if (i >= p.n_tris) return;
  const bool is_cam = VIEWS ? o < pv->n_views : o == 0;
  const int l = VIEWS ? o - pv->n_views : o - 1;   // light of a light origin
  const float *cam = VIEWS ? pv->cam[is_cam ? o : 0] : p.cam;
  const float focal = VIEWS ? cam[3] : p.focal;
  const float dmax = VIEWS ? pv->dmax[is_cam ? o : 0] : p.dmax;
  const float4 g0 = p.geom[3 * i], g1 = p.geom[3 * i + 1], g2 = p.geom[3 * i + 2];
  const double e1[3] = {g0.w, g1.x, g1.y}, e2[3] = {g1.z, g1.w, g2.x};
  const float v0[3] = {g0.x, g0.y, g0.z};
  double s[3];
  if (is_cam) {
    // exactly the reference's `start - v0` (skeleton.cpp:296)
    for (int k = 0; k < 3; ++k) s[k] = (double)xsub(cam[k], v0[k]);
  } else {
    for (int k = 0; k < 3; ++k) s[k] = (double)p.lights[l][k] - (double)v0[k];
  }
  const double N[3] = {e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2],
                       e1[0] * e2[1] - e1[1] * e2[0]};
  const double Dt = s[0] * N[0] + s[1] * N[1] + s[2] * N[2];
  const double sg = Dt < 0 ? -1.0 : 1.0;
  // PU = -sg (s x e2), PV = -sg (e1 x s), PN = -sg (e1 x e2), PW = PN - PU - PV
  double PU[3] = {-sg * (s[1] * e2[2] - s[2] * e2[1]), -sg * (s[2] * e2[0] - s[0] * e2[2]),
                  -sg * (s[0] * e2[1] - s[1] * e2[0])};
  double PV[3] = {-sg * (e1[1] * s[2] - e1[2] * s[1]), -sg * (e1[2] * s[0] - e1[0] * s[2]),
                  -sg * (e1[0] * s[1] - e1[1] * s[0])};
  double PW[3];
  for (int k = 0; k < 3; ++k) PW[k] = -sg * N[k] - PU[k] - PV[k];

  const double eps = 5.9604644775390625e-08;  // 2^-24
  const double a1 = fmax(fabs(e1[0]), fmax(fabs(e1[1]), fabs(e1[2])));
  const double a2 = fmax(fabs(e2[0]), fmax(fabs(e2[1]), fabs(e2[2])));
  const double N1 = fabs(N[0]) + fabs(N[1]) + fabs(N[2]);
  const double N2 = sqrt(N[0] * N[0] + N[1] * N[1] + N[2] * N[2]);
  float4 q0, q1, q2;
  bool degenerate = !(isfinite(Dt) && isfinite(N1) && a1 < 1e18 && a2 < 1e18);
  if (is_cam) {
    const double sm = fmax(fabs(s[0]), fmax(fabs(s[1]), fabs(s[2])));
    // Rounding-error bound of the reference's three determinants plus this
    // filter's own (planes rounded to float, FMA chains): each is below
    // 54 eps |d|inf X Y; 256 leaves a wide safety factor.
    const double E = 256.0 * eps * (a1 * a2 + sm * (a1 + a2)) * (double)dmax * 1.01;
    const double dt_lo = fabs(Dt) * (1.0 - 1e-6) - 256.0 * eps * sm * a1 * a2;
    if (!(dt_lo > 0.0)) degenerate = true;   // camera (numerically) in the triangle's plane
    const double f = (double)focal;
    const double h = 0.5 * fmax(fabs(PU[0]) + fabs(PU[1]), fmax(fabs(PV[0]) + fabs(PV[1]), fabs(PW[0]) + fabs(PW[1])));
    q0 = make_float4((float)PU[0], (float)PU[1], (float)(PU[2] * f), (float)PV[0]);
    q1 = make_float4((float)PV[1], (float)(PV[2] * f), (float)PW[0], (float)PW[1]);
    q2 = make_float4((float)(PW[2] * f), __double2float_ru(E), __double2float_rd(dt_lo),
                     __double2float_ru((E + h) * (1.0 + 1e-6)));
  } else {
    const double S = (double)p.world_S;
    const double ns = (double)p.n_scale;
    const double E = 256.0 * eps * (a1 * a2 + S * (a1 + a2)) + 6.2e-5 * ns * (a1 + a2);
    const double slackT = 256.0 * eps * S * a1 * a2 + 1.01e-5 * ns * N1 + 1e-6 * fabs(Dt);
    // light closer than 1e-3 S to the plane: the "beyond the light" argument
    // loses its margin, leave the triangle to the reference arithmetic
    if (!(fabs(Dt) > 1e-3 * S * N2) || !(fabs(Dt) - slackT > 0.0)) degenerate = true;
    // Shadow rays from a hit p on this triangle: D = -(L - p).N up to the rounding of r = L - p and of
    // xdet3 (together below 36 eps S a1 a2), and (L - p).N = Dt - (p - v0).N.  p = cam + t d in the
    // reference's arithmetic, off the plane by the errors of t's two determinants and of the products and
    // sums that form p: |(p - v0).N| < 80 eps (C + S) a1 a2, C = |cam|inf, assuming |t d| and |p| below
    // C + S / 2 (|cam - v0| is): hit points within the scene, the assumption world_S already makes for slackT
    // (not proven for a ray that grazes the triangle).  256 eps (C + 2S) a1 a2 covers both with a factor
    // two; outside that band sign(D) = -sign(Dt) and |D| < |Dt| + B.  rt_ex_shadow's guards on r.r hold
    // too: |Dt| > 2B and |Dt| > 1e-3 S N2 keep |r| above 5e-4 S (S >= 1e-3), and |r|inf <= S < 1e14.
    // Batched views share these records: C is the largest |cam|inf of the launch's views, which only
    // widens B, so the bound holds for the hit points of every view.
    const double C = VIEWS ? (double)pv->cam_inf
                           : fmax(fabs((double)p.cam[0]), fmax(fabs((double)p.cam[1]), fabs((double)p.cam[2])));
    const double B = 256.0 * eps * (C + 2.0 * S) * a1 * a2 + 1e-6 * fabs(Dt);
    const bool known = !degenerate && fabs(Dt) > 2.0 * B && fabs(Dt) + B < 1e29 && S < 1e14;
    const float dhi = __double2float_ru((fabs(Dt) + B) * (1.0 + 1e-6));
    if (p.self_D) p.self_D[(size_t)l * p.n_tris + i] = !known ? 0.0f : (Dt > 0.0 ? -dhi : dhi);
    q0 = make_float4((float)PU[0], (float)PU[1], (float)PU[2], (float)PV[0]);
    q1 = make_float4((float)PV[1], (float)PV[2], (float)PW[0], (float)PW[1]);
    q2 = make_float4((float)PW[2], __double2float_ru(E), __double2float_rd(fabs(Dt) - slackT),
                     __double2float_ru(fabs(Dt) + slackT));
  }
  if (degenerate || !isfinite(q0.x + q0.y + q0.z + q0.w + q1.x + q1.y + q1.z + q1.w + q2.x)) {
    // always "ambiguous": every ray runs the reference arithmetic on this triangle
    q0 = make_float4(0.f, 0.f, 0.f, 0.f);
    q1 = make_float4(0.f, 0.f, 0.f, 0.f);
    q2 = make_float4(0.f, INFINITY, -INFINITY, INFINITY);
  }
  float4 *dst = p.planes + (size_t)o * p.origin_stride_f4 + (size_t)i * RT_REC_F4;
  dst[0] = q0; dst[1] = q1; dst[2] = q2;
  if (is_cam) {
    // numerator of t (skeleton.cpp:305-306): the same for every primary ray, exact float ops
    const float sx = xsub(cam[0], v0[0]), sy = xsub(cam[1], v0[1]), sz = xsub(cam[2], v0[2]);
    p.dt_cam[(VIEWS ? (size_t)o * p.n_tris : 0) + i] = xdet3(sx, sy, sz, g0.w, g1.x, g1.y, g1.z, g1.w, g2.x);
  }
}

__global__ void rt_prep_planes_kernel(const __grid_constant__ RtPrepParams p) { rt_prep_planes_body<false>(p, nullptr); }
// p.cam / p.focal / p.dmax unused: per view in v
__global__ void rt_prep_planes_views_kernel(const __grid_constant__ RtPrepParams p, const __grid_constant__ RtPrepViews v) {
  rt_prep_planes_body<true>(p, &v);
}

// ---- bundle-box tests shared by the render kernel (L0) and the grid builder -------
// A triangle can matter to a ray only if all three edge values are >= -E there.  Over a
// box of directions (centre c, half-widths h >= 0) each edge value is linear, so its
// maximum is known exactly; the same holds for the sums of two and of all three, which
// must then be >= -2E / -3E.  The sums catch what the single planes cannot: triangles
// seen nearly edge-on, whose two long edge planes almost coincide and straddle the box.
// (Coefficient sums are rounded once more; the factors leave room for that.)
// PAIRS = false (small scenes streamed whole, where a few extra L0 survivors cost less than
// the test) checks the single planes only.
template <bool PAIRS = true>
__device__ __forceinline__ bool rt_box_may_hit_light(const float4 q0, const float4 q1, const float4 q2, const float *c,
                                                     const float *h, float Eg) {
  const float U[3] = {q0.x, q0.y, q0.z}, V[3] = {q0.w, q1.x, q1.y}, W[3] = {q1.z, q1.w, q2.x};
  auto hi = [&](float x, float y, float z) {
    return fmaf(x, c[0], fmaf(y, c[1], z * c[2])) + fmaf(fabsf(x), h[0], fmaf(fabsf(y), h[1], fabsf(z) * h[2]));
  };
  if (fminf(fminf(hi(U[0], U[1], U[2]), hi(V[0], V[1], V[2])), hi(W[0], W[1], W[2])) < -Eg) return false;
  if (!PAIRS) return true;
  const float uv = hi(U[0] + V[0], U[1] + V[1], U[2] + V[2]);
  const float vw = hi(V[0] + W[0], V[1] + W[1], V[2] + W[2]);
  const float uw = hi(U[0] + W[0], U[1] + W[1], U[2] + W[2]);
  if (fminf(fminf(uv, vw), uw) < -2.1f * Eg) return false;
  return true;
}
// camera: directions (dx, dy, f) with the z term folded into the constant; E absolute
template <bool PAIRS = true>
__device__ __forceinline__ bool rt_box_may_hit_cam(const float4 q0, const float4 q1, const float4 q2, float c0, float c1,
                                                   float h0, float h1) {
  auto hi = [&](float x, float y, float k) {
    return fmaf(x, c0, fmaf(y, c1, k)) + fmaf(fabsf(x), h0, fabsf(y) * h1);
  };
  const float E = q2.y;
  if (fminf(fminf(hi(q0.x, q0.y, q0.z), hi(q0.w, q1.x, q1.y)), hi(q1.z, q1.w, q2.x)) < -E) return false;
  if (!PAIRS) return true;
  const float uv = hi(q0.x + q0.w, q0.y + q1.x, q0.z + q1.y);
  const float vw = hi(q0.w + q1.z, q1.x + q1.w, q1.y + q2.x);
  const float uw = hi(q0.x + q1.z, q0.y + q1.w, q0.z + q2.x);
  if (fminf(fminf(uv, vw), uw) < -2.1f * E) return false;
  return true;
}

#include "rt_filtered_kernel.cuh"
