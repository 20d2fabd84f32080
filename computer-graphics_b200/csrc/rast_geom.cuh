// Device helpers of the rasteriser's geometry stage (rasteriser/Source/skeleton.cpp:205-241):
// toCameraSpace :701-716, createShadowVolume :1676-1722, rotation :223-228, toClipSpace
// :691-699 and the six-plane clip :720-1673.  Shared by the list-building kernels
// (rast_geom.cu) and the fused scatter / resolve kernels (rast_fast.cuh), which run the same
// code per triangle instead of reading a clipped list back from HBM.
#pragma once
#include "common.cuh"

// What the per-triangle transform needs of the camera and the light.
struct GeomXform {
  int W, H;
  float focal;
  float cam[4];
  float R[16];
  float light_cam[4];   // sceneCoordinatesLightPos - cameraPos, w = 1 (before rotation)
};

struct GV { float x, y, z, w; };
struct GTri { GV v[3]; };

__device__ __forceinline__ GV gv_lerp(const GV &a, const GV &b, float t) {   // a + t * (b - a)
  GV o;
  o.x = xadd(a.x, xmul(t, xsub(b.x, a.x)));
  o.y = xadd(a.y, xmul(t, xsub(b.y, a.y)));
  o.z = xadd(a.z, xmul(t, xsub(b.z, a.z)));
  o.w = xadd(a.w, xmul(t, xsub(b.w, a.w)));
  return o;
}

// glm mat4 * vec4 (glm/glm/detail/type_mat4x4.inl:640-652)
__device__ __forceinline__ GV gv_rotate(const float *R, const GV &v) {
  GV o;
  o.x = xadd(xadd(xmul(R[0], v.x), xmul(R[4], v.y)), xadd(xmul(R[8], v.z), xmul(R[12], v.w)));
  o.y = xadd(xadd(xmul(R[1], v.x), xmul(R[5], v.y)), xadd(xmul(R[9], v.z), xmul(R[13], v.w)));
  o.z = xadd(xadd(xmul(R[2], v.x), xmul(R[6], v.y)), xadd(xmul(R[10], v.z), xmul(R[14], v.w)));
  o.w = xadd(xadd(xmul(R[3], v.x), xmul(R[7], v.y)), xadd(xmul(R[11], v.z), xmul(R[15], v.w)));
  return o;
}

struct ClipCtx { int plane, W, H; float focal, wfar; };   // wfar = 5 / focal, the far limit of w (:1509)

__device__ __forceinline__ float clip_coord(const ClipCtx &c, const GV &v) {
  return c.plane <= 2 ? v.x : (c.plane <= 4 ? v.y : v.w);
}
// the plane's limit for this vertex: `dot[k]` (:732, :922, :1115, :1307) or wlimit (:1509)
__device__ __forceinline__ float clip_limit(const ClipCtx &c, const GV &v) {
  switch (c.plane) {
    // x / 2 == x * 0.5f bit for bit for every float (a power-of-two scale is exact; the one rounding
    // at the bottom of the denormal range is the same real number rounded the same way)
    case 1: return xmul(xmul(v.w, (float)(-c.W)), 0.5f);
    case 2: return xmul(xmul(v.w, (float)(c.W)), 0.5f);
    case 3: return xmul(xmul(v.w, (float)(c.H)), 0.5f);
    case 4: return xmul(xmul(v.w, (float)(-c.H)), 0.5f);
    default: return c.wfar;
  }
}
__device__ __forceinline__ bool clip_in(const ClipCtx &c, const GV &v) {
  const float a = clip_coord(c, v), l = clip_limit(c, v);
  return (c.plane == 1 || c.plane == 4) ? a > l : (c.plane == 6 ? a <= l : a < l);
}
__device__ __forceinline__ bool clip_out(const ClipCtx &c, const GV &v) {
  const float a = clip_coord(c, v), l = clip_limit(c, v);
  return (c.plane == 1 || c.plane == 4) ? a <= l : (c.plane == 6 ? a > l : a >= l);
}
// intersection parameter along a (inside) -> b (outside), e.g. t_01 at :753 / :943 / :1524
__device__ __forceinline__ float clip_t(const ClipCtx &c, const GV &a, const GV &b) {
  if (c.plane == 6) return xdiv(xsub(c.wfar, a.w), xsub(b.w, a.w));
  const int S = c.plane <= 2 ? c.W : c.H;
  const float h = (float)(S / 2), nh = (float)((-S) / 2);
  const float ca = c.plane <= 2 ? a.x : a.y, cb = c.plane <= 2 ? b.x : b.y;
  if (c.plane == 1 || c.plane == 4)
    return xdiv(xadd(ca, xmul(h, a.w)), xadd(xsub(xadd(xmul(nh, b.w), xmul(h, a.w)), cb), ca));
  return xdiv(xsub(ca, xmul(h, a.w)), xadd(xsub(xsub(xmul(h, b.w), xmul(h, a.w)), cb), ca));
}

// One triangle through one plane: 0, 1 or 2 results.
__device__ __forceinline__ int clip_one(const ClipCtx &c, const GTri &in, GTri &o0, GTri &o1) {
  const GV &a = in.v[0], &b = in.v[1], &d = in.v[2];
  if (c.plane == 5) {                                           // :1497-1505: dropped, never split
    if (a.z > 0.01f && b.z > 0.01f && d.z > 0.01f) { o0 = in; return 1; }
    return 0;
  }
  const bool i0 = clip_in(c, a), i1 = clip_in(c, b), i2 = clip_in(c, d);
  const bool x0 = clip_out(c, a), x1 = clip_out(c, b), x2 = clip_out(c, d);
  o0 = in;
  if (i0 && i1 && i2) return 1;
  if (i0 && x1 && x2) { o0.v[1] = gv_lerp(a, b, clip_t(c, a, b)); o0.v[2] = gv_lerp(a, d, clip_t(c, a, d)); return 1; }
  if (x0 && i1 && x2) { o0.v[0] = gv_lerp(b, a, clip_t(c, b, a)); o0.v[2] = gv_lerp(b, d, clip_t(c, b, d)); return 1; }
  if (x0 && x1 && i2) { o0.v[1] = gv_lerp(d, b, clip_t(c, d, b)); o0.v[0] = gv_lerp(d, a, clip_t(c, d, a)); return 1; }
  if (i0 && i1 && x2) {                                         // :814-846
    const GV np12 = gv_lerp(b, d, clip_t(c, b, d)), np02 = gv_lerp(a, d, clip_t(c, a, d));
    o0.v[2] = np02;
    o1.v[0] = np02; o1.v[1] = np12; o1.v[2] = b;
    return 2;
  }
  const bool c02 = c.plane == 6 ? (i0 && x1 && d.x <= c.wfar) : (i0 && x1 && i2);   // :1607
  if (c02) {                                                    // :849-881
    const float t01 = clip_t(c, a, b);
    const float t21 = c.plane == 6 ? xdiv(xsub(c.wfar, d.w), xsub(b.w, a.w))        // :1615
                                   : clip_t(c, d, b);
    const GV np01 = gv_lerp(a, b, t01), np21 = gv_lerp(d, b, t21);
    o0.v[1] = np01;
    o1.v[0] = np01; o1.v[1] = np21; o1.v[2] = d;
    return 2;
  }
  if (x0 && i1 && i2) {                                         // :883-916
    const GV np10 = gv_lerp(b, a, clip_t(c, b, a)), np20 = gv_lerp(d, a, clip_t(c, d, a));
    o0.v[0] = np10;
    o1.v[0] = np10; o1.v[1] = np20; o1.v[2] = d;
    return 2;
  }
  return 0;   // NaNs, or the far plane's unmatched combination: dropped
}

// The general case: the triangle's descendants through the six planes, in the
// reference's list order.  cur[0] holds the input; returns the count.
static __device__ __noinline__ int clip_six_planes(int W, int H, float focal, GTri *cur) {
  GTri nxt[32];
  int n_cur = 1;
  const float wfar = xdiv(5.0f, focal);
  for (int plane = 1; plane <= 6; ++plane) {
    ClipCtx c;
    c.plane = plane; c.W = W; c.H = H; c.focal = focal; c.wfar = wfar;
    int n_nxt = 0;
    for (int i = 0; i < n_cur; ++i) {
      GTri o0, o1;
      const int m = clip_one(c, cur[i], o0, o1);
      if (m >= 1) nxt[n_nxt++] = o0;
      if (m == 2) nxt[n_nxt++] = o1;
    }
    for (int i = 0; i < n_nxt; ++i) cur[i] = nxt[i];
    n_cur = n_nxt;
    if (n_cur == 0) break;
  }
  return n_cur;
}

// The pre-clip triangle (Draw :205-228, :691-699): `src` is a room triangle (s == 0) or a box
// triangle whose shadow-volume side s - 1 (0..5) is wanted (createShadowVolume :1695-1710);
// camera space, rotated, w = z / focal.  attr: normal[4], color[3], texture, index (bit-cast).
__device__ __forceinline__ void geom_preclip(const GeomXform &p, const rast_triangle *srcp, int s, GTri &t, float *attr) {
  GV o[3];
  const float *vin[3] = {srcp->v0, srcp->v1, srcp->v2};
#pragma unroll
  for (int k = 0; k < 3; ++k) {                                // toCameraSpace :701-711
    o[k].x = xsub(vin[k][0], p.cam[0]); o[k].y = xsub(vin[k][1], p.cam[1]); o[k].z = xsub(vin[k][2], p.cam[2]);
    o[k].w = 1.0f;
  }
  if (s == 0) {
    t.v[0] = o[0]; t.v[1] = o[1]; t.v[2] = o[2];
#pragma unroll
    for (int k = 0; k < 4; ++k) attr[k] = srcp->normal[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) attr[4 + k] = srcp->color[k];
    attr[7] = __int_as_float(srcp->texture);
    attr[8] = __int_as_float(srcp->index);
  } else {
    GV n[3];                                                   // createShadowVolume :1695-1697
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      n[k].x = xmul(xsub(o[k].x, p.light_cam[0]), 100.0f);
      n[k].y = xmul(xsub(o[k].y, p.light_cam[1]), 100.0f);
      n[k].z = xmul(xsub(o[k].z, p.light_cam[2]), 100.0f);
      n[k].w = xmul(xsub(o[k].w, p.light_cam[3]), 100.0f);
    }
    const int e = (s - 1) >> 1, e1 = (e + 1) % 3;              // :1705-1710
    if ((s - 1) & 1) { t.v[0] = n[e]; t.v[1] = o[e1]; t.v[2] = n[e1]; }
    else { t.v[0] = o[e]; t.v[1] = n[e]; t.v[2] = o[e1]; }
    // Triangle::ComputeNormal (rasteriser/Source/TestModelH.h:32-41)
    const float ax = xsub(t.v[1].x, t.v[0].x), ay = xsub(t.v[1].y, t.v[0].y), az = xsub(t.v[1].z, t.v[0].z);
    const float bx = xsub(t.v[2].x, t.v[0].x), by = xsub(t.v[2].y, t.v[0].y), bz = xsub(t.v[2].z, t.v[0].z);
    const float cx = xsub(xmul(by, az), xmul(ay, bz)), cy = xsub(xmul(bz, ax), xmul(az, bx)),
                cz = xsub(xmul(bx, ay), xmul(ax, by));
    const float inv = xdiv(1.0f, xsqrt(xdot3(cx, cy, cz, cx, cy, cz)));
    attr[0] = xmul(cx, inv); attr[1] = xmul(cy, inv); attr[2] = xmul(cz, inv); attr[3] = 1.0f;
    attr[4] = attr[5] = attr[6] = -1.0f;
    attr[7] = __int_as_float(0);
    attr[8] = __int_as_float(0);   // uninitialised in the reference; never read for texture 0
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    t.v[k] = gv_rotate(p.R, t.v[k]);                           // :224-228
    t.v[k].w = xdiv(t.v[k].z, p.focal);                        // :695-697
  }
}

// NaN bits of the clipped list (DESIGN §4.1).  The reference's geometry runs on x86, where an invalid operation
// (0 * inf, inf - inf, 0 / 0) yields the indefinite NaN 0xffc00000 and later operations pass it on unchanged; here
// it yields 0x7fffffff.  With finite scene inputs every NaN the stage computes begins as such an operation (a
// caller's NaN or inf vertex is dropped by the clip before it can reach the list), so the list writers store every
// computed NaN -- vertices and shadow-volume normals, not attributes copied from the caller -- as 0xffc00000
// (x86_nan, common.cuh).

// A triangle inside all six planes comes out of the clip unchanged (one descendant).
__device__ __forceinline__ bool geom_all_in(const GeomXform &p, const GTri &t) {
  bool all_in = true;
  const float wfar = xdiv(5.0f, p.focal);
#pragma unroll
  for (int plane = 1; plane <= 6; ++plane) {
    ClipCtx c;
    c.plane = plane; c.W = p.W; c.H = p.H; c.focal = p.focal; c.wfar = wfar;
    if (plane == 5) all_in = all_in && t.v[0].z > 0.01f && t.v[1].z > 0.01f && t.v[2].z > 0.01f;
    else all_in = all_in && clip_in(c, t.v[0]) && clip_in(c, t.v[1]) && clip_in(c, t.v[2]);
  }
  return all_in;
}
