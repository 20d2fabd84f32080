/* oracle_rast_geom.c -- CPU restatement of the reference rasteriser's geometry
 * stage (the part of Draw before the triangle loop, rasteriser/Source/
 * skeleton.cpp:205-241): toCameraSpace :701-716, createShadowVolume :1676-1722,
 * rotation :223-228, toClipSpace :691-699 and the six-plane clip :720-1673.
 *
 * TEST INFRASTRUCTURE ONLY (see oracle_rast.c).  Parity status: PINNED --
 * tests/test_oracle_rast.py compares the clipped list byte-for-byte with the one
 * the unmodified reference builds (oracle/_ref), on the Cornell box at several
 * camera poses/yaws and on random scenes, and with the committed goldens.
 *
 * The reference spells the clip out as 6 planes x 7 hand-copied cases.  They all
 * instantiate one pattern, restated here once, with the reference's two slips in
 * the far plane kept (:1607 tests v2.x instead of v2.w; :1615 divides by
 * (w1 - w0) instead of (w1 - w2)).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct {
  float v[3][4];
  float normal[4], color[3];
  int32_t texture, index;
} g_tri; /* 84 B */

static void compute_normal(g_tri *t) { /* rasteriser/Source/TestModelH.h:32-41 */
  float e1[3], e2[3];
  for (int k = 0; k < 3; ++k) { e1[k] = t->v[1][k] - t->v[0][k]; e2[k] = t->v[2][k] - t->v[0][k]; }
  float c[3] = {e2[1] * e1[2] - e1[1] * e2[2], e2[2] * e1[0] - e1[2] * e2[0], e2[0] * e1[1] - e1[0] * e2[1]};
  float inv = 1.0f / sqrtf((c[0] * c[0] + c[1] * c[1]) + c[2] * c[2]);
  t->normal[0] = c[0] * inv; t->normal[1] = c[1] * inv; t->normal[2] = c[2] * inv; t->normal[3] = 1.0f;
}

/* glm mat4 * vec4 (glm/glm/detail/type_mat4x4.inl:640-652), column-major R */
static void mat_vec(const float *R, float *v) {
  float o[4];
  for (int r = 0; r < 4; ++r) o[r] = (R[0 + r] * v[0] + R[4 + r] * v[1]) + (R[8 + r] * v[2] + R[12 + r] * v[3]);
  memcpy(v, o, sizeof o);
}

/* a + t * (b - a) on vec4 */
static void lerp4(const float *a, const float *b, float t, float *o) {
  for (int k = 0; k < 4; ++k) o[k] = a[k] + t * (b[k] - a[k]);
}

/* Clip census: how often each branch of clip_one was taken since the last reset, so that tests can
 * check which cases their scenes reach.  Counting only; the arithmetic is untouched.  Layout (the
 * indices oracle_rast_clip_census copies out):
 *   CEN_BRANCH + 8 * i + k   plane i = 0..4 for planes 1, 2, 3, 4, 6; k = 0 all in, 1 only v0 in,
 *                            2 only v1, 3 only v2, 4 v0 and v1, 5 v0 and v2, 6 v1 and v2, 7 all out
 *   CEN_FAR_REFUSED          far plane, v0 and v2 in but v2.x > 5 / f (:1607): dropped
 *   CEN_NEAR_KEPT / _DROPPED plane 5 (:1497-1505)
 *   CEN_NAN                  dropped because a vertex is neither inside nor outside (NaN)
 *   CEN_ZERO_DEN             intersection parameters whose denominator is exactly 0 (t = +-inf or NaN; odd W or H
 *                            make one possible on planes 1-4, whose t uses the truncated W / 2, H / 2)
 *   CEN_ON_LIMIT + p - 1     vertices exactly on plane p's limit (x or y == the bound, z == 0.01,
 *                            w == 5 / f), each time a triangle meets that plane
 *   CEN_DESC + n             pre-clip triangles with n descendants in the final list (0..32) */
enum { CEN_BRANCH = 0, CEN_FAR_REFUSED = 40, CEN_NEAR_KEPT, CEN_NEAR_DROPPED, CEN_NAN, CEN_ZERO_DEN, CEN_ON_LIMIT,
       CEN_DESC = CEN_ON_LIMIT + 6, CEN_N = CEN_DESC + 33 };
static long long census[CEN_N];

/* Copies min(cap, CEN_N) counters to out (when not NULL), clears them when reset != 0 and returns
 * CEN_N. */
int oracle_rast_clip_census(long long *out, int cap, int reset) {
  if (out) memcpy(out, census, (size_t)(cap < CEN_N ? cap : CEN_N) * sizeof(long long));
  if (reset) memset(census, 0, sizeof census);
  return CEN_N;
}

typedef struct { int plane, W, H; float focal; } clip_ctx;

static int inside(const clip_ctx *c, const float *v) {
  switch (c->plane) {
    case 1: return v[0] > (v[3] * (float)(-c->W)) / 2.0f;   /* :732, :737 */
    case 2: return v[0] < (v[3] * (float)(c->W)) / 2.0f;    /* :922, :927 */
    case 3: return v[1] < (v[3] * (float)(c->H)) / 2.0f;    /* :1115 */
    case 4: return v[1] > (v[3] * (float)(-c->H)) / 2.0f;   /* :1307 */
    default: return v[3] <= 5.0f / c->focal;                /* :1509-1512 */
  }
}
static int outside(const clip_ctx *c, const float *v) {
  switch (c->plane) {
    case 1: return v[0] <= (v[3] * (float)(-c->W)) / 2.0f;
    case 2: return v[0] >= (v[3] * (float)(c->W)) / 2.0f;
    case 3: return v[1] >= (v[3] * (float)(c->H)) / 2.0f;
    case 4: return v[1] <= (v[3] * (float)(-c->H)) / 2.0f;
    default: return v[3] > 5.0f / c->focal;
  }
}

/* num / den, counting an exactly zero denominator */
static float t_div(float num, float den) {
  census[CEN_ZERO_DEN] += den == 0.0f;
  return num / den;
}

/* intersection parameter along a (inside) -> b (outside) */
static float t_param(const clip_ctx *c, const float *a, const float *b) {
  switch (c->plane) {
    case 1: { float h = (float)(c->W / 2), nh = (float)((-c->W) / 2);   /* :753 */
      return t_div(a[0] + h * a[3], ((nh * b[3] + h * a[3]) - b[0]) + a[0]); }
    case 2: { float h = (float)(c->W / 2);                               /* :943 */
      return t_div(a[0] - h * a[3], ((h * b[3] - h * a[3]) - b[0]) + a[0]); }
    case 3: { float h = (float)(c->H / 2);                               /* :1136 */
      return t_div(a[1] - h * a[3], ((h * b[3] - h * a[3]) - b[1]) + a[1]); }
    case 4: { float h = (float)(c->H / 2), nh = (float)((-c->H) / 2);   /* :1328 */
      return t_div(a[1] + h * a[3], ((nh * b[3] + h * a[3]) - b[1]) + a[1]); }
    default: { float wl = 5.0f / c->focal;                               /* :1524 */
      return t_div(wl - a[3], b[3] - a[3]); }
  }
}

/* a vertex exactly on the plane's limit */
static int on_limit(const clip_ctx *c, const float *v) {
  switch (c->plane) {
    case 1: return v[0] == (v[3] * (float)(-c->W)) / 2.0f;
    case 2: return v[0] == (v[3] * (float)(c->W)) / 2.0f;
    case 3: return v[1] == (v[3] * (float)(c->H)) / 2.0f;
    case 4: return v[1] == (v[3] * (float)(-c->H)) / 2.0f;
    case 5: return v[2] == 0.01f;
    default: return v[3] == 5.0f / c->focal;
  }
}

/* One triangle through one plane (0, 1 or 2 results appended to out). */
static int clip_one(const clip_ctx *c, const g_tri *in, g_tri *out) {
  for (int k = 0; k < 3; ++k) census[CEN_ON_LIMIT + c->plane - 1] += on_limit(c, in->v[k]);
  if (c->plane == 5) {                                                   /* :1497-1505 */
    if (in->v[0][2] > 0.01f && in->v[1][2] > 0.01f && in->v[2][2] > 0.01f) {
      census[CEN_NEAR_KEPT]++; out[0] = *in; return 1;
    }
    census[CEN_NEAR_DROPPED]++;
    return 0;
  }
  const int i0 = inside(c, in->v[0]), i1 = inside(c, in->v[1]), i2 = inside(c, in->v[2]);
  const int o0 = outside(c, in->v[0]), o1 = outside(c, in->v[1]), o2 = outside(c, in->v[2]);
  long long *br = census + CEN_BRANCH + 8 * (c->plane == 6 ? 4 : c->plane - 1);
  g_tri t = *in;
  if (i0 && i1 && i2) { br[0]++; out[0] = t; return 1; }
  if (i0 && o1 && o2) {                                                  /* only v0 in */
    br[1]++;
    float t01 = t_param(c, t.v[0], t.v[1]), t02 = t_param(c, t.v[0], t.v[2]);
    lerp4(in->v[0], in->v[1], t01, t.v[1]);
    lerp4(in->v[0], in->v[2], t02, t.v[2]);
    out[0] = t; return 1;
  }
  if (o0 && i1 && o2) {                                                  /* only v1 in */
    br[2]++;
    float t10 = t_param(c, t.v[1], t.v[0]), t12 = t_param(c, t.v[1], t.v[2]);
    lerp4(in->v[1], in->v[0], t10, t.v[0]);
    lerp4(in->v[1], in->v[2], t12, t.v[2]);
    out[0] = t; return 1;
  }
  if (o0 && o1 && i2) {                                                  /* only v2 in */
    br[3]++;
    float t21 = t_param(c, t.v[2], t.v[1]), t20 = t_param(c, t.v[2], t.v[0]);
    lerp4(in->v[2], in->v[1], t21, t.v[1]);
    lerp4(in->v[2], in->v[0], t20, t.v[0]);
    out[0] = t; return 1;
  }
  g_tri extra = *in;   /* keeps the parent's normal / colour / texture / index (:838-841) */
  if (i0 && i1 && o2) {                                                  /* v0, v1 in */
    br[4]++;
    float t12 = t_param(c, in->v[1], in->v[2]), t02 = t_param(c, in->v[0], in->v[2]);
    float np12[4], np02[4];
    lerp4(in->v[1], in->v[2], t12, np12);
    lerp4(in->v[0], in->v[2], t02, np02);
    memcpy(t.v[2], np02, 16);
    memcpy(extra.v[0], np02, 16); memcpy(extra.v[1], np12, 16); memcpy(extra.v[2], in->v[1], 16);
    out[0] = t; out[1] = extra; return 2;
  }
  /* v0, v2 in: the far plane's version of this test reads v2.x (:1607) */
  int c02 = c->plane == 6 ? (i0 && o1 && in->v[2][0] <= 5.0f / c->focal) : (i0 && o1 && i2);
  if (c02) {
    br[5]++;
    float t01 = t_param(c, in->v[0], in->v[1]);
    float t21 = c->plane == 6 ? (5.0f / c->focal - in->v[2][3]) / (in->v[1][3] - in->v[0][3])   /* :1615 */
                              : t_param(c, in->v[2], in->v[1]);
    float np01[4], np21[4];
    lerp4(in->v[0], in->v[1], t01, np01);
    lerp4(in->v[2], in->v[1], t21, np21);
    memcpy(t.v[1], np01, 16);
    memcpy(extra.v[0], np01, 16); memcpy(extra.v[1], np21, 16); memcpy(extra.v[2], in->v[2], 16);
    out[0] = t; out[1] = extra; return 2;
  }
  if (o0 && i1 && i2) {                                                  /* v1, v2 in */
    br[6]++;
    float t10 = t_param(c, in->v[1], in->v[0]), t20 = t_param(c, in->v[2], in->v[0]);
    float np10[4], np20[4];
    lerp4(in->v[1], in->v[0], t10, np10);
    lerp4(in->v[2], in->v[0], t20, np20);
    memcpy(t.v[0], np10, 16);
    memcpy(extra.v[0], np10, 16); memcpy(extra.v[1], np20, 16); memcpy(extra.v[2], in->v[2], 16);
    out[0] = t; out[1] = extra; return 2;
  }
  if (o0 && o1 && o2) br[7]++;
  else if (i0 && o1 && i2) census[CEN_FAR_REFUSED]++;
  else census[CEN_NAN]++;
  return 0;   /* NaNs, or the far plane's unmatched combination: dropped */
}

/* Draw :205-241.  Returns the number of clipped triangles (or -1 when out_cap is
 * too small); light_cam4 receives the camera-space, rotated lightPos. */
int oracle_rast_geometry(int W, int H, float focal, const float *cam, const float *R,
                         const float *light_pos4, const void *room_, int n_room, const void *boxes_,
                         int n_boxes, void *out_, int out_cap, float *light_cam4) {
  const g_tri *room = (const g_tri *)room_, *boxes = (const g_tri *)boxes_;
  g_tri *out = (g_tri *)out_;
  float lp[4] = {light_pos4[0] - cam[0], light_pos4[1] - cam[1], light_pos4[2] - cam[2], 1.0f};  /* :211-212 */
  float lpr[4];
  memcpy(lpr, lp, sizeof lp);
  mat_vec(R, lpr);                                                                               /* :223 */
  if (light_cam4) memcpy(light_cam4, lpr, sizeof lpr);
  const int n_pre = n_room + 7 * n_boxes;
  int n_out = 0;
  g_tri cur[64], nxt[64];
  for (int j = 0; j < n_pre; ++j) {
    g_tri t;
    if (j < n_room) {
      t = room[j];
      for (int k = 0; k < 3; ++k) { for (int c = 0; c < 3; ++c) t.v[k][c] = t.v[k][c] - cam[c]; t.v[k][3] = 1.0f; }
    } else {
      const int b = (j - n_room) / 7, s = (j - n_room) % 7;
      g_tri o = boxes[b];
      for (int k = 0; k < 3; ++k) { for (int c = 0; c < 3; ++c) o.v[k][c] = o.v[k][c] - cam[c]; o.v[k][3] = 1.0f; }
      if (s == 0) t = o;
      else {
        /* createShadowVolume :1695-1710: far vertices n = (v - light) * 100 */
        float n[3][4];
        for (int k = 0; k < 3; ++k) for (int c = 0; c < 4; ++c) n[k][c] = (o.v[k][c] - lp[c]) * 100.0f;
        const float *vs[6][3] = {{o.v[0], n[0], o.v[1]}, {n[0], o.v[1], n[1]}, {o.v[1], n[1], o.v[2]},
                                 {n[1], o.v[2], n[2]}, {o.v[2], n[2], o.v[0]}, {n[2], o.v[0], n[0]}};
        memset(&t, 0, sizeof t);
        for (int k = 0; k < 3; ++k) memcpy(t.v[k], vs[s - 1][k], 16);
        t.color[0] = t.color[1] = t.color[2] = -1.0f;
        t.texture = 0;
        t.index = 0;   /* uninitialised in the reference; never read for texture 0 */
        compute_normal(&t);
      }
    }
    for (int k = 0; k < 3; ++k) mat_vec(R, t.v[k]);                        /* :224-228 */
    for (int k = 0; k < 3; ++k) t.v[k][3] = t.v[k][2] / focal;             /* :695-697 */
    int n_cur = 1;
    cur[0] = t;
    for (int plane = 1; plane <= 6; ++plane) {                             /* :236-241 */
      clip_ctx c = {plane, W, H, focal};
      int n_nxt = 0;
      for (int i = 0; i < n_cur; ++i) n_nxt += clip_one(&c, &cur[i], &nxt[n_nxt]);
      memcpy(cur, nxt, (size_t)n_nxt * sizeof(g_tri));
      n_cur = n_nxt;
    }
    census[CEN_DESC + n_cur]++;
    if (n_out + n_cur > out_cap) return -1;
    memcpy(out + n_out, cur, (size_t)n_cur * sizeof(g_tri));
    n_out += n_cur;
  }
  return n_out;
}
