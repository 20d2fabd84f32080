"""World-space scenes for the rasteriser's geometry stage (tests/test_rast_clip_gpu.py) that aim pre-clip triangles at
chosen branches of the six-plane clip (Draw :205-241, restated in oracle/oracle_rast_geom.c).

Most cases are built in camera space -- camera at the origin, R the identity, so that world and camera coordinates
are the same floats -- which lets a vertex sit exactly on a plane's limit.  The rotated cases place camera-space
triangles through the inverse of their camera transform (a yaw, pitch and roll, and a translation column in R);
there the float32 round trip moves vertices by an ulp or so, which does not matter for what they are for.
`CASES` lists them; `oracle_census` runs the oracle's geometry stage over them and reads back which branches were
taken (oracle_rast_clip_census).  Nothing here loads the product library.
"""
import ctypes

import numpy as np

import helpers as h

f32 = np.float32
FRAMES = {"64x48": (64, 48, 36.0), "320x240": (320, 240, 170.0), "37x23": (37, 23, 20.0),
          "32768x48": (32768, 48, 16384.0)}
GEOM_WARP_MAX_PRE = 8192            # rast_geom.cu: pipelined frames up to this many pre-clip triangles take a warp each
FAST_PIPE_BYTES = 16 << 20          # rast_upload_scene: shadow-free scenes this large travel in chunks
NONE = np.zeros(0, h.RAST_TRI)

# ---- oracle_rast_clip_census layout (oracle/oracle_rast_geom.c) ----------------------------------
CLIP_PLANES = (1, 2, 3, 4, 6)
BRANCHES = ("all in", "only v0 in", "only v1 in", "only v2 in", "v0 v1 in", "v0 v2 in", "v1 v2 in", "all out")
CEN_FAR_REFUSED, CEN_NEAR_KEPT, CEN_NEAR_DROPPED, CEN_NAN, CEN_ZERO_DEN, CEN_ON_LIMIT = 40, 41, 42, 43, 44, 45
CEN_DESC = CEN_ON_LIMIT + 6
CEN_N = CEN_DESC + 33


def census_read(reset=True):
    """{name: count} of the oracle's clip census (and the descendant histogram under "descendants")."""
    raw = np.zeros(CEN_N, np.int64)
    assert h.oracle().oracle_rast_clip_census(h.ptr(raw), ctypes.c_int(CEN_N), ctypes.c_int(1 if reset else 0)) == CEN_N
    out = {}
    for i, p in enumerate(CLIP_PLANES):
        for k, b in enumerate(BRANCHES):
            out[f"plane {p}: {b}"] = int(raw[8 * i + k])
    out["plane 6: v0 v2 in refused (v2.x > 5 / f)"] = int(raw[CEN_FAR_REFUSED])
    out["plane 5: kept"] = int(raw[CEN_NEAR_KEPT])
    out["plane 5: dropped"] = int(raw[CEN_NEAR_DROPPED])
    out["NaN dropped"] = int(raw[CEN_NAN])
    out["t_param denominator exactly 0"] = int(raw[CEN_ZERO_DEN])
    for p in range(1, 7):
        out[f"plane {p}: vertex on the limit"] = int(raw[CEN_ON_LIMIT + p - 1])
    return out, raw[CEN_DESC:].copy()


# ---- building blocks (camera space unless stated) -----------------------------------------------
def tris_from(P, color=None, rng=None):
    """(n, 3, 3) vertex positions -> RAST_TRI with w = 1, the given or random colours and computed normals."""
    P = np.asarray(P, f32).reshape(-1, 3, 3)
    t = np.zeros(len(P), h.RAST_TRI)
    for k, name in enumerate(("v0", "v1", "v2")):
        t[name][:, :3] = P[:, k]
        t[name][:, 3] = 1.0
    if color is None:
        rng = rng or np.random.default_rng(0)
        color = rng.uniform(0.15, 0.75, (len(P), 3))
    t["color"] = np.asarray(color, f32)
    with np.errstate(all="ignore"):
        h.compute_normals(t)
    return t


def fuzz(rng, n, zlo=-1.0, zhi=9.0):
    """Triangles of every size around the view volume: behind the camera, across the near, side and far planes."""
    s = (10 ** rng.uniform(-1, 1.5, (n, 1, 1))).astype(f32)
    P = rng.uniform(-1, 1, (n, 3, 3)).astype(f32) * s
    P[:, :, 2] = rng.uniform(zlo, zhi, (n, 3))
    return tris_from(P, rng=rng)


def box_tris(rng, n, near=0.3, far=3.0, size=0.6):
    """Box triangles in front of the camera (each becomes itself and six shadow-volume sides)."""
    c = np.stack([rng.uniform(-0.8, 0.8, n), rng.uniform(-0.6, 0.6, n), rng.uniform(near, far, n)], 1)
    P = c[:, None, :] + rng.uniform(-size, size, (n, 3, 3))
    return tris_from(P, rng=rng)


def closed_box(lo, hi, rng):
    """The 12 triangles of an axis-aligned box."""
    x0, y0, z0 = lo
    x1, y1, z1 = hi
    c = [(x, y, z) for x in (x0, x1) for y in (y0, y1) for z in (z0, z1)]
    quads = [(0, 1, 3, 2), (4, 6, 7, 5), (0, 4, 5, 1), (2, 3, 7, 6), (0, 2, 6, 4), (1, 5, 7, 3)]
    P = []
    for a, b, cc, d in quads:
        P += [(c[a], c[b], c[cc]), (c[a], c[cc], c[d])]
    return tris_from(P, rng=rng)


def on_limits(W, H, f):
    """Triangles with a vertex exactly on the limit of each plane: x = (w * -W) / 2 and the rest as the oracle
    computes them, z = 0.01, and z = 5 (w = 5 / f)."""
    F = f32(f)
    P = []
    for z in (f32(1.0), f32(2.5), f32(4.0)):
        w = z / F
        lim = {1: (w * f32(-W)) / f32(2), 2: (w * f32(W)) / f32(2), 3: (w * f32(H)) / f32(2), 4: (w * f32(-H)) / f32(2)}
        for p, l in lim.items():
            ax = 0 if p <= 2 else 1
            inward = f32(-1) if p in (2, 3) else f32(1)
            on = [f32(0), f32(0), z]
            on[ax] = l
            for other in ((0.3, 0.2), (-0.3, 0.4), (3.0, -0.2)):     # inside, inside, outside along the axis
                a = [f32(0.1), f32(0.1), z]
                b = [f32(-0.1), f32(0.2), z + f32(0.5)]
                a[ax] = l + inward * f32(other[0])
                b[ax] = l + inward * f32(other[1])
                P += [(on, a, b), (a, on, b), (a, b, on)]
    for zn, zo in ((f32(0.01), f32(1.0)), (f32(5.0), f32(3.0)), (f32(5.0), f32(7.0))):   # near and far limits
        P += [((0.0, 0.0, zn), (0.2, 0.0, zo), (0.0, 0.2, zo)), ((0.0, 0.0, zo), (0.1, 0.1, zn), (-0.2, 0.1, zo))]
    return tris_from(P)


def far_plane(f):
    """Each combination across z = 5: the far plane's v0 v2 case taken (v2.x <= 5 / f) and refused (v2.x > 5 / f,
    :1607), its (w1 - w0) divisor (:1615) with w1 - w0 small and large, and the other branches."""
    wl = 5.0 / f
    P = [((0.0, 0.0, 4.0), (0.3, 0.0, 6.0), (-0.4, 0.2, 4.5)),          # v0 v2 in, v2.x <= 5 / f: split
         ((0.0, 0.0, 4.9), (0.1, 0.1, 5.2), (-0.3, -0.2, 1.0)),         # (w1 - w0 small)
         ((0.0, 0.0, 1.0), (0.2, 0.1, 9.0), (wl * 0.5, 0.3, 3.0)),
         ((0.0, 0.0, 4.0), (0.3, 0.0, 6.0), (0.4, 0.2, 4.5)),           # v0 v2 in, v2.x > 5 / f: dropped
         ((0.0, 0.0, 2.0), (0.3, 0.0, 8.0), (wl * 2.0, -0.1, 3.0)),
         ((0.0, 0.0, 4.0), (0.3, 0.0, 6.0), (0.1, 0.2, 7.5)),           # only v0 in
         ((0.0, 0.0, 6.0), (0.3, 0.0, 4.0), (0.1, 0.2, 7.5)),           # only v1 in
         ((0.0, 0.0, 6.0), (0.3, 0.0, 7.0), (0.1, 0.2, 2.5)),           # only v2 in
         ((0.0, 0.0, 3.0), (0.3, 0.0, 4.0), (0.1, 0.2, 7.5)),           # v0 v1 in
         ((0.0, 0.0, 6.0), (0.3, 0.0, 4.0), (0.1, 0.2, 2.5)),           # v1 v2 in
         ((0.0, 0.0, 6.0), (0.3, 0.0, 7.0), (0.1, 0.2, 8.5))]           # all out
    return tris_from(P)


# A single triangle that the clip cuts into 20 (a search over the oracle at 64 x 48, f = 36, camera at the origin):
# lanes above 16 of rast_geom_warp_kernel hold its descendants.
MANY_DESCENDANTS = [[-0.6088365316390991, 3.0481772422790527, 4.701173782348633],
                    [14.409987449645996, 15.761775016784668, -1.432137370109558],
                    [-14.197898864746094, -21.227373123168945, 10.985888481140137]]


def rot(yaw, pitch, roll):
    """A rotation (yaw about y, pitch about x, roll about z), 3 x 3 row-major."""
    cy, sy, cp, sp, cr, sr = np.cos(yaw), np.sin(yaw), np.cos(pitch), np.sin(pitch), np.cos(roll), np.sin(roll)
    Ry = np.array([[cy, 0, -sy], [0, 1, 0], [sy, 0, cy]])
    Rx = np.array([[1, 0, 0], [0, cp, sp], [0, -sp, cp]])
    Rz = np.array([[cr, sr, 0], [-sr, cr, 0], [0, 0, 1]])
    return Rz @ Rx @ Ry


def camera_R(M, T=(0.0, 0.0, 0.0)):
    """glm's column-major mat4 of rotation M (row-major 3 x 3) and translation column T."""
    R = np.eye(4)
    R[:3, :3] = M
    R[:3, 3] = T
    return np.ascontiguousarray(R.T, np.float32).reshape(-1).copy()


def to_world(t, M, T, cam):
    """Camera-space triangles -> world space for camera position `cam` and R = [M | T] (float64, then float32)."""
    t = t.copy()
    for k in ("v0", "v1", "v2"):
        p = t[k][:, :3].astype(np.float64)
        t[k][:, :3] = ((p - np.asarray(T)) @ M + np.asarray(cam[:3])).astype(f32)   # M^T (p - T) + cam, row vectors
    with np.errstate(all="ignore"):
        h.compute_normals(t)
    return t


# ---- the cases -----------------------------------------------------------------------------------
def C(name, frame, build, light, cam=(0.0, 0.0, 0.0, 1.0), R=None, shadow=True, large=False):
    """shadow: the scene has box triangles (shadow volumes); large: more than 8192 pre-clip triangles.  Both are
    stated here so that the tests can choose cases without building them (test_cases_have_what_they_are_named_for
    checks them)."""
    return dict(name=name, frame=frame, build=build, light=light, cam=tuple(cam), R=R, shadow=shadow, large=large)


def _fuzz_scene(seed, n_room, n_boxes, zhi=9.0):
    rng = np.random.default_rng(seed)
    room = fuzz(rng, n_room, zhi=zhi)
    return room, box_tris(rng, n_boxes) if n_boxes else NONE


def _rotated(seed, n_room, n_boxes, M, T, cam):
    room, boxes = _fuzz_scene(seed, n_room, n_boxes)
    return to_world(room, M, T, cam), (to_world(boxes, M, T, cam) if n_boxes else NONE)


def _degenerate_shadow():
    # a box triangle with the edge (0, 0, 1) - (0, 0, 2) on a line through the camera, light on the camera: the
    # shadow-volume sides of that edge have no area and ComputeNormal computes 0 * inf
    b = tris_from([((0, 0, 1), (0, 0, 2), (0.5, 0.25, 1))], color=[(0.5, 0.5, 0.5)])
    return tris_from([((-1, -1, 3), (1, -1, 3), (0, 1, 3))], color=[(0.4, 0.5, 0.6)]), b


def _light_in_box():
    rng = np.random.default_rng(77)
    room = fuzz(rng, 40, zlo=0.5)
    return room, closed_box((-0.4, -0.3, 1.6), (0.4, 0.5, 2.4), rng)


def _zero_denominator():
    # H = 23: plane 3's inside test is y < w * 23 / 2, t_param uses h = (float)(23 / 2) = 11.  v0 at y = 22.75,
    # w = 2 is inside, v1 at y = 11.75, w = 1 outside: the denominator is exactly 0, t_param is inf and the new
    # vertex infinite; plane 4 and the near plane drop what the later lerps make of it
    f = f32(20.0)
    P = [((0.5, 22.75, 2 * f), (0.25, 11.75, f), (-0.5, 0.0, 1.5 * f)),
         ((0.5, 22.75, 2 * f), (0.25, 11.75, f), (0.25, 21.0, 2 * f)),
         ((0.25, 11.75, f), (0.5, 22.75, 2 * f), (-0.5, 0.0, 1.5 * f))]
    room = tris_from(P, rng=np.random.default_rng(3))
    rng = np.random.default_rng(23)
    return np.concatenate([room, fuzz(rng, 60, zlo=0.5, zhi=4.0)]), NONE


def _many_descendants():
    # with a box triangle, so that pipelined frames take rast_geom_warp_kernel
    rng = np.random.default_rng(17)
    return np.concatenate([tris_from([MANY_DESCENDANTS], rng=rng), fuzz(rng, 5)]), box_tris(rng, 1)


def _on_limits(frame):
    W, H, f = FRAMES[frame]
    return lambda: (np.concatenate([on_limits(W, H, f), far_plane(f)]), box_tris(np.random.default_rng(5), 3))


def _caller_nan():
    rng = np.random.default_rng(41)
    room = fuzz(rng, 30, zlo=0.5, zhi=6.0)
    room["v1"][3, 0] = np.nan           # a caller's NaN and inf vertices: dropped by the clip
    room["v2"][7, 2] = np.inf
    room["v0"][11, 1] = -np.inf
    return room, NONE


# The far plane's v0 v2 case lerps v2 towards v1 with (5 / f - w2) / (w1 - w0) (:1615).  With w0 and w1 an ulp
# either side of 5 / f and v2 a little nearer, the parameter is in the thousands and the new vertex lands 5.25e7
# pixels right of the frame's centre at W = 32768: finite, and converted to int and drawn by the reference.
FAR_SLIP = [(0.0, 0.0, 5.0), (4.950000286102295, 0.0, 5.000000476837158), (-4.948431015014648, 0.0, 4.998414993286133)]


def _far_slip(boxes):
    rng = np.random.default_rng(61)
    room = np.concatenate([tris_from([FAR_SLIP], rng=rng), fuzz(rng, 20, zlo=0.5, zhi=6.0)])
    return room, box_tris(rng, 2) if boxes else NONE


def _chunked():
    # shadow-free and at least 16 MB: travels in chunks, and the geometry stage runs once per chunk
    soup = h.scene_soup_rast(200_000, edge=0.02)
    for k in ("v0", "v1", "v2"):
        soup[k][:, 2] += f32(3.0)
    rng = np.random.default_rng(99)
    extra = fuzz(rng, 400, zhi=6.0)
    return np.concatenate([extra[:200], soup, extra[200:]]), NONE


M_YPR = rot(0.7, -0.45, 0.3)
T_COL = (0.25, -0.4, 0.6)
LIGHT = dict(h.DEFAULT_RAST_LIGHT)
CASES = [
    C("fuzz_64x48", "64x48", lambda: _fuzz_scene(1, 600, 12), dict(LIGHT, pos=(0.2, -0.3, 0.5, 1.0))),
    C("fuzz_320x240", "320x240", lambda: _fuzz_scene(2, 300, 20), dict(LIGHT, pos=(-0.3, 0.2, 0.1, 1.0))),
    C("fuzz_37x23", "37x23", lambda: _fuzz_scene(3, 400, 10), dict(LIGHT, pos=(0.1, 0.1, 0.2, 1.0))),
    C("shadow_free_64x48", "64x48", lambda: _fuzz_scene(4, 700, 0), LIGHT, shadow=False),
    C("shadow_free_320x240", "320x240", lambda: _fuzz_scene(5, 333, 0), LIGHT, shadow=False),
    C("on_limits_64x48", "64x48", _on_limits("64x48"), dict(LIGHT, pos=(0.0, 0.3, 0.2, 1.0))),
    C("on_limits_320x240", "320x240", _on_limits("320x240"), dict(LIGHT, pos=(0.0, 0.3, 0.2, 1.0))),
    C("on_limits_37x23", "37x23", _on_limits("37x23"), dict(LIGHT, pos=(0.0, 0.3, 0.2, 1.0))),
    C("degenerate_shadow_sides", "64x48", _degenerate_shadow, dict(LIGHT, pos=(0.0, 0.0, 0.0, 1.0))),
    C("light_inside_a_box", "320x240", _light_in_box, dict(LIGHT, pos=(0.05, 0.1, 2.0, 1.0))),
    C("yaw_pitch_roll_translated_64x48", "64x48",
      lambda: _rotated(6, 500, 10, M_YPR, T_COL, (0.3, -0.2, -1.0)),
      dict(LIGHT, pos=(0.5, 0.2, -0.5, 1.0)), cam=(0.3, -0.2, -1.0, 1.0), R=camera_R(M_YPR, T_COL)),
    C("yaw_pitch_roll_320x240", "320x240",
      lambda: _rotated(7, 260, 16, rot(-1.1, 0.6, -0.8), (0, 0, 0), (-0.5, 0.4, 0.7)),
      dict(LIGHT, pos=(0.1, 0.2, 0.3, 1.0)), cam=(-0.5, 0.4, 0.7, 1.0), R=camera_R(rot(-1.1, 0.6, -0.8))),
    C("many_descendants", "64x48", _many_descendants, LIGHT),
    C("caller_nan_and_inf_vertices", "64x48", _caller_nan, LIGHT, shadow=False),
    C("zero_denominator_37x23", "37x23", _zero_denominator, LIGHT, shadow=False),
    C("far_slip_32768x48", "32768x48", lambda: _far_slip(False), LIGHT, shadow=False),
    C("far_slip_shadow_32768x48", "32768x48", lambda: _far_slip(True), dict(LIGHT, pos=(0.1, -0.2, 0.3, 1.0))),
    C("tiled_shadow_64x48", "64x48", lambda: _fuzz_scene(8, 8000, 40), dict(LIGHT, pos=(0.2, -0.3, 0.5, 1.0)),
      large=True),
    C("tiled_shadow_free_320x240", "320x240", lambda: _fuzz_scene(9, 9000, 0), LIGHT, shadow=False, large=True),
    C("chunked_upload_320x240", "320x240", _chunked, LIGHT, shadow=False, large=True),
]
BY_NAME = {c["name"]: c for c in CASES}


def build(c):
    """(room, boxes, W, H, f, cam, R, light) of a case."""
    W, H, f = FRAMES[c["frame"]]
    room, boxes = c["build"]()
    R = c["R"] if c["R"] is not None else h.identity_R()
    return (np.ascontiguousarray(room), np.ascontiguousarray(boxes), W, H, f, h.f32(*c["cam"]), R, c["light"])


def n_pre(room, boxes):
    return len(room) + 7 * len(boxes)


def convertible(clipped, W, H, f):
    """Per triangle: every vertex's screen position converts to int (VertexShader :513-516 in float32 steps: finite
    and inside int range, beyond which rast_vertex drops a triangle)."""
    ok = np.ones(len(clipped), bool)
    with np.errstate(all="ignore"):
        for k in ("v0", "v1", "v2"):
            v = clipped[k]
            x = (f32(f) * (v[:, 0] / v[:, 2]).astype(f32)).astype(f32) + f32(W // 2)
            y = (f32(f) * (v[:, 1] / v[:, 2]).astype(f32)).astype(f32) + f32(H // 2)
            ok &= np.isfinite(x) & np.isfinite(y) & (np.abs(x) < 2.0 ** 31) & (np.abs(y) < 2.0 ** 31)
    return ok


def band_rows(clipped, H, f):
    """ymin, ymax of each triangle's truncated vertex rows, as rast_geom_kernel<2> computes them when it culls a
    band (f * (y / z) + (float)(H / 2), then static_cast<int>); rows of triangles that do not convert are 0."""
    with np.errstate(all="ignore"):
        Y = np.stack([(f32(f) * (clipped[k][:, 1] / clipped[k][:, 2]).astype(f32)).astype(f32) + f32(H // 2)
                      for k in ("v0", "v1", "v2")], 1)
        ok = (np.abs(Y) < f32(2.0 ** 31)).all(1)
        Yi = np.where(np.abs(Y) < f32(2.0 ** 31), Y, 0).astype(np.int64)
    return ok, Yi.min(1), Yi.max(1)


def oracle_geometry(W, H, f, cam, R, light, room, boxes):
    """oracle_rast_geometry with room for 4 descendants per pre-clip triangle (the cases stay well below that)."""
    return h.oracle_rast_geometry(W, H, f, cam, R, light, room, boxes, cap=4 * n_pre(room, boxes) + 4096)


def oracle_census(cases=CASES):
    """The oracle's census over the given cases' geometry stages: ({name: count}, descendant histogram)."""
    census_read(reset=True)
    for c in cases:
        room, boxes, W, H, f, cam, R, light = build(c)
        oracle_geometry(W, H, f, cam, R, light, room, boxes)
    return census_read(reset=True)
