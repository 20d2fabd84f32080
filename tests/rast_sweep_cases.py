"""Camera-space clipped lists for the rasteriser sweep (tests/test_rast_sweep_gpu.py) whose pixel footprints
are exact, and what each list makes the triangle loop do.

Vertices are placed on chosen pixels through a numpy float32 restatement of rast_vertex
(computer-graphics_b200/csrc/rast_kernels.cu, VertexShader of the reference): x = int(f * (X / Z) + (float)(W / 2)),
every operation rounded on its own, no FMA.  From the same restatement `describe` derives the quantities the
kernels branch on: the list length, each triangle's row span and `xmax - vxmin` (the scatter path's small / big
split, S2_ROWS / S2_XSPAN in rast_fast.cuh), the per-tile list lengths at tile sizes 8, 16 and 32 (bounding
boxes widened by the minor-axis undershoot, as rast_spread_kernel / rast_short_kernel count them), and the branch
of the closed-form edge walk (edge_run) that each edge takes.  Nothing here loads the product library.
"""
import numpy as np

import helpers as h

f32 = np.float32
S2_ROWS, S2_XSPAN = 24, 60          # rast_fast.cuh
BITS_MAX_TRIS = 2048                # RAST_BITS_MAX_TRIS: longer lists take setup / spread / scan
LIST_CAP = 2048                     # RAST_LIST_CAP: longer tile lists take the global sort
SPREAD_BLOCK_MAX = 8192             # rast_spread_launch: one block per triangle up to this length

# strategies: (OPT_RAST_PATH, OPT_RAST_TILE_LOG2)
AUTO, SCATTER, ORD8, ORD16, ORD32 = (0, 5), (2, 5), (1, 3), (1, 4), (1, 5)
ORDERED = (ORD8, ORD16, ORD32)
ALL = (AUTO, SCATTER) + ORDERED
LIGHT_CAM = (0.1, -0.3, 1.2, 1.0)
TEX_CAM = (0.2, -0.1, -1.5, 1.0)


# ---- rast_vertex restated ------------------------------------------------------------------------
def pixel(c, z, f, size):
    """int(f * (c / z) + (float)(size / 2)) in float32 steps (truncation towards zero, as static_cast<int>)."""
    q = (np.asarray(c, f32) / np.asarray(z, f32)).astype(f32)
    v = ((f32(f) * q).astype(f32) + f32(size // 2)).astype(f32)
    return np.trunc(v).astype(np.int64)


def coord(p, z, f, size):
    """A camera-space coordinate at depth z that lands on pixel p (checked through `pixel`)."""
    p, z = np.asarray(p, np.int64), np.asarray(z, f32)
    target = np.where(p >= 0, p + 0.5, p - 0.5)              # the middle of the interval int() maps to p
    c = ((target - size // 2) * z.astype(np.float64) / f).astype(f32)
    got = pixel(c, z, f, size)
    assert np.array_equal(got, p), (p[got != p], got[got != p])
    return c


def make_tris(px, py, z, W, H, f, shadow=None, rng=None):
    """Triangles with vertex k on pixel (px[:, k], py[:, k]) at depth z[:, k] (w = z / f, as the clip stage leaves it)."""
    px, py = np.atleast_2d(px), np.atleast_2d(py)
    n = len(px)
    z = np.broadcast_to(np.asarray(z, f32).reshape(n, -1), (n, 3))
    rng = rng or np.random.default_rng(0)
    t = np.zeros(n, h.RAST_TRI)
    for k, name in enumerate(("v0", "v1", "v2")):
        t[name][:, 0] = coord(px[:, k], z[:, k], f, W)
        t[name][:, 1] = coord(py[:, k], z[:, k], f, H)
        t[name][:, 2] = z[:, k]
        t[name][:, 3] = z[:, k] / f32(f)
    t["color"] = rng.uniform(0.15, 0.75, (n, 3)).astype(f32)
    if shadow is not None:
        t["color"][shadow] = -1.0
    with np.errstate(all="ignore"):
        h.compute_normals(t)
    bad = ~np.isfinite(t["normal"]).all(axis=1)               # points and slivers: no normal of their own
    t["normal"][bad] = (0.0, 0.0, -1.0, 1.0)
    return t


# ---- footprints (pixel coordinates, one row per triangle, columns = vertices) -------------------------
def fp_tiny(rng, n, W, H):
    """1-3 px triangles anywhere on the frame."""
    x0, y0 = rng.integers(0, W, n), rng.integers(0, H, n)
    dx, dy = rng.integers(-2, 3, (n, 2)), rng.integers(-2, 3, (n, 2))
    return np.stack([x0, x0 + dx[:, 0], x0 + dx[:, 1]], 1), np.stack([y0, y0 + dy[:, 0], y0 + dy[:, 1]], 1)


def fp_exact(rng, n, W, H, rows, cols):
    """Exactly `rows` rows (ymax - ymin + 1) and `cols` = xmax - vxmin, vertex order and interior vertex random."""
    x0, y0 = rng.integers(-cols // 2, W - cols // 2, n), rng.integers(-rows // 2, H - rows // 2, n)
    px = np.stack([x0, x0 + cols, x0 + rng.integers(0, cols + 1, n)], 1)
    py = np.stack([y0, y0 + rng.integers(0, rows, n), y0 + rows - 1], 1)
    flip = rng.uniform(size=n) < 0.5                           # the lone vertex at the bottom instead of the top
    py[flip] = (2 * y0[flip] + rows - 1)[:, None] - py[flip]
    perm = np.argsort(rng.uniform(size=(n, 3)), axis=1)
    return np.take_along_axis(px, perm, 1), np.take_along_axis(py, perm, 1)


def fp_big(rng, n, W, H):
    """Hundreds of rows, many partly off screen on one side or another."""
    cx, cy = rng.integers(-W // 4, W + W // 4, n), rng.integers(-H // 4, H + H // 4, n)
    px = cx[:, None] + rng.integers(-W // 2 - 150, W // 2 + 150, (n, 3))
    py = cy[:, None] + rng.integers(-H // 2 - 150, H // 2 + 150, (n, 3))
    py[:, 0] = cy - 160                                        # at least ~ 300 rows
    py[:, 1] = cy + 160
    return px, py


def fp_degenerate(rng, n, W, H):
    """Points, horizontal and vertical slivers, nearly collinear triangles (one vertex 1 px off a long line)."""
    x0, y0 = rng.integers(-5, W + 5, n), rng.integers(-5, H + 5, n)
    px, py = np.stack([x0, x0, x0], 1), np.stack([y0, y0, y0], 1)
    kind = np.arange(n) % 4
    L = rng.integers(3, 120, n)
    hs, vs, co = kind == 1, kind == 2, kind == 3
    px[hs, 1] += L[hs]; px[hs, 2] += L[hs] // 3
    py[vs, 1] += L[vs]; py[vs, 2] += L[vs] // 2
    ex, ey = rng.integers(-90, 91, n), rng.integers(-40, 41, n)
    px[co, 1] += ex[co]; py[co, 1] += ey[co]
    px[co, 2] += ex[co] // 2 + 1; py[co, 2] += ey[co] // 2
    return px, py


def fp_shallow(rng, n, W, H):
    """Long shallow edges: |dx| >> |dy| > 0, far more than 8 samples."""
    x0, y0 = rng.integers(-40, W, n), rng.integers(0, H, n)
    dx = rng.integers(20, 260, n) * np.where(rng.uniform(size=n) < 0.5, -1, 1)
    dy = rng.integers(1, 7, n) * np.where(rng.uniform(size=n) < 0.5, -1, 1)
    px = np.stack([x0, x0 + dx, x0 + dx // 2 + rng.integers(-3, 4, n)], 1)
    py = np.stack([y0, y0 + dy, y0 + rng.integers(-9, 10, n)], 1)
    return px, py


def fp_crowd(rng, n, x0, y0):
    """Inside the 6 x 6 block at (x0, y0) (x0 - 1 on the same 8-px tile column): one tile at every tile size."""
    return rng.integers(x0, x0 + 6, (n, 3)), rng.integers(y0, y0 + 6, (n, 3))


FOOTPRINTS = {"tiny": fp_tiny, "big": fp_big, "degenerate": fp_degenerate, "shallow": fp_shallow,
              "r24": lambda r, n, W, H: fp_exact(r, n, W, H, 24, 40), "r25": lambda r, n, W, H: fp_exact(r, n, W, H, 25, 40),
              "c60": lambda r, n, W, H: fp_exact(r, n, W, H, 12, 60), "c61": lambda r, n, W, H: fp_exact(r, n, W, H, 12, 61),
              "r24c60": lambda r, n, W, H: fp_exact(r, n, W, H, 24, 60)}
BOUNDARY = {"r24": 1, "r25": 1, "c60": 1, "c61": 1, "r24c60": 1}


def build_list(n, W, H, f, seed, mix, shadow=0.0, ties=0, crowd=None):
    """n triangles: footprint kinds drawn with weights `mix`, a fraction `shadow` of shadow-volume triangles,
    `ties` coincident copies (same vertices, hence the same zinv at every pixel, new colour) of earlier triangles
    placed later in the list, and `crowd` = (count, x0, y0) triangles piled over one tile."""
    rng = np.random.default_rng(seed)
    kinds = list(mix)
    w = np.array([mix[k] for k in kinds], float)
    n_crowd = crowd[0] if crowd else 0
    n_free = n - ties - n_crowd
    counts = np.floor(w / w.sum() * n_free).astype(int)
    counts[0] += n_free - counts.sum()
    pxs, pys = [], []
    for k, c in zip(kinds, counts):
        if c:
            px, py = FOOTPRINTS[k](rng, int(c), W, H)
            pxs.append(px); pys.append(py)
    if n_crowd:
        px, py = fp_crowd(rng, n_crowd, crowd[1], crowd[2])
        pxs.append(px); pys.append(py)
    px, py = np.concatenate(pxs), np.concatenate(pys)
    order = rng.permutation(len(px))
    px, py = px[order], py[order]
    z = rng.uniform(1.0, 4.0, (len(px), 1)) * (1 + rng.uniform(-0.2, 0.2, (len(px), 3)))
    sh = rng.uniform(size=len(px)) < shadow
    t = make_tris(px, py, z, W, H, f, sh, rng)
    if ties:
        src = rng.integers(0, len(t), ties)
        pos = np.sort(rng.integers(0, len(t) + 1, ties))
        dup = t[src].copy()
        dup["color"] = rng.uniform(0.15, 0.75, (ties, 3)).astype(f32)    # opaque copies: the later one must win
        t = np.insert(t, np.maximum(pos, src + 1), dup)
    assert len(t) == n, (len(t), n)
    return t


def texture_fields(t, seed):
    """Every texture on every object index, garbage indices among them (as test_textured_random_clipped_lists)."""
    rng = np.random.default_rng(1000 + seed)
    t["texture"] = rng.integers(0, 4, len(t))
    t["index"] = rng.integers(0, 6, len(t))
    t["index"][::7] = 0x01000003
    t["index"][3::11] = -7
    t["texture"][t["color"][:, 0] < 0] = 0
    return t


# ---- what the kernels will do with a list ----------------------------------------------------------
EDGE_BRANCHES = ("dy0", "steep", "short", "shallow")


def describe(t, W, H, f, fb=None):
    """Per-triangle pixel geometry and the kernels' classes, from the float32 restatement only."""
    fb0, fb1 = fb if fb else (0, H)
    X = np.stack([pixel(t[v][:, 0], t[v][:, 2], f, W) for v in ("v0", "v1", "v2")], 1)
    Y = np.stack([pixel(t[v][:, 1], t[v][:, 2], f, H) for v in ("v0", "v1", "v2")], 1)
    ymin, ymax = Y.min(1), Y.max(1)
    vxmin, xmax = X.min(1), X.max(1)
    xorg = vxmin - 1                                           # a minor-axis sample can undershoot by one
    row0 = np.maximum(ymin, fb0)
    nrows = np.maximum(0, np.minimum(ymax, fb1 - 1) - row0 + 1)
    nrows[(xmax <= 0) | (xorg >= W) | (xmax <= xorg)] = 0
    span_rows, xspan = ymax - ymin + 1, xmax - vxmin
    big = (nrows > 0) & ((span_rows > S2_ROWS) | (xspan > S2_XSPAN))
    edges = []
    for e in range(3):
        dx = np.abs(X[:, e] - X[:, (e + 1) % 3]); dy = np.abs(Y[:, e] - Y[:, (e + 1) % 3])
        n = np.maximum(dx, dy) + 1
        edges.append(np.where(dy == 0, 0, np.where(dy >= dx, 1, np.where(n <= 8, 2, 3))))
    edges = np.stack(edges, 1)
    tiles, tile_span = {}, {}
    vis = nrows > 0
    for ts in (3, 4, 5):
        tx = (W + (1 << ts) - 1) >> ts
        ty0 = fb0 >> ts
        ty = ((fb1 - 1) >> ts) - ty0 + 1
        a = np.maximum(0, xorg) >> ts
        b = np.minimum(W - 1, xmax - 1) >> ts
        c = row0 >> ts
        d = (row0 + nrows - 1) >> ts
        grid = np.zeros((ty + 1, tx + 1), np.int64)            # 2-D difference array of the bounding boxes
        for (yy, xx, s) in ((c, a, 1), (c, b + 1, -1), (d + 1, a, -1), (d + 1, b + 1, 1)):
            np.add.at(grid, (yy[vis] - ty0, xx[vis]), s)
        tiles[ts] = grid.cumsum(0).cumsum(1)[:ty, :tx]
        tile_span[ts] = np.where(vis, (b - a + 1) * (d - c + 1), 0)
    shadow = ~(t["color"][:, 0] >= 0)
    return dict(n=len(t), X=X, Y=Y, span_rows=span_rows, xspan=xspan, nrows=nrows, big=big, edges=edges,
                tiles=tiles, tile_span=tile_span, shadow=shadow, W=W, H=H)


def footprint_classes(d):
    """Names of the footprint classes present among the triangles that reach the frame."""
    X, Y, W, H = d["X"], d["Y"], d["W"], d["H"]
    vis = d["nrows"] > 0
    r, c = d["span_rows"], d["xspan"]
    same_x, same_y = (X == X[:, :1]).all(1), (Y == Y[:, :1]).all(1)
    area2 = np.abs((X[:, 1] - X[:, 0]) * (Y[:, 2] - Y[:, 0]) - (X[:, 2] - X[:, 0]) * (Y[:, 1] - Y[:, 0]))
    out = set()
    tests = {
        "tiny 1-3 px": (r <= 3) & (c <= 2),
        "24 rows": (r == 24) & (c <= S2_XSPAN), "25 rows": r == 25,
        "60 columns": (c == 60) & (r <= S2_ROWS), "61 columns": c == 61,
        "hundreds of rows": r >= 200,
        "off left": X.min(1) < 0, "off right": X.max(1) >= W, "off top": Y.min(1) < 0, "off bottom": Y.max(1) >= H,
        "point": same_x & same_y, "horizontal sliver": same_y & ~same_x, "vertical sliver": same_x & ~same_y,
        "nearly collinear": ~same_x & ~same_y & (area2 <= np.maximum(np.abs(X - X[:, :1]).max(1), 1)) & (np.maximum(r, c) > 8),
        "long shallow edge": (d["edges"] == 3).any(1),
    }
    for k, m in tests.items():
        if (m & vis).any():
            out.add(k)
    for i, name in enumerate(EDGE_BRANCHES):
        if ((d["edges"] == i).any(1) & vis).any():
            out.add("edge " + name)
    return out
