"""Sweep of the rasteriser's triangle-loop strategies and size classes against the plain-C oracle, bit for bit.

The triangle loop picks its kernels from the list length (bit-per-triangle tile lists up to 2048 triangles, then
setup / spread / scan, and from 8193 on the owners of the row slots written by the setup kernel), from each triangle's
footprint (the scatter path's small / big split at 24 rows and 60 columns), from shadow-volume triangles, textures
and colour modes, from the tile size, the row band and pipelining.  Every case below is a clipped list with exact
pixel footprints (tests/rast_sweep_cases.py); `test_sweep_reaches_every_class` checks, without a GPU, that the
cases reach every class, and each GPU case checks from the launch timeline (B200_TIMELINE) that the kernels of
its class ran.
"""
import os
import re

import numpy as np
import pytest

import helpers as h
import rast_sweep_cases as sc
from rast_sweep_cases import ALL, AUTO, ORD8, ORD16, ORD32, ORDERED, SCATTER

FRAMES = {"250x170": (250, 170, 150.0), "37x23": (37, 23, 20.0), "96x64": (96, 64, 60.0), "1920x1080": (1920, 1080, 900.0)}
SMALL_MIX = {"tiny": 6, "r24": 1, "r25": 1, "c60": 1, "c61": 1, "degenerate": 1, "shallow": 1}
MIXED = dict(SMALL_MIX, big=0.05)
BIG_MIX = {"tiny": 4, "big": 1, "degenerate": 1, "shallow": 1}
BOUNDARY = {"r24": 1, "r25": 1, "c60": 1, "c61": 1, "r24c60": 1, "tiny": 1}
CROWD = (2600, 17, 9)     # 2600 triangles inside pixels 17..22 x 9..14: one tile at 8, 16 and 32 px


def C(name, n, frame, mix, strategies, shadow=0.0, tex=False, colour=0, indirect=0.2, ties=0, crowd=None,
      bands=True, seed=None):
    return dict(name=name, n=n, frame=frame, mix=mix, strategies=strategies, shadow=shadow, tex=tex, colour=colour,
                indirect=indirect, ties=ties, crowd=crowd, bands=bands and not colour,
                seed=seed if seed is not None else sum(map(ord, name)))


A_ORD = (AUTO,) + ORDERED
CASES = [
    # ---- one triangle ----
    C("n1_big", 1, "250x170", {"big": 1}, ALL),
    C("n1_big_shadow", 1, "37x23", {"big": 1}, A_ORD, shadow=1.0),
    C("n1_tiny", 1, "37x23", {"tiny": 1}, ALL),
    C("n1_r25_tex", 1, "96x64", {"r25": 1}, (AUTO, ORD8), tex=True),
    C("n1_shallow_colour1", 1, "96x64", {"shallow": 1}, (AUTO, ORD16), colour=1),
    C("n1_degenerate", 1, "37x23", {"degenerate": 1}, ALL),
    # ---- short lists: bit-per-triangle tile lists, rast_short_kernel ----
    C("n2047_tiny", 2047, "250x170", {"tiny": 1}, ALL),
    C("n2047_boundary", 2047, "37x23", BOUNDARY, ALL),
    C("n2047_mixed_shadow", 2047, "250x170", MIXED, A_ORD, shadow=0.25),
    C("n2047_tex", 2047, "250x170", MIXED, (AUTO, ORD8, ORD32), tex=True),
    C("n2047_colour1_shadow", 2047, "96x64", SMALL_MIX, (AUTO, ORD8), shadow=0.25, colour=1),
    C("n2047_indirect", 2047, "96x64", SMALL_MIX, ALL, indirect=0.15),
    C("n2047_degenerate_shallow", 2047, "250x170", {"degenerate": 1, "shallow": 1}, ALL),
    C("n2048_boundary", 2048, "250x170", BOUNDARY, ALL),
    C("n2048_big_shadow_ties", 2048, "250x170", BIG_MIX, A_ORD, shadow=0.25, ties=300),
    C("n2048_tex_ties", 2048, "96x64", MIXED, (AUTO, ORD16), tex=True, ties=300),
    C("n2048_colour2", 2048, "250x170", MIXED, (AUTO, ORD32), colour=2),
    C("n2048_ties", 2048, "37x23", SMALL_MIX, ALL, ties=400),
    # ---- long lists: setup / spread (one block per triangle) / scan / rows ----
    C("n2049_boundary", 2049, "250x170", BOUNDARY, ALL),
    C("n2049_boundary_37x23", 2049, "37x23", BOUNDARY, ALL),
    C("n2049_mixed_shadow", 2049, "250x170", MIXED, A_ORD, shadow=0.25),
    C("n2049_big_shadow_37x23", 2049, "37x23", BIG_MIX, A_ORD, shadow=0.25),
    C("n2049_tex", 2049, "250x170", MIXED, A_ORD, tex=True),
    C("n2049_colour1", 2049, "250x170", MIXED, (AUTO, ORD8, ORD32), colour=1),
    C("n2049_colour2_shadow", 2049, "96x64", MIXED, (AUTO, ORD16), shadow=0.25, colour=2),
    C("n2049_ties", 2049, "250x170", MIXED, ALL, ties=400),
    C("n2049_ties_shadow", 2049, "96x64", MIXED, A_ORD, shadow=0.25, ties=400),
    C("n2049_indirect", 2049, "250x170", SMALL_MIX, ALL, indirect=0.15),
    C("n2049_indirect_tex", 2049, "96x64", MIXED, (AUTO, ORD8), tex=True, indirect=0.205),
    C("n4000_degenerate_shallow", 4000, "250x170", {"degenerate": 1, "shallow": 1}, ALL),
    C("n8192_big_shadow", 8192, "250x170", BIG_MIX, A_ORD, shadow=0.25),
    C("n8192_big", 8192, "96x64", BIG_MIX, ALL),
    C("n8192_boundary", 8192, "250x170", BOUNDARY, ALL),
    C("n8192_tex", 8192, "250x170", MIXED, (AUTO, ORD16), tex=True),
    C("n8192_colour2", 8192, "250x170", MIXED, (AUTO, ORD8), colour=2),
    # ---- over 8192: the setup kernel writes the row-slot owners, one thread per triangle in the spread kernel ----
    C("n8193_big_shadow", 8193, "250x170", BIG_MIX, A_ORD, shadow=0.25),
    C("n8193_big_shadow_37x23", 8193, "37x23", BIG_MIX, A_ORD, shadow=0.25),
    C("n8193_big", 8193, "250x170", BIG_MIX, ALL),
    C("n8193_boundary", 8193, "96x64", BOUNDARY, ALL),
    C("n8193_tex", 8193, "250x170", BIG_MIX, A_ORD, tex=True),
    C("n8193_colour1_shadow", 8193, "250x170", MIXED, (AUTO, ORD32), shadow=0.25, colour=1),
    C("n8193_colour2", 8193, "96x64", BIG_MIX, (AUTO, ORD8), colour=2),
    C("n8193_indirect_shadow", 8193, "250x170", MIXED, A_ORD, shadow=0.25, indirect=0.205),
    C("n8193_ties_shadow", 8193, "250x170", BIG_MIX, A_ORD, shadow=0.25, ties=1000),
    C("n8193_ties", 8193, "96x64", MIXED, ALL, ties=1000),
    C("n20000_tiny", 20000, "250x170", {"tiny": 1}, ALL),
    C("n20000_mixed_shadow", 20000, "250x170", MIXED, A_ORD, shadow=0.25),
    C("n20000_big_shadow_37x23", 20000, "37x23", BIG_MIX, A_ORD, shadow=0.25),
    C("n20000_boundary", 20000, "250x170", BOUNDARY, ALL),
    C("n20000_big", 20000, "96x64", BIG_MIX, ALL),
    C("n20000_tex", 20000, "250x170", MIXED, (AUTO, ORD8, ORD32), tex=True),
    C("n20000_colour1", 20000, "96x64", MIXED, (AUTO, ORD16), colour=1),
    C("n20000_indirect", 20000, "250x170", MIXED, ALL, indirect=0.15),
    C("n20000_ties", 20000, "250x170", MIXED, ALL, ties=3000),
    C("n20000_ties_shadow", 20000, "96x64", MIXED, A_ORD, shadow=0.25, ties=3000),
    # ---- more than 2048 triangles over one tile: the global sort ----
    C("crowd_n2600", 2600, "250x170", {"tiny": 1}, ALL, crowd=(2600, 17, 9)),
    C("crowd_n3000_shadow", 3000, "250x170", MIXED, A_ORD, shadow=0.25, crowd=CROWD),
    C("crowd_n3000_37x23", 3000, "37x23", SMALL_MIX, ALL, crowd=CROWD),
    C("crowd_n3000_tex", 3000, "250x170", MIXED, A_ORD, tex=True, crowd=CROWD),
    C("crowd_n3000_colour1", 3000, "96x64", SMALL_MIX, (AUTO, ORD8), colour=1, crowd=CROWD),
    C("crowd_n9000_big_shadow", 9000, "250x170", BIG_MIX, A_ORD, shadow=0.25, crowd=CROWD),
    C("crowd_n9000_tex", 9000, "96x64", MIXED, (AUTO, ORD8, ORD32), tex=True, crowd=CROWD),
    # ---- long edges at full HD ----
    C("hd_n300_big", 300, "1920x1080", {"big": 1}, (AUTO, SCATTER, ORD16, ORD32)),
    C("hd_n300_big_shadow", 300, "1920x1080", {"big": 1, "shallow": 1}, (AUTO, ORD32), shadow=0.25),
    C("hd_n2500_shallow", 2500, "1920x1080", {"shallow": 1, "r24c60": 1, "c61": 1}, ALL),
]
BY_NAME = {c["name"]: c for c in CASES}


def build_case(c):
    W, H, f = FRAMES[c["frame"]]
    t = sc.build_list(c["n"], W, H, f, c["seed"], c["mix"], shadow=c["shadow"], ties=c["ties"], crowd=c["crowd"])
    if c["tex"]:
        sc.texture_fields(t, c["seed"])
    return t, W, H, f


def band_edges(H):
    """The whole frame and three bands whose edges are not multiples of 8 (nor of 32)."""
    a, b = min(8 * (H // 24) + 3, H - 2), min(8 * (2 * H // 24) + 5, H - 1)
    return [(0, H)] + [(0, a), (a, b), (b, H)]


# ---------------------------------------------------------------------------------------------
# without a GPU: the cases reach every class
# ---------------------------------------------------------------------------------------------
def test_sweep_reaches_every_class():
    seen = set()
    def mark(*k):
        seen.add(k)
    for c in CASES:
        t, W, H, f = build_case(c)
        d = sc.describe(t, W, H, f)
        n = d["n"]
        assert n == c["n"]
        mark("length", n)
        for s in c["strategies"]:
            mark("strategy", s)
            if c["ties"] and n > sc.BITS_MAX_TRIS:
                mark("ties on a long list", s)
            # more than 2048 triangles over one tile of a frame of several tiles (the scatter path has no tiles)
            if s[0] != 2 and d["tiles"][s[1]].max() > sc.LIST_CAP and d["tiles"][s[1]].size > 1:
                mark("crowded tile", s[1])
                if c["tex"]:
                    mark("crowded tile, textured", s[1])
            # a range of more than 32 row slots and of more than 32 tiles: warp_spread's cooperative branch
            if (s[0] == 1 and n > sc.SPREAD_BLOCK_MAX and (d["nrows"] > 32).any() and (d["tile_span"][s[1]] > 32).any()):
                mark("over 8192, ordered, cooperative warp_spread", "big" if d["big"].any() else "",
                     "shadow" if d["shadow"].any() else "")
            if c["bands"]:
                mark("bands", s)
        shadow = d["shadow"].any()
        mark("content", "shadow" if 0.15 < d["shadow"].mean() < 0.35 else "shadow-free" if not shadow else "other")
        if c["tex"]:
            mark("content", "textured", "long" if n > sc.BITS_MAX_TRIS else "short")
        if c["colour"]:
            mark("content", f"colour {c['colour']}", "long" if n > sc.BITS_MAX_TRIS else "short")
        if c["indirect"] != 0.2 and n > sc.BITS_MAX_TRIS:
            mark("content", "entry indirect value on a long list")
        for k in sc.footprint_classes(d):
            mark("footprint", k)
        if c["frame"] in ("250x170", "37x23"):
            mark("frame", "not a multiple of 8 or 32")
        if c["frame"] == "1920x1080":
            mark("frame", "1920x1080")
    want = [("length", n) for n in (1, 2047, 2048, 2049, 8192, 8193, 20000)]
    want += [("strategy", s) for s in ALL] + [("ties on a long list", s) for s in ALL]
    want += [("crowded tile", ts) for ts in (3, 4, 5)] + [("crowded tile, textured", ts) for ts in (3, 5)]
    want += [("over 8192, ordered, cooperative warp_spread", "big", ""), ("over 8192, ordered, cooperative warp_spread", "big", "shadow")]
    want += [("bands", s) for s in ALL]
    want += [("content", k) for k in ("shadow", "shadow-free")]
    want += [("content", k, l) for k in ("textured", "colour 1", "colour 2") for l in ("short", "long")]
    want += [("content", "entry indirect value on a long list")]
    want += [("footprint", k) for k in ("tiny 1-3 px", "24 rows", "25 rows", "60 columns", "61 columns", "hundreds of rows",
                                        "off left", "off right", "off top", "off bottom", "point", "horizontal sliver",
                                        "vertical sliver", "nearly collinear", "long shallow edge",
                                        "edge dy0", "edge steep", "edge short", "edge shallow")]
    want += [("frame", "not a multiple of 8 or 32"), ("frame", "1920x1080")]
    missing = [k for k in want if k not in seen]
    assert not missing, f"classes no case reaches: {missing}"
    assert 60 <= len(CASES) <= 120 and len(BY_NAME) == len(CASES)


def test_generator_places_vertices_on_their_pixels():
    """The restated rast_vertex agrees with the chosen pixels, on and off screen, at the boundaries that decide
    the small / big split."""
    W, H, f = 250, 170, 150.0
    rng = np.random.default_rng(5)
    for rows, cols in ((24, 60), (25, 60), (24, 61), (1, 0)):
        px, py = sc.fp_exact(rng, 500, W, H, rows, cols) if rows > 1 else sc.fp_tiny(rng, 500, W, H)
        t = sc.make_tris(px, py, rng.uniform(0.5, 6.0, (500, 3)), W, H, f)
        d = sc.describe(t, W, H, f)
        assert np.array_equal(d["X"], px) and np.array_equal(d["Y"], py)
        if rows > 1:
            assert (d["span_rows"] == rows).all() and (d["xspan"] == cols).all()
            vis = d["nrows"] > 0
            assert np.array_equal(d["big"][vis], np.full(vis.sum(), rows > 24 or cols > 60))
    assert sc.pixel(sc.coord(-3, 2.0, f, W), 2.0, f, W) == -3     # int() truncates towards zero off screen


# ---------------------------------------------------------------------------------------------
# on the GPU
# ---------------------------------------------------------------------------------------------
def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def same(tag, key, got, want):
    g, w = np.asarray(got), np.asarray(want)
    if g.dtype == np.float32:
        g, w = bits(g), bits(w)
    bad = np.argwhere(g != w)
    if len(bad):
        first = tuple(bad[0][:2])
        raise AssertionError(f"{tag}: {key} differs at {len({tuple(b[:2]) for b in bad})} px, first (y, x) = {first}: "
                             f"{np.asarray(got)[first]} vs {np.asarray(want)[first]}")


@pytest.fixture(scope="module")
def tl_renderer(b200):
    """A context of its own with the launch timeline on (read when the context is created)."""
    old = os.environ.get("B200_TIMELINE")
    os.environ["B200_TIMELINE"] = "1"
    try:
        r = b200.Renderer(0)
    finally:
        if old is None:
            del os.environ["B200_TIMELINE"]
        else:
            os.environ["B200_TIMELINE"] = old
    yield r
    r.close()


@pytest.fixture(scope="module")
def tex():
    return h.synthetic_textures()


TL = re.compile(r"^\[b200 timeline\] (.+?)\s+-?[0-9.]+ us$")


def launched(capfd):
    names = []
    for line in capfd.readouterr().err.splitlines():
        m = TL.match(line.strip())
        if m and m.group(1) != "frame":
            names.append(m.group(1))
    return names


def check_kernels(tag, names, c, s, d):
    """The kernels the strategy must have launched for this list (and those it must not have)."""
    n, path = d["n"], s[0]
    shadow = bool(d["shadow"].any())
    fast = path == 2 or (path == 0 and not shadow and not c["tex"] and not c["colour"])
    def need(k, present=True):
        assert (k in names) == present, f"{tag}: {k} {'missing from' if present else 'in'} the launches {names}"
    if fast:
        need("rast_scatter2_kernel<count>"); need("rast_scatter2_kernel"); need("rast_resolve_kernel")
        need("rast_fill_kernel", False); need("rast_short_kernel", False); need("rast_setup_kernel", False)
        big = bool(d["big"].any())
        need("rast_setup_big_kernel", big); need("rast_scatter_kernel", big)
        return
    need("rast_fill_kernel"); need("rast_scatter2_kernel", False); need("rast_setup_big_kernel", False)
    need("rast_short_kernel", n <= sc.BITS_MAX_TRIS)
    need("rast_setup_kernel", n > sc.BITS_MAX_TRIS); need("rast_scan_kernel", n > sc.BITS_MAX_TRIS)
    if n > sc.BITS_MAX_TRIS:
        # fan-out: row-slot owners + tile counts + tile lists; from 8193 triangles on the setup kernel writes the owners
        want = 2 if n > sc.SPREAD_BLOCK_MAX else 3
        assert names.count("rast_spread_kernel") == want, f"{tag}: {names.count('rast_spread_kernel')} spread launches"
    fused = path == 0 or bool(c["colour"])
    need("rast_resolve_kernel<ordered>", fused); need("rast_post_kernel", not fused)
    need("rast_fill_kernel<emit>", bool(c["colour"]))
    need("rast_first_fragment_kernel", c["indirect"] != 0.2 and not c["colour"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c["name"] for c in CASES])
def test_sweep(b200, tl_renderer, tex, capfd, name):
    import torch
    c = BY_NAME[name]
    r = tl_renderer
    t, W, H, f = build_case(c)
    d = sc.describe(t, W, H, f)
    light = dict(h.DEFAULT_RAST_LIGHT, indirect=(c["indirect"],) * 3)
    cam = b200.make_camera(sc.TEX_CAM, f, h.identity_R(), W, H)
    L = b200.make_rast_light(sc.LIGHT_CAM, light["power"], light["indirect"])
    seed = 4242 + c["seed"]
    try:
        if c["tex"]:
            r.set_textures(tex)
            h.oracle_rast_set_textures(tex, sc.TEX_CAM, h.identity_R(), 0.0)
        if c["colour"]:
            h.oracle().oracle_rast_set_colour_mode(c["colour"])
            r.set_option(b200.OPT_RAST_COLOUR_MODE, c["colour"])
            h.srand(seed)
        want = h.oracle_rast_draw_clipped(W, H, f, h.f32(*sc.LIGHT_CAM), light, t)
        next_rand = h.rand() if c["colour"] else None
        for s in c["strategies"]:
            tag = f"{name} [path {s[0]}, tile {1 << s[1]}]"
            r.set_option(b200.OPT_RAST_PATH, s[0])
            r.set_option(b200.OPT_RAST_TILE_LOG2, s[1])
            launched(capfd)
            if c["colour"]:
                h.srand(seed)
            got = r.render_raster_clipped(t, cam, L)
            if c["colour"]:
                assert h.rand() == next_rand, f"{tag}: the rand() stream ends elsewhere than the oracle's"
            check_kernels(tag, launched(capfd), c, s, d)
            for key in ("index", "depth", "rgb"):
                same(tag, key, got[key], want[key])
            assert r.stats()["fragments"] == want["fragments"], f"{tag}: fragments {r.stats()['fragments']} vs {want['fragments']}"
            if s[0] == 1 and not c["colour"]:
                buf = r.raster_read_buffers(W, H)
                for key in ("screen", "low", "high", "shadow"):
                    same(tag, key, buf[key], want[key])
            if c["colour"]:
                r.rast_upload_clipped(t)
                with pytest.raises(b200.B200Error):     # the fragments are numbered over the whole frame
                    r.rast_render_device(cam, L, 1, H)
                continue
            if not c["bands"]:
                continue
            rgb = torch.full((H, W, 3), 7.0, dtype=torch.float32, device="cuda")
            depth = torch.full((H, W), 7.0, dtype=torch.float32, device="cuda")
            index = torch.full((H, W), -7, dtype=torch.int32, device="cuda")
            r.rast_upload_clipped(t)
            for a, b in band_edges(H)[1:]:
                r.rast_render_device(cam, L, a, b, rgb.data_ptr(), depth.data_ptr(), index.data_ptr())
            r.synchronize()
            launched(capfd)
            btag = f"{tag} bands {band_edges(H)[1:]}"
            same(btag, "index", index.cpu().numpy(), want["index"])
            same(btag, "depth", depth.cpu().numpy(), want["depth"])
            same(btag, "rgb", rgb.cpu().numpy(), want["rgb"])
    finally:
        r.set_option(b200.OPT_RAST_PATH, 0)
        r.set_option(b200.OPT_RAST_TILE_LOG2, 5)
        if c["colour"]:
            r.set_option(b200.OPT_RAST_COLOUR_MODE, 0)
            h.oracle().oracle_rast_set_colour_mode(0)
        if c["tex"]:
            r.set_textures(None)
            h.oracle_rast_set_textures(None)


# ---- pipelined frames whose successor changes class -------------------------------------------------
@pytest.mark.gpu
def test_pipelined_class_changes(b200, tl_renderer, capfd):
    """B200_OPT_RAST_PIPELINED sizes a frame from its verified predecessor of the same shape (list length, band,
    strategy option, tile size).  Lists of one length that cross classes in both directions: no big triangle ->
    big triangles (the scatter path skips the big-triangle kernels, flags the overflow and renders the frame
    again), shadow-free -> shadows (scatter -> ordered tiles), and back; a repeated frame stays pipelined."""
    import torch
    r = tl_renderer
    W, H, f = FRAMES["250x170"]
    light = h.DEFAULT_RAST_LIGHT
    cam = b200.make_camera(sc.TEX_CAM, f, h.identity_R(), W, H)
    L = b200.make_rast_light(sc.LIGHT_CAM, light["power"], light["indirect"])
    n = 3000
    lists = {"tiny": sc.build_list(n, W, H, f, 1, {"tiny": 1}),
             "big": sc.build_list(n, W, H, f, 2, BIG_MIX),
             "shadow": sc.build_list(n, W, H, f, 3, MIXED, shadow=0.25),
             "tiny-shadow": sc.build_list(n, W, H, f, 4, {"tiny": 1}, shadow=0.25)}
    assert not sc.describe(lists["tiny"], W, H, f)["big"].any() and sc.describe(lists["big"], W, H, f)["big"].any()
    # (list, whether the guess from the frame before must fail)
    seq = [("tiny", None), ("tiny", False), ("big", True), ("big", False), ("shadow", True), ("shadow", False),
           ("big", True), ("tiny", False), ("tiny-shadow", True), ("tiny-shadow", False), ("tiny", False)]
    rgb = torch.zeros(H, W, 3, device="cuda")
    depth = torch.zeros(H, W, device="cuda")
    index = torch.zeros(H, W, dtype=torch.int32, device="cuda")
    r.set_option(b200.OPT_RAST_PATH, 0)
    r.set_option(b200.OPT_RAST_PIPELINED, 1)
    try:
        for i, (key, respec) in enumerate(seq):
            t = lists[key]
            before = r.stats()["respeculated"]
            r.rast_upload_clipped(t)
            r.rast_render_device(cam, L, 0, H, rgb.data_ptr(), depth.data_ptr(), index.data_ptr())
            r.synchronize()
            grew = r.stats()["respeculated"] - before
            tag = f"pipelined frame {i} ({key})"
            want = h.oracle_rast_draw_clipped(W, H, f, h.f32(*sc.LIGHT_CAM), light, t)
            same(tag, "index", index.cpu().numpy(), want["index"])
            same(tag, "depth", depth.cpu().numpy(), want["depth"])
            same(tag, "rgb", rgb.cpu().numpy(), want["rgb"])
            assert r.stats()["fragments"] == want["fragments"], tag
            if respec is not None:
                assert (grew > 0) == respec, f"{tag}: respeculated grew by {grew}"
        launched(capfd)
    finally:
        r.set_option(b200.OPT_RAST_PIPELINED, 0)


@pytest.mark.gpu
def test_pipelined_frame_settled_before_host_draw(b200):
    """A pipelined whole-Draw frame that outgrew its guess and is still in flight when a host-pointer Draw (raytraced
    or rasterised) starts on the same context is rendered again before that Draw's rows begin to leave for the
    caller's buffer: nothing is written around the band, the band equals the same Draw on a fresh context, and the
    frame in flight equals its own fresh render."""
    import torch
    W, H, f = 200, 160, 110.0
    soup = h.scene_soup_rast(3000, edge=0.03)
    none = np.zeros(0, h.RAST_TRI)
    light = h.DEFAULT_RAST_LIGHT
    L = b200.make_rast_light(light["pos"], light["power"], light["indirect"])
    far, near = -3.001, 0.2      # far -> near outgrows the guess (test_pipelined_whole_draw_short_and_long)
    cam_at = lambda z: b200.make_camera(h.f32(0.0, 0.0, z, 1.0), f, h.identity_R(), W, H)
    tris, sph = h.golden_cornell_rt()
    rt_cam = b200.make_camera(h.f32(0, 0, -3, 1), 100.0, h.identity_R(), W, H)
    r0, r1, guard, sentinel = 40, 60, H, 0x5A5A5A5A
    argb = torch.zeros(H, W, dtype=torch.int32, device="cuda")
    r, fresh = b200.Renderer(0), b200.Renderer(0)

    def guarded(draw):
        buf = np.full((guard + r1 - r0 + guard, W), sentinel, np.uint32)
        draw(buf.ctypes.data + guard * W * 4)
        assert (buf[:guard] == sentinel).all() and (buf[guard + r1 - r0:] == sentinel).all(), "written outside the band"
        return buf[guard:guard + r1 - r0]

    try:
        fresh.rast_upload_scene(soup, none)
        fresh.rast_draw_device(cam_at(near), L, 0, H, None, None, None, argb.data_ptr())
        fresh.synchronize()
        want_frame = argb.cpu().numpy().copy()
        r.set_option(b200.OPT_RAST_PIPELINED, 1)
        r.rast_upload_scene(soup, none)
        host_draws = (
            (lambda p: r.draw_raytrace_band(tris, sph, rt_cam, h.DEFAULT_RT_LIGHTS, r0, r1, p),
             fresh.draw_raytrace(tris, sph, rt_cam, h.DEFAULT_RT_LIGHTS)[r0:r1]),
            (lambda p: r.draw_raster_band(soup, none, cam_at(far), L, r0, r1, p),
             fresh.draw_raster(soup, none, cam_at(far), L)[r0:r1]))
        for k, (draw, want_band) in enumerate(host_draws):
            for z in (far, far):
                r.rast_draw_device(cam_at(z), L, 0, H, None, None, None, argb.data_ptr())
                r.synchronize()
            before = r.stats()["respeculated"]
            argb.zero_()
            r.rast_draw_device(cam_at(near), L, 0, H, None, None, None, argb.data_ptr())   # in flight, outgrown
            band = guarded(draw)
            assert r.stats()["respeculated"] == before + 1, k
            assert np.array_equal(band, want_band), k
            assert np.array_equal(argb.cpu().numpy(), want_frame), k
    finally:
        r.close()
        fresh.close()


@pytest.mark.gpu
def test_pipelined_whole_draw_short_and_long(b200, tl_renderer, capfd):
    """Whole-Draw frames of one scene whose clipped list crosses 2048 triangles with the camera: the guessed
    list length of a short frame cannot hold the long one (rendered again), the long frame's guess holds a
    short one (launched for the long length, clamped to the short one on the device), repeated frames stay
    pipelined."""
    import torch
    r = tl_renderer
    W, H, f = 200, 160, 110.0
    soup = h.scene_soup_rast(3000, edge=0.03)
    none = np.zeros(0, h.RAST_TRI)
    light = h.DEFAULT_RAST_LIGHT
    L = b200.make_rast_light(light["pos"], light["power"], light["indirect"])
    far, near = (0.0, 0.0, -3.001), (0.0, 0.0, 0.2)
    # far -> near: shorter, but with big triangles (close to the camera) where the far frame had none: rendered again
    seq = [(far, None), (far, False), (near, True), (near, False), (far, True), (far, False)]
    rgb = torch.zeros(H, W, 3, device="cuda")
    depth = torch.zeros(H, W, device="cuda")
    index = torch.zeros(H, W, dtype=torch.int32, device="cuda")
    r.set_option(b200.OPT_RAST_PATH, 0)
    r.rast_upload_scene(soup, none)
    r.set_option(b200.OPT_RAST_PIPELINED, 1)
    try:
        for i, (pos, respec) in enumerate(seq):
            cam_pos = h.f32(*pos, 1.0)
            before = r.stats()["respeculated"]
            r.rast_draw_device(b200.make_camera(cam_pos, f, h.identity_R(), W, H), L, 0, H, rgb.data_ptr(),
                               depth.data_ptr(), index.data_ptr())
            r.synchronize()
            grew = r.stats()["respeculated"] - before
            want = h.oracle_rast_draw(W, H, f, cam_pos, h.identity_R(), light, soup, none)
            tag = f"whole-Draw frame {i} at z = {pos[2]} ({len(want['clipped'])} clipped triangles)"
            assert (len(want["clipped"]) > sc.BITS_MAX_TRIS) == (pos == far), tag
            assert sc.describe(want["clipped"], W, H, f)["big"].any() == (pos == near), tag
            same(tag, "index", index.cpu().numpy(), want["index"])
            same(tag, "depth", depth.cpu().numpy(), want["depth"])
            same(tag, "rgb", rgb.cpu().numpy(), want["rgb"])
            if respec is not None:
                assert (grew > 0) == respec, f"{tag}: respeculated grew by {grew}"
        launched(capfd)
    finally:
        r.set_option(b200.OPT_RAST_PIPELINED, 0)
