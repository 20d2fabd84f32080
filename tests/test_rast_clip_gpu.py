"""The rasteriser's geometry stage (camera transform, shadow volumes, rotation, six-plane clip: Draw :205-241)
against the plain-C oracle, bit for bit, on scenes aimed at every branch of the clip (tests/rast_clip_cases.py).

Without a GPU: the oracle's clip census (oracle_rast_clip_census) shows that the cases reach every branch of every
plane, vertices exactly on each limit, NaN drops and a triangle with more than 16 descendants; where the compiled
reference is built, the oracle's clipped list and frame equal the reference's on the cases of its frame sizes.

On the GPU each case goes through every geometry kernel it can reach, checked from the launch timeline
(B200_TIMELINE): rast_geom_kernel's count / scan / write (frames that are not pipelined), rast_geom_warp_kernel
(pipelined, shadow volumes, up to 8192 pre-clip triangles), rast_geom_kernel<2> (pipelined with shadow volumes past
8192, and shadow-free frames, whose geometry kernel also clears the scatter path's keys, whole or culled to a band,
and in chunks behind a large upload).  The clipped list (raster_read_clipped) is compared byte for byte, and so are
colour, depth, owner index and fragments, which read the camera-space light.  Every case's list converts to pixel
positions -- the far-plane cases at W = 32768 with a vertex 5.25e7 pixels off screen, which the triangle loop draws
as the reference does.
"""
import os
import re

import numpy as np
import pytest

import helpers as h
import rast_clip_cases as cc

REFERENCE_FRAMES = ("64x48", "320x240")


# ---------------------------------------------------------------------------------------------
# without a GPU
# ---------------------------------------------------------------------------------------------
def test_census_reaches_every_branch():
    census, desc = cc.oracle_census()
    missing = [k for k, v in census.items() if v == 0]
    assert not missing, f"clip branches no case reaches: {missing}"
    assert np.nonzero(desc)[0].max() >= 17, f"descendants per pre-clip triangle: {desc}"
    assert desc[0] > 0 and desc[1] > 0 and desc[2] > 0


def test_cases_have_what_they_are_named_for():
    seen = set()
    for c in cc.CASES:
        room, boxes, W, H, f, cam, R, light = cc.build(c)
        n_pre = cc.n_pre(room, boxes)
        cc.census_read(reset=True)
        clipped, lc = cc.oracle_geometry(W, H, f, cam, R, light, room, boxes)
        census, desc = cc.census_read(reset=True)
        assert cc.convertible(clipped, W, H, f).all(), c["name"]       # the triangle loop runs on every list
        assert c["shadow"] == bool(len(boxes)) and c["large"] == (n_pre > cc.GEOM_WARP_MAX_PRE), c["name"]
        if W % 2 or H % 2:
            seen.add("odd frame")
        if len(room) > 128 and len(room) % 128:
            seen.add("more than 128 room triangles, not a multiple of 128")
        if n_pre > cc.GEOM_WARP_MAX_PRE:
            seen.add("shadows past 8192" if len(boxes) else "shadow-free past 8192")
        if len(boxes) and n_pre <= cc.GEOM_WARP_MAX_PRE:
            seen.add("shadows up to 8192")
            if desc[17:].any():                               # lanes above 16 of rast_geom_warp_kernel
                seen.add("17 or more descendants on the warp kernel")
        if not len(boxes):
            seen.add("shadow-free")
        if not len(boxes) and room.nbytes >= cc.FAST_PIPE_BYTES:
            seen.add("chunked upload")
        Rm = np.asarray(R, np.float32).reshape(4, 4)          # glm column-major: Rm[c, r]
        if Rm[3, :3].any():
            seen.add("translation column")
        if Rm[1, 2] != 0 and Rm[0, 1] != 0:                   # rotation about x and z as well as y
            seen.add("yaw, pitch and roll")
        if census["t_param denominator exactly 0"]:
            seen.add("zero t_param denominator")
        V = np.stack([clipped[k] for k in ("v0", "v1", "v2")], 1)
        assert np.isfinite(V).all(), c["name"]                     # (no NaN or inf vertex reaches any list)
        with np.errstate(all="ignore"):
            px = (np.float32(f) * (V[..., 0] / V[..., 2]).astype(np.float32)).astype(np.float32) + np.float32(W // 2)
        if np.abs(px).max() > 2 ** 24:                              # (float32 no longer holds every integer)
            seen.add("vertex tens of millions of pixels off screen" + (", shadows" if len(boxes) else ""))
        nan_normals = np.isnan(clipped["normal"]).any(1)
        if nan_normals.any():
            assert (clipped["normal"][nan_normals][:, :3].view(np.uint32) == 0xffc00000).all(), c["name"]
            assert (clipped["color"][nan_normals] < 0).all(), c["name"]     # only shadow-volume sides
            seen.add("NaN shadow normals")
    assert seen == {"odd frame", "more than 128 room triangles, not a multiple of 128", "shadows past 8192",
                    "shadow-free past 8192", "shadows up to 8192", "shadow-free", "chunked upload",
                    "translation column", "yaw, pitch and roll", "NaN shadow normals",
                    "17 or more descendants on the warp kernel", "zero t_param denominator",
                    "vertex tens of millions of pixels off screen",
                    "vertex tens of millions of pixels off screen, shadows"}, seen
    assert cc.oracle_census([cc.BY_NAME["zero_denominator_37x23"]])[0]["t_param denominator exactly 0"] > 0


@pytest.mark.parametrize("name", [c["name"] for c in cc.CASES if c["frame"] in REFERENCE_FRAMES and not c["large"]])
def test_oracle_vs_compiled_reference(name):
    W, H = (int(x) for x in cc.BY_NAME[name]["frame"].split("x"))
    if not h.have_ref(h.ref_rast_name(W, H)):
        pytest.skip("oracle/_ref not built")
    room, boxes, W, H, f, cam, R, light = cc.build(cc.BY_NAME[name])
    r = h.ref_rast_draw(W, H, f, cam, R, light, room, boxes)
    clipped, lc = cc.oracle_geometry(W, H, f, cam, R, light, room, boxes)
    assert h.clipped_equal(clipped, r["clipped"])
    assert np.array_equal(bits(lc), bits(r["light_cam"]))
    o = h.oracle_rast_draw_clipped(W, H, f, lc, light, clipped)
    for key in ("rgb", "depth", "low", "high"):
        assert np.array_equal(bits(o[key]), bits(r[key])), key
    assert np.array_equal(o["shadow"], r["shadow"]) and np.array_equal(o["argb"], r["argb"])


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


def same_list(tag, got, want):
    """Byte equality of two clipped lists; the first differing triangle and field on failure."""
    if len(got) != len(want):
        raise AssertionError(f"{tag}: clipped list of {len(got)} triangles, the oracle's has {len(want)}")
    g, w = (np.ascontiguousarray(a).view(np.uint8).reshape(len(a), h.RAST_TRI.itemsize) for a in (got, want))
    bad = np.nonzero((g != w).any(1))[0]
    if len(bad):
        i = bad[0]
        fields = [k for k in h.RAST_TRI.names if got[k][i].tobytes() != want[k][i].tobytes()]
        raise AssertionError(f"{tag}: {len(bad)} clipped triangles differ, first #{i} in {fields}: "
                             + "; ".join(f"{k} {got[k][i].view(np.uint32)} vs {want[k][i].view(np.uint32)}"
                                         if got[k].dtype == np.float32 else f"{k} {got[k][i]} vs {want[k][i]}"
                                         for k in fields))


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


TL = re.compile(r"^\[b200 timeline\] (.+?)\s+-?[0-9.]+ us$")


def launched(capfd):
    names = []
    for line in capfd.readouterr().err.splitlines():
        m = TL.match(line.strip())
        if m and m.group(1) != "frame":
            names.append(m.group(1))
    return names


GEOM = ("rast_geom_kernel", "rast_geom_warp_kernel", "rast_geom_kernel<2>")


def check_geom(tag, names, kernel):
    """`kernel` is the one geometry kernel of the frame (count / scan / write for "rast_geom_kernel")."""
    ran = [k for k in GEOM if k in names]
    assert ran == [kernel], f"{tag}: geometry kernels {ran} ran, expected {kernel} ({names})"
    if kernel == "rast_geom_kernel":
        assert names.count("rast_geom_kernel") == 2 and "scan_apply_kernel" in names, f"{tag}: {names}"


_want = {}


def want_of(name):
    """The case's scene, the oracle's geometry stage and its frame (cached)."""
    if name not in _want:
        c = cc.BY_NAME[name]
        room, boxes, W, H, f, cam, R, light = cc.build(c)
        clipped, lc = cc.oracle_geometry(W, H, f, cam, R, light, room, boxes)
        assert cc.convertible(clipped, W, H, f).all(), name
        frame = h.oracle_rast_draw_clipped(W, H, f, lc, light, clipped)
        _want[name] = dict(room=room, boxes=boxes, W=W, H=H, f=f, cam=cam, R=R, light=light, clipped=clipped,
                           light_cam=lc, frame=frame)
    return _want[name]


def check_frame(tag, r, w, rgb, depth, index):
    same(tag, "index", index, w["frame"]["index"])
    same(tag, "depth", depth, w["frame"]["depth"])
    same(tag, "rgb", rgb, w["frame"]["rgb"])
    assert r.stats()["fragments"] == w["frame"]["fragments"], f"{tag}: fragments {r.stats()['fragments']} vs {w['frame']['fragments']}"


def collapsed(w):
    """The case's scene with every vertex moved onto the camera: the same shape (room and box counts), a far
    shorter list."""
    out = []
    for t in (w["room"], w["boxes"]):
        t = t.copy()
        for k in ("v0", "v1", "v2"):
            t[k][:, :3] = w["cam"][:3]
        out.append(t)
    return out


def lights(b200, w):
    return b200.make_rast_light(w["light"]["pos"], w["light"]["power"], w["light"]["indirect"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c["name"] for c in cc.CASES])
def test_not_pipelined(b200, tl_renderer, capfd, name):
    """render_raster on the ordered path: rast_geom_kernel count / scan / write, the ordered tiles' buffers."""
    r, w = tl_renderer, want_of(name)
    W, H = w["W"], w["H"]
    cam = b200.make_camera(w["cam"], w["f"], w["R"], W, H)
    r.set_option(b200.OPT_RAST_PIPELINED, 0)
    r.set_option(b200.OPT_RAST_PATH, 1)
    try:
        launched(capfd)
        got = r.render_raster(w["room"], w["boxes"], cam, lights(b200, w))
        check_geom(name, launched(capfd), "rast_geom_kernel")
        same_list(name, r.raster_read_clipped(), w["clipped"])
        check_frame(name, r, w, got["rgb"], got["depth"], got["index"])
        buf = r.raster_read_buffers(W, H)
        for key in ("screen", "low", "high", "shadow"):
            same(name, key, buf[key], w["frame"][key])
    finally:
        r.set_option(b200.OPT_RAST_PATH, 0)
        r.set_option(b200.OPT_RAST_PIPELINED, 0)


def pipelined_kernel(w):
    """rast_geometry's choice for a whole pipelined frame: rast_geom_kernel<2> past 8192 pre-clip triangles, and on a
    shadow-free frame whose key rows it can clear (in 16-byte units: W * H even); the warp kernel otherwise."""
    shadow = len(w["boxes"]) > 0 or (w["room"]["color"][:, 0] < 0).any()
    clear = not shadow and (w["W"] * w["H"]) % 2 == 0
    return "rast_geom_warp_kernel" if cc.n_pre(w["room"], w["boxes"]) <= cc.GEOM_WARP_MAX_PRE and not clear \
        else "rast_geom_kernel<2>"


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c["name"] for c in cc.CASES if c["name"] != "chunked_upload_320x240"])
def test_pipelined(b200, tl_renderer, capfd, name):
    """rast_draw_device with B200_OPT_RAST_PIPELINED: the case, again (its own length guessed), the same scene
    collapsed onto the camera (a guess far too long), and the case once more (a guess that a list of more than
    ~1000 triangles outgrows: rendered again without pipelining)."""
    import torch
    r, w = tl_renderer, want_of(name)
    W, H, f = w["W"], w["H"], w["f"]
    cam = b200.make_camera(w["cam"], f, w["R"], W, H)
    L = lights(b200, w)
    small = collapsed(w)
    small_list, _ = cc.oracle_geometry(W, H, f, w["cam"], w["R"], w["light"], *small)
    assert len(small_list) < len(w["clipped"]), name
    kernel = pipelined_kernel(w)
    rgb = torch.zeros(H, W, 3, device="cuda")
    depth = torch.zeros(H, W, device="cuda")
    index = torch.zeros(H, W, dtype=torch.int32, device="cuda")
    r.set_option(b200.OPT_RAST_PATH, 0)
    r.set_option(b200.OPT_RAST_PIPELINED, 1)
    try:
        # (scene, whether the frame must be rendered again): the last frame's list outgrows the guess from the
        # collapsed one when it is longer than rast_spec_cap.  The ordered path's row and tile guesses may send a
        # frame round again as well (the second frame of some shadowed cases); such a frame must then have been
        # rendered by count / scan / write, any other by the pipelined kernel.
        outgrows = len(w["clipped"]) > len(small_list) + len(small_list) // 32 + 1024
        seq = [("case", None), ("case", None), ("collapsed", False), ("case", True if outgrows else None)]
        for i, (what, respec) in enumerate(seq):
            scene = (w["room"], w["boxes"]) if what == "case" else small
            tag = f"{name} frame {i} ({what})"
            r.rast_upload_scene(*scene)
            before = r.stats()["respeculated"]
            launched(capfd)
            r.rast_draw_device(cam, L, 0, H, rgb.data_ptr(), depth.data_ptr(), index.data_ptr())
            r.synchronize()
            names = launched(capfd)
            grew = r.stats()["respeculated"] - before
            if respec is not None:
                assert (grew > 0) == respec, f"{tag}: respeculated grew by {grew}"
            check_geom(tag, names, "rast_geom_kernel" if i == 0 or grew else kernel)
            same_list(tag, r.raster_read_clipped(), w["clipped"] if what == "case" else small_list)
            if what == "case":
                check_frame(tag, r, w, rgb.cpu().numpy(), depth.cpu().numpy(), index.cpu().numpy())
    finally:
        r.set_option(b200.OPT_RAST_PIPELINED, 0)


def band_edges(H):
    a, b = H // 3 + 1, (2 * H) // 3 - 1
    return [(0, a), (a, b), (b, H)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c["name"] for c in cc.CASES if c["name"] != "chunked_upload_320x240"
                                  and not c["shadow"]])
def test_band_culled(b200, tl_renderer, capfd, name):
    """Shadow-free pipelined frames of three bands with B200_OPT_RAST_BAND_CULL: rast_geom_kernel<2> keeps the
    triangles whose truncated vertex rows meet the band widened by two rows (the oracle's list filtered by that
    rule, restated in float32), and the bands make up the oracle's frame, owner indices in the complete list."""
    import torch
    r, w = tl_renderer, want_of(name)
    W, H, f = w["W"], w["H"], w["f"]
    cam = b200.make_camera(w["cam"], f, w["R"], W, H)
    L = lights(b200, w)
    ok, ymin, ymax = cc.band_rows(w["clipped"], H, f)
    rgb = torch.full((H, W, 3), 7.0, device="cuda")
    depth = torch.full((H, W), 7.0, device="cuda")
    index = torch.full((H, W), -7, dtype=torch.int32, device="cuda")
    r.set_option(b200.OPT_RAST_PATH, 0)
    r.rast_upload_scene(w["room"], w["boxes"])
    r.set_option(b200.OPT_RAST_PIPELINED, 1)
    r.set_option(b200.OPT_RAST_BAND_CULL, 1)
    try:
        for a, b in band_edges(H):
            fb0, fb1 = max(a - 2, 0), min(b + 2, H)
            keep = ok & (ymax >= fb0) & (ymin < fb1)
            for rep in range(2):                     # the first frame of a band sizes the second, culled one
                tag = f"{name} band [{a}, {b}) frame {rep}"
                before = r.stats()["respeculated"]
                launched(capfd)
                r.rast_draw_device(cam, L, a, b, rgb.data_ptr(), depth.data_ptr(), index.data_ptr())
                r.synchronize()
                names = launched(capfd)
                if rep:
                    assert r.stats()["respeculated"] == before, tag
                    check_geom(tag, names, "rast_geom_kernel<2>")
                    same_list(tag, r.raster_read_clipped(), w["clipped"][keep])
        same(name, "index", index.cpu().numpy(), w["frame"]["index"])
        same(name, "depth", depth.cpu().numpy(), w["frame"]["depth"])
        same(name, "rgb", rgb.cpu().numpy(), w["frame"]["rgb"])
    finally:
        r.set_option(b200.OPT_RAST_BAND_CULL, 0)
        r.set_option(b200.OPT_RAST_PIPELINED, 0)


@pytest.mark.gpu
def test_chunked_upload(b200, tl_renderer, capfd):
    """draw_raster on a shadow-free scene of 16 MB or more: from the second call on, the scene travels in chunks
    and rast_geom_kernel<2> runs once per chunk behind its copy."""
    name = "chunked_upload_320x240"
    r, w = tl_renderer, want_of(name)
    assert w["room"].nbytes >= cc.FAST_PIPE_BYTES and not len(w["boxes"])
    W, H, f = w["W"], w["H"], w["f"]
    cam = b200.make_camera(w["cam"], f, w["R"], W, H)
    r.set_option(b200.OPT_RAST_PATH, 0)
    for call in range(3):
        tag = f"{name} call {call}"
        launched(capfd)
        argb = r.draw_raster(w["room"], w["boxes"], cam, lights(b200, w))
        check_geom(tag, launched(capfd), "rast_geom_kernel" if call == 0 else "rast_geom_kernel<2>")
        same(tag, "argb", argb, w["frame"]["argb"])
        same_list(tag, r.raster_read_clipped(), w["clipped"])
