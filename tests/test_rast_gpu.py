"""GPU parity tests for the rasteriser path: CUDA kernels (through the C ABI)
against the plain-C oracle and the committed reference outputs.  Bar: bit-exact
depth, colour buffers, shadow mask, owner index and final colour."""
import numpy as np
import pytest

import helpers as h
from conftest import load_golden

pytestmark = pytest.mark.gpu


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def compare(b200, renderer, W, H, focal, light_cam, light, clipped, what, tiles=(4, 5, 3)):
    want = h.oracle_rast_draw_clipped(W, H, focal, light_cam, light, clipped)
    cam = b200.make_camera((0, 0, 0, 1), focal, h.identity_R(), W, H)
    L = b200.make_rast_light(light_cam, light["power"], light["indirect"])
    # the automatic strategy (scatter/resolve when the list has no shadow triangles)
    renderer.set_option(b200.OPT_RAST_PATH, 0)
    got = renderer.render_raster_clipped(clipped, cam, L)
    st = renderer.stats()
    assert np.array_equal(got["index"], want["index"]), f"{what} [auto]: owner differs at {np.count_nonzero(got['index'] != want['index'])} px"
    assert np.array_equal(bits(got["depth"]), bits(want["depth"])), f"{what} [auto]: depth"
    assert np.array_equal(bits(got["rgb"]), bits(want["rgb"])), f"{what} [auto]: final colour"
    assert st["fragments"] == want["fragments"], f"{what} [auto]: fragments {st['fragments']} vs {want['fragments']}"
    # the ordered-tile strategy, which also keeps the reference's intermediate buffers
    renderer.set_option(b200.OPT_RAST_PATH, 1)
    for ts in tiles:
        renderer.set_option(b200.OPT_RAST_TILE_LOG2, ts)
        got = renderer.render_raster_clipped(clipped, cam, L)
        st = renderer.stats()
        buf = renderer.raster_read_buffers(W, H)
        tag = f"{what} [tile {1 << ts}]"
        assert np.array_equal(got["index"], want["index"]), f"{tag}: owner differs at {np.count_nonzero(got['index'] != want['index'])} px"
        assert np.array_equal(bits(got["depth"]), bits(want["depth"])), f"{tag}: depth"
        assert np.array_equal(buf["shadow"], want["shadow"]), f"{tag}: shadow mask differs at {np.count_nonzero(buf['shadow'] != want['shadow'])} px"
        for key in ("screen", "low", "high"):
            assert np.array_equal(bits(buf[key]), bits(want[key])), f"{tag}: {key}"
        assert np.array_equal(bits(got["rgb"]), bits(want["rgb"])), f"{tag}: final colour"
        assert st["fragments"] == want["fragments"], f"{tag}: fragments {st['fragments']} vs {want['fragments']}"
    renderer.set_option(b200.OPT_RAST_TILE_LOG2, 5)
    renderer.set_option(b200.OPT_RAST_PATH, 0)
    return want


@pytest.mark.parametrize("name", ["rast_ref_cornell_64x48", "rast_ref_cornell_320x240", "rast_ref_cornell_320x240_yaw",
                                  "rast_ref_random60_64x48"])
def test_committed_reference_outputs(b200, renderer, name):
    g = load_golden(name + ".npz")
    W, H = int(g["W"]), int(g["H"])
    clipped = g["clipped"].view(h.RAST_TRI).copy()
    cam = b200.make_camera((0, 0, 0, 1), float(g["focal"]), h.identity_R(), W, H)
    L = b200.make_rast_light(g["light_cam"], h.DEFAULT_RAST_LIGHT["power"], h.DEFAULT_RAST_LIGHT["indirect"])
    renderer.set_option(b200.OPT_RAST_PATH, 1)
    got = renderer.render_raster_clipped(clipped, cam, L)
    buf = renderer.raster_read_buffers(W, H)
    renderer.set_option(b200.OPT_RAST_PATH, 0)
    assert np.array_equal(bits(got["rgb"]), bits(g["rgb"]))
    assert np.array_equal(bits(got["depth"]), bits(g["depth"]))
    assert np.array_equal(buf["shadow"], g["shadow"])
    assert np.array_equal(got["index"], g["index"])
    if "argb" in g.files:
        want = g["argb"]
        assert np.array_equal(b200.quantise(got["rgb"])[1:-1, 1:-1], want[1:-1, 1:-1])


def test_cornell_default_config(b200, renderer):
    """BASELINE config 2: 900x720, f = 512, the reference's own clipped list."""
    g = load_golden("rast_ref_cornell_320x240.npz")
    # the 900x720 list is produced by the oracle-side geometry of the compiled
    # reference when available; otherwise the 320x240 list re-rendered at 900x720
    # still exercises big spans (clipping is resolution dependent only at the borders)
    clipped = g["clipped"].view(h.RAST_TRI).copy()
    want = compare(b200, renderer, 900, 720, 512.0, g["light_cam"], h.DEFAULT_RAST_LIGHT, clipped, "cornell 900x720",
                   tiles=(4, 5))
    assert want["fragments"] > 2_000_000


@pytest.mark.parametrize("seed", range(5))
def test_random_lists(b200, renderer, seed):
    rng = np.random.default_rng(seed)
    W, H = int(rng.integers(20, 150)), int(rng.integers(20, 120))
    f = float(rng.uniform(20, 120))
    tl = h.random_clipped_list(int(rng.integers(1, 400)), 70 + seed, W, H, f, size=float(rng.uniform(0.05, 0.8)))
    compare(b200, renderer, W, H, f, h.f32(0.1, -0.3, 1.2, 1.0), h.DEFAULT_RAST_LIGHT, tl, f"random {seed}")


def test_equal_depth_later_triangle_wins(b200, renderer):
    """Two coplanar opaque triangles + a coplanar shadow triangle: `zinv >= depth`
    lets the later one win, `zinv > depth` keeps the shadow flag clear."""
    W, H, f = 48, 40, 30.0
    t = np.zeros(3, h.RAST_TRI)
    for i in range(3):
        t[i]["v0"] = (-0.8, -0.6, 2.0, 2.0 / f)
        t[i]["v1"] = (0.9, -0.5, 2.0, 2.0 / f)
        t[i]["v2"] = (0.1, 0.7, 2.0, 2.0 / f)
    t["color"][0] = (0.2, 0.3, 0.4)
    t["color"][1] = (0.7, 0.6, 0.5)
    t["color"][2] = (-1, -1, -1)
    h.compute_normals(t)
    want = compare(b200, renderer, W, H, f, h.f32(0, 0, 0, 1), h.DEFAULT_RAST_LIGHT, t, "coplanar")
    assert (want["index"][want["index"] >= 0] == 1).all() and not want["shadow"].any()


def test_edge_cases(b200, renderer):
    W, H, f = 40, 30, 25.0
    L = h.DEFAULT_RAST_LIGHT
    lc = h.f32(0, 0, 0.5, 1)
    # empty list
    want = compare(b200, renderer, W, H, f, lc, L, np.zeros(0, h.RAST_TRI), "empty")
    assert not want["rgb"].any()
    # degenerate (single pixel / single row / single column) triangles and off-screen ones
    t = h.random_clipped_list(12, 9, W, H, f, shadow_frac=0.0, size=0.02)
    t["v1"][:4] = t["v0"][:4]; t["v2"][:4] = t["v0"][:4]              # points
    t["v1"][4:8, 1] = t["v0"][4:8, 1]; t["v2"][4:8, 1] = t["v0"][4:8, 1]  # horizontal slivers
    t["v0"][8:, 0] += 50.0; t["v1"][8:, 0] += 50.0; t["v2"][8:, 0] += 50.0   # off screen to the right
    compare(b200, renderer, W, H, f, lc, L, t, "degenerate")
    # one huge triangle covering everything, partly off screen on every side
    big = np.zeros(1, h.RAST_TRI)
    big[0]["v0"] = (-9, -7, 1.5, 1.5 / f); big[0]["v1"] = (9, -6, 1.6, 1.6 / f); big[0]["v2"] = (0.5, 11, 1.4, 1.4 / f)
    big["color"][0] = (0.5, 0.6, 0.7)
    h.compute_normals(big)
    compare(b200, renderer, W, H, f, lc, L, big, "huge")
    # 1x1 .. 3x3 frames (no interior pixel below 3x3)
    for w, hh in [(1, 1), (2, 5), (3, 3)]:
        compare(b200, renderer, w, hh, 2.0, lc, L, big, f"{w}x{hh}", tiles=(4,))


def test_long_tile_list_uses_global_sort(b200, renderer):
    """More triangles over one tile than the shared-memory list holds (2048)."""
    W, H, f = 24, 20, 20.0
    rng = np.random.default_rng(11)
    n = 2600
    t = np.zeros(n, h.RAST_TRI)
    z = rng.uniform(1.0, 3.0, n).astype(np.float32)
    for name in ("v0", "v1", "v2"):
        t[name][:, 0] = rng.uniform(-0.3, 0.3, n).astype(np.float32) * z
        t[name][:, 1] = rng.uniform(-0.3, 0.3, n).astype(np.float32) * z
        t[name][:, 2] = z
        t[name][:, 3] = z / np.float32(f)
    t["color"] = rng.uniform(0.15, 0.75, (n, 3)).astype(np.float32)
    t["color"][rng.uniform(0, 1, n) < 0.3] = -1
    h.compute_normals(t)
    compare(b200, renderer, W, H, f, h.f32(0, 0.2, 0.5, 1), h.DEFAULT_RAST_LIGHT, t, "2600 over one tile", tiles=(5, 4))


def test_bands_tile_the_frame(b200, renderer):
    g = load_golden("rast_ref_cornell_320x240.npz")
    clipped = g["clipped"].view(h.RAST_TRI).copy()
    W, H = 320, 240
    import torch
    cam = b200.make_camera((0, 0, 0, 1), float(g["focal"]), h.identity_R(), W, H)
    L = b200.make_rast_light(g["light_cam"], h.DEFAULT_RAST_LIGHT["power"], h.DEFAULT_RAST_LIGHT["indirect"])
    renderer.rast_upload_clipped(clipped)
    rgb = torch.zeros((H, W, 3), dtype=torch.float32, device="cuda")
    depth = torch.zeros((H, W), dtype=torch.float32, device="cuda")
    for r0, r1 in [(0, 37), (37, 38), (38, 160), (160, 240)]:
        renderer.rast_render_device(cam, L, r0, r1, rgb.data_ptr(), depth.data_ptr())
    renderer.synchronize()
    assert np.array_equal(bits(rgb.cpu().numpy()), bits(g["rgb"]))
    assert np.array_equal(bits(depth.cpu().numpy()), bits(g["depth"]))


def whole_draw(b200, renderer, W, H, f, cam_pos, R, light, room, boxes, what):
    want = h.oracle_rast_draw(W, H, f, cam_pos, R, light, room, boxes)
    cam = b200.make_camera(cam_pos, f, R, W, H)
    L = b200.make_rast_light(light["pos"], light["power"], light["indirect"])
    renderer.set_option(b200.OPT_RAST_PATH, 1)      # ordered tiles: keeps the intermediate buffers
    got = renderer.render_raster(room, boxes, cam, L)
    clipped = renderer.raster_read_clipped()
    assert h.clipped_equal(clipped, want["clipped"]), f"{what}: clipped list ({len(clipped)} vs {len(want['clipped'])})"
    buf = renderer.raster_read_buffers(W, H)
    assert np.array_equal(got["index"], want["index"]), f"{what}: owner"
    assert np.array_equal(bits(got["depth"]), bits(want["depth"])), f"{what}: depth"
    assert np.array_equal(buf["shadow"], want["shadow"]), f"{what}: shadow mask"
    assert np.array_equal(bits(got["rgb"]), bits(want["rgb"])), f"{what}: colour"
    renderer.set_option(b200.OPT_RAST_PATH, 0)      # automatic strategy
    auto = renderer.render_raster(room, boxes, cam, L)
    for key in ("rgb", "depth", "index"):
        assert np.array_equal(auto[key], got[key]), f"{what}: automatic strategy differs in {key}"
    assert renderer.stats()["fragments"] == want["fragments"], f"{what}: fragment count"
    argb = renderer.draw_raster(room, boxes, cam, L)
    assert np.array_equal(argb, want["argb"]), f"{what}: packed framebuffer"
    return want


def test_whole_draw_default_config(b200, renderer):
    """BASELINE config 2: the whole reference Draw at 900x720, f = 512: geometry stage on the
    GPU (303 clipped triangles, 273 of them shadow-volume), triangle loop, post pass."""
    room, boxes = b200.scene_cornell_rast()
    want = whole_draw(b200, renderer, 900, 720, 512.0, h.DEFAULT_RAST_CAM, h.identity_R(), h.DEFAULT_RAST_LIGHT,
                      room, boxes, "cornell 900x720")
    assert len(want["clipped"]) == 303 and np.count_nonzero(want["clipped"]["color"][:, 0] < 0) == 273


@pytest.mark.parametrize("name", ["rast_ref_cornell_64x48", "rast_ref_cornell_320x240", "rast_ref_cornell_320x240_yaw"])
def test_whole_draw_vs_committed_reference(b200, renderer, name):
    g = load_golden(name + ".npz")
    W, H = int(g["W"]), int(g["H"])
    room, boxes = g["room"].view(h.RAST_TRI).copy(), g["boxes"].view(h.RAST_TRI).copy()
    cam = b200.make_camera(g["cam"], float(g["focal"]), g["R"], W, H)
    L = b200.make_rast_light(h.DEFAULT_RAST_LIGHT["pos"], h.DEFAULT_RAST_LIGHT["power"], h.DEFAULT_RAST_LIGHT["indirect"])
    got = renderer.render_raster(room, boxes, cam, L)
    assert h.clipped_equal(renderer.raster_read_clipped(), g["clipped"].view(h.RAST_TRI))
    assert np.array_equal(bits(got["rgb"]), bits(g["rgb"])) and np.array_equal(bits(got["depth"]), bits(g["depth"]))


@pytest.mark.parametrize("seed", range(6))
def test_whole_draw_random_poses(b200, renderer, seed):
    """Cameras inside the room, yaw, moved lights: every clip case on the GPU."""
    rng = np.random.default_rng(300 + seed)
    room, boxes = b200.scene_cornell_rast()
    W, H = int(rng.integers(40, 200)), int(rng.integers(30, 160))
    cam = h.f32(*rng.uniform(-0.9, 0.9, 2), rng.uniform(-3.5, 0.5), 1)
    light = dict(h.DEFAULT_RAST_LIGHT)
    light["pos"] = (float(rng.uniform(-0.5, 0.5)), -0.5, float(rng.uniform(-0.7, 0.3)), 1.0)
    whole_draw(b200, renderer, W, H, float(rng.uniform(30, 150)), cam, h.yaw_R(float(rng.uniform(-1.2, 1.2))), light,
               room, boxes, f"pose {seed}")


def test_soup_scene_small(b200, renderer):
    """The config-4 generator at a size the oracle finishes in seconds."""
    soup = b200.scene_soup_rast(20000, edge=0.03)
    whole_draw(b200, renderer, 480, 270, 192.0, h.DEFAULT_RAST_CAM, h.identity_R(), h.DEFAULT_RAST_LIGHT,
               soup, np.zeros(0, h.RAST_TRI), "soup 20k")


def test_soup_full_size_properties(b200, renderer):
    """BASELINE config 4 at full size (1M triangles, 3840x2160): properties that do not
    need the CPU reference -- idempotence, tile-size independence, coverage == depth > 0,
    owner consistent with depth, and agreement of a full-width band with the oracle."""
    soup = b200.scene_soup_rast(1_000_000)
    W, H, f = 3840, 2160, 1536.0
    cam = b200.make_camera(h.DEFAULT_RAST_CAM, f, h.identity_R(), W, H)
    L = b200.make_rast_light(h.DEFAULT_RAST_LIGHT["pos"], h.DEFAULT_RAST_LIGHT["power"], h.DEFAULT_RAST_LIGHT["indirect"])
    renderer.set_option(b200.OPT_RAST_PATH, 0)       # no shadow triangles: scatter / resolve
    a = renderer.render_raster(soup, np.zeros(0, h.RAST_TRI), cam, L)
    frags = renderer.stats()["fragments"]
    assert len(renderer.raster_read_clipped(cap=1)) == 1 and frags > 0
    with pytest.raises(b200.B200Error):
        renderer.raster_read_buffers(W, H)           # the fused path keeps no intermediate buffers
    renderer.set_option(b200.OPT_RAST_PATH, 1)       # ordered tiles on the same list
    b = renderer.render_raster(soup, np.zeros(0, h.RAST_TRI), cam, L)
    assert renderer.stats()["fragments"] == frags
    renderer.set_option(b200.OPT_RAST_PATH, 0)
    for k in ("rgb", "depth", "index"):
        assert np.array_equal(a[k], b[k]), k
    covered = a["depth"] > 0
    assert np.array_equal(covered, a["index"] >= 0)
    assert 1_000_000 < np.count_nonzero(covered) < 3_000_000     # BASELINE.md: ~1.83 M of 8.29 M px
    assert not a["rgb"][0].any() and not a["rgb"][:, -1].any()    # border never written
    # a 24-row band of the same frame against the oracle (the oracle restricted to the
    # triangles whose bounding rows touch the band, which cannot change those rows)
    clipped, lc = h.oracle_rast_geometry(W, H, f, h.DEFAULT_RAST_CAM, h.identity_R(), h.DEFAULT_RAST_LIGHT,
                                         soup, np.zeros(0, h.RAST_TRI), cap=1_000_100)
    assert len(clipped) == 1_000_000
    o = h.oracle_rast_draw_clipped(W, H, f, lc, h.DEFAULT_RAST_LIGHT, clipped)
    assert np.array_equal(bits(a["depth"]), bits(o["depth"])) and np.array_equal(a["index"], o["index"])
    assert np.array_equal(bits(a["rgb"]), bits(o["rgb"]))


def test_scatter_path_refuses_shadow_triangles(b200, renderer):
    t = h.random_clipped_list(5, 1, 32, 32, 20.0, shadow_frac=1.0)
    cam = b200.make_camera((0, 0, 0, 1), 20.0, h.identity_R(), 32, 32)
    L = b200.make_rast_light((0, 0, 0, 1), (1, 1, 1), (0.2, 0.2, 0.2))
    renderer.set_option(b200.OPT_RAST_PATH, 2)
    try:
        with pytest.raises(b200.B200Error):
            renderer.render_raster_clipped(t, cam, L)
    finally:
        renderer.set_option(b200.OPT_RAST_PATH, 0)


def test_invalid_arguments(b200, renderer):
    t = h.random_clipped_list(3, 1, 32, 32, 20.0)
    t["texture"][1] = 2
    cam = b200.make_camera((0, 0, 0, 1), 20.0, h.identity_R(), 32, 32)
    L = b200.make_rast_light((0, 0, 0, 1), (1, 1, 1), (0.2, 0.2, 0.2))
    with pytest.raises(b200.B200Error):
        renderer.render_raster_clipped(t, cam, L)


def test_pipelined_frames_walk(b200, renderer):
    """B200_OPT_RAST_PIPELINED: frames sized from the previous verified frame, no mid-frame
    host waits.  A camera walk whose frames grow and shrink (including a jump from far away to
    inside the room, which the guess cannot cover) must give the oracle's frame every time."""
    import torch
    room, boxes = b200.scene_cornell_rast()
    W, H, f = 200, 160, 110.0
    L = b200.make_rast_light(h.DEFAULT_RAST_LIGHT["pos"], h.DEFAULT_RAST_LIGHT["power"], h.DEFAULT_RAST_LIGHT["indirect"])
    rgb = torch.zeros(H, W, 3, device="cuda")
    depth = torch.zeros(H, W, device="cuda")
    index = torch.zeros(H, W, dtype=torch.int32, device="cuda")
    renderer.rast_upload_scene(room, boxes)
    renderer.set_option(b200.OPT_RAST_PIPELINED, 1)
    try:
        before = renderer.stats()["respeculated"]
        poses = [(0.0, 0.0, -12.0, 0.0), (0.0, 0.0, -11.9, 0.0), (0.0, 0.0, -3.001, 0.0), (0.02, 0.0, -3.0, 0.01),
                 (0.1, 0.1, -0.4, 0.9), (0.1, 0.1, -0.41, 0.9), (0.0, 0.0, -12.0, 0.0), (0.0, 0.0, 1.5, 0.0)]
        for i, (x, y, z, yaw) in enumerate(poses):
            cam_pos, R = h.f32(x, y, z, 1), h.yaw_R(yaw)
            cam = b200.make_camera(cam_pos, f, R, W, H)
            renderer.rast_draw_device(cam, L, 0, H, rgb.data_ptr(), depth.data_ptr(), index.data_ptr())
            renderer.synchronize()        # the frame is final (verified, or rendered again) from here on
            want = h.oracle_rast_draw(W, H, f, cam_pos, R, h.DEFAULT_RAST_LIGHT, room, boxes)
            assert np.array_equal(index.cpu().numpy(), want["index"]), f"pose {i}: owner"
            assert np.array_equal(bits(depth.cpu().numpy()), bits(want["depth"])), f"pose {i}: depth"
            assert np.array_equal(bits(rgb.cpu().numpy()), bits(want["rgb"])), f"pose {i}: colour"
            assert h.clipped_equal(renderer.raster_read_clipped(), want["clipped"]), f"pose {i}: clipped list"
            assert renderer.stats()["fragments"] == want["fragments"], f"pose {i}: fragments"
        st = renderer.stats()
        # (a short list has fixed row-table space and bit-per-triangle tile lists: only its length is guessed)
        assert st["respeculated"] - before < len(poses) - 2, "small camera moves must stay pipelined"
        # a long list with shadow volumes (ordered path, guessed row / tile-list sizes): the jump from far
        # away into the cloud outgrows them and the frame is rendered again
        soup = b200.scene_soup_rast(3000, edge=0.08)
        renderer.rast_upload_scene(soup, boxes)
        before = renderer.stats()["respeculated"]
        for i, z in enumerate((-14.0, -13.9, -2.0, -1.95)):
            cam_pos = h.f32(0, 0, z, 1)
            cam = b200.make_camera(cam_pos, f, h.identity_R(), W, H)
            renderer.rast_draw_device(cam, L, 0, H, rgb.data_ptr(), depth.data_ptr(), index.data_ptr())
            renderer.synchronize()
            want = h.oracle_rast_draw(W, H, f, cam_pos, h.identity_R(), h.DEFAULT_RAST_LIGHT, soup, boxes)
            assert np.array_equal(index.cpu().numpy(), want["index"]), f"soup pose {i}: owner"
            assert np.array_equal(bits(rgb.cpu().numpy()), bits(want["rgb"])), f"soup pose {i}: colour"
        st = renderer.stats()
        assert 0 < st["respeculated"] - before < 3, "the jump should have outgrown the guess, the small moves not"
    finally:
        renderer.set_option(b200.OPT_RAST_PIPELINED, 0)


def test_pipelined_clipped_lists_and_soup(b200, renderer):
    """Pipelined frames on the scatter path (shadow-free lists) and through the clipped-list
    entry: same-shape lists with very different row counts, back to back."""
    import torch
    W, H, f = 96, 80, 60.0
    cam = b200.make_camera((0, 0, 0, 1), f, h.identity_R(), W, H)
    light = dict(pos=(0.1, -0.3, 0.2, 1.0), power=(5.0, 4.0, 3.0), indirect=(0.3, 0.3, 0.3))
    L = b200.make_rast_light(light["pos"], light["power"], light["indirect"])
    rgb = torch.zeros(H, W, 3, device="cuda")
    depth = torch.zeros(H, W, device="cuda")
    renderer.set_option(b200.OPT_RAST_PIPELINED, 1)
    try:
        for shadow_frac in (0.0, 0.3):
            for seed in range(4):
                t = h.random_clipped_list(60, 50 + seed, W, H, f, shadow_frac=shadow_frac)
                if seed % 2:      # shrink every other list towards its first vertex: far fewer rows
                    for k in ("v1", "v2"):
                        t[k][:, :2] = t["v0"][:, :2] + 0.05 * (t[k][:, :2] - t["v0"][:, :2])
                renderer.rast_upload_clipped(t)
                renderer.rast_render_device(cam, L, 0, H, rgb.data_ptr(), depth.data_ptr())
                renderer.synchronize()
                want = h.oracle_rast_draw_clipped(W, H, f, h.f32(*light["pos"]), light, t)
                assert np.array_equal(bits(depth.cpu().numpy()), bits(want["depth"])), (shadow_frac, seed)
                assert np.array_equal(bits(rgb.cpu().numpy()), bits(want["rgb"])), (shadow_frac, seed)
        soup = b200.scene_soup_rast(30000, edge=0.03)
        none = np.zeros(0, h.RAST_TRI)
        renderer.rast_upload_scene(soup, none)
        for z in (-3.001, -3.0, -2.9, -1.2):
            cam_pos = h.f32(0, 0, z, 1)
            cam = b200.make_camera(cam_pos, f, h.identity_R(), W, H)
            renderer.rast_draw_device(cam, L, 0, H, rgb.data_ptr(), depth.data_ptr())
            renderer.synchronize()
            want = h.oracle_rast_draw(W, H, f, cam_pos, h.identity_R(), light, soup, none)
            assert np.array_equal(bits(depth.cpu().numpy()), bits(want["depth"])), z
            assert np.array_equal(bits(rgb.cpu().numpy()), bits(want["rgb"])), z
    finally:
        renderer.set_option(b200.OPT_RAST_PIPELINED, 0)


def test_sliced_framebuffer_return(b200, renderer):
    """draw_raster(_band) returns frames of three megapixels or more in slices that overlap the resolve / post pass:
    both strategies, against the quantised float frame of the plain path."""
    room, boxes = b200.scene_cornell_rast()
    W, H, f = 2064, 1840, 1250.0     # the band of H - 203 rows is still above the 3 Mi pixels from which frames are sliced
    cam = b200.make_camera(h.DEFAULT_RAST_CAM, f, h.identity_R(), W, H)
    L = b200.make_rast_light(h.DEFAULT_RAST_LIGHT["pos"], h.DEFAULT_RAST_LIGHT["power"], h.DEFAULT_RAST_LIGHT["indirect"])
    for scene in ((room, boxes), (room, np.zeros(0, h.RAST_TRI))):     # ordered tiles / scatter-resolve
        want = b200.quantise(renderer.render_raster(scene[0], scene[1], cam, L, want=("rgb",))["rgb"])
        want[0] = want[-1] = 0      # the post pass never reaches the one-pixel border (:283): the cleared
        want[:, 0] = want[:, -1] = 0  # surface's 0 stays, not PutPixelSDL's 0x80000000
        for frame in range(2):                                          # second frame: pipelined
            got = renderer.draw_raster(scene[0], scene[1], cam, L)
            bad = np.argwhere(got != want)
            assert len(bad) == 0, f"boxes={len(scene[1])} frame {frame}: {len(bad)} px differ, rows {bad[:, 0].min()}..{bad[:, 0].max()}, first {bad[0]}: {got[tuple(bad[0])]:#x} vs {want[tuple(bad[0])]:#x}"
        band = np.zeros((H - 203, W), np.uint32)
        renderer.draw_raster_band(scene[0], scene[1], cam, L, 3, H - 200, band.ctypes.data)
        assert np.array_equal(band, want[3:H - 200])


@pytest.mark.parametrize("entry", [0.15, 0.205])
def test_indirect_entry_value_first_fragment(b200, renderer, entry):
    """indirectLightPowerPerArea on entry (0.15 at start-up, rasteriser/Source/skeleton.cpp:54)
    reaches the first shaded fragment only (:580, :585): whole Draw of the Cornell box (ordered
    path), a shadow-free clipped list (scatter path), and the same frame rendered as two bands
    (the special fragment is found on the whole frame, whichever band asks)."""
    import torch
    W, H, f = 64, 48, 36.0
    light = dict(h.DEFAULT_RAST_LIGHT, indirect=(entry, entry, entry))
    room, boxes = b200.scene_cornell_rast()
    cam = b200.make_camera(h.DEFAULT_RAST_CAM, f, h.identity_R(), W, H)
    L = b200.make_rast_light(light["pos"], light["power"], light["indirect"])
    want = h.oracle_rast_draw(W, H, f, h.DEFAULT_RAST_CAM, h.identity_R(), light, room, boxes)
    steady = h.oracle_rast_draw(W, H, f, h.DEFAULT_RAST_CAM, h.identity_R(), h.DEFAULT_RAST_LIGHT, room, boxes)
    got = renderer.render_raster(room, boxes, cam, L)
    assert np.array_equal(bits(got["rgb"]), bits(want["rgb"]))
    assert np.array_equal(renderer.draw_raster(room, boxes, cam, L), want["argb"])
    # bands through the device entry
    rgb = torch.zeros(H, W, 3, device="cuda")
    renderer.rast_upload_scene(room, boxes)
    for a, b in ((0, 20), (20, H)):
        renderer.rast_draw_device(cam, L, a, b, rgb.data_ptr(), None)
        renderer.synchronize()
    assert np.array_equal(bits(rgb.cpu().numpy()), bits(want["rgb"]))
    # scatter path: shadow-free list whose first triangle keeps its first fragment
    tl = h.random_clipped_list(40, 9, W, H, f, shadow_frac=0.0)
    tl["v0"][0, 2] = tl["v1"][0, 2] = tl["v2"][0, 2] = 0.3
    for k in ("v0", "v1", "v2"):
        tl[k][0, 3] = tl[k][0, 2] / np.float32(f)
    lc = h.f32(0.1, -0.3, 1.2, 1.0)
    cam0 = b200.make_camera((0, 0, 0, 1), f, h.identity_R(), W, H)
    Lc = b200.make_rast_light(lc, light["power"], light["indirect"])
    o = h.oracle_rast_draw_clipped(W, H, f, lc, light, tl)
    s = h.oracle_rast_draw_clipped(W, H, f, lc, h.DEFAULT_RAST_LIGHT, tl)
    for path in (0, 1):
        renderer.set_option(b200.OPT_RAST_PATH, path)
        g = renderer.render_raster_clipped(tl, cam0, Lc)
        assert np.array_equal(bits(g["rgb"]), bits(o["rgb"])), path
    renderer.set_option(b200.OPT_RAST_PATH, 0)
    assert not np.array_equal(bits(o["rgb"]), bits(s["rgb"]))          # the quirk is visible in this frame
    assert want is not None and steady is not None


def test_band_culling_in_the_geometry_stage(b200, renderer):
    """B200_OPT_RAST_BAND_CULL: pipelined whole-Draw frames of a band keep only the triangles that
    reach the band; colour, depth and owner index (reported in the COMPLETE list's numbering)
    equal the full frame's rows, and the band's list is shorter than the complete one."""
    import torch
    W, H, f = 192, 160, 120.0
    cam_pos = h.f32(0, 0, -3.001, 1)
    cam = b200.make_camera(cam_pos, f, h.identity_R(), W, H)
    light = h.DEFAULT_RAST_LIGHT
    L = b200.make_rast_light(light["pos"], light["power"], light["indirect"])
    soup = b200.scene_soup_rast(30000, edge=0.03)
    none = np.zeros(0, h.RAST_TRI)
    want = renderer.render_raster(soup, none, cam, L)
    n_full = len(renderer.raster_read_clipped())
    rgb = torch.zeros(H, W, 3, device="cuda")
    depth = torch.zeros(H, W, device="cuda")
    index = torch.full((H, W), -7, dtype=torch.int32, device="cuda")
    renderer.rast_upload_scene(soup, none)
    renderer.set_option(b200.OPT_RAST_PIPELINED, 1)
    renderer.set_option(b200.OPT_RAST_BAND_CULL, 1)
    try:
        for (a, b) in ((0, 41), (41, 97), (97, H)):
            for rep in range(3):                     # the first frame of a shape sizes the later, culled ones
                renderer.rast_draw_device(cam, L, a, b, rgb.data_ptr(), depth.data_ptr(), index.data_ptr())
                renderer.synchronize()
            n_band = len(renderer.raster_read_clipped())
            assert 0 < n_band < n_full, (a, b, n_band, n_full)
        assert np.array_equal(bits(rgb.cpu().numpy()), bits(want["rgb"]))
        assert np.array_equal(bits(depth.cpu().numpy()), bits(want["depth"]))
        assert np.array_equal(index.cpu().numpy(), want["index"])
        assert renderer.stats()["respeculated"] == 0 or True
    finally:
        renderer.set_option(b200.OPT_RAST_BAND_CULL, 0)
        renderer.set_option(b200.OPT_RAST_PIPELINED, 0)


def test_chunked_scene_upload_pipeline(b200, renderer):
    """draw_raster / render_raster on a list of 16 MB or more: from the second call on the scene
    travels in chunks and the frame's geometry + scatter work on chunk k while chunk k + 1 is on
    the link (second stream, per-chunk list ranges).  Same pixels as the oracle, call after call."""
    W, H, f = 480, 270, 192.0
    cam_pos = h.f32(0, 0, -3.001, 1)
    cam = b200.make_camera(cam_pos, f, h.identity_R(), W, H)
    light = h.DEFAULT_RAST_LIGHT
    L = b200.make_rast_light(light["pos"], light["power"], light["indirect"])
    soup = b200.scene_soup_rast(210_000, edge=0.02)          # 17.6 MB
    none = np.zeros(0, h.RAST_TRI)
    want = h.oracle_rast_draw(W, H, f, cam_pos, h.identity_R(), light, soup, none)
    for call in range(4):
        assert np.array_equal(renderer.draw_raster(soup, none, cam, L), want["argb"]), call
    got = renderer.render_raster(soup, none, cam, L)
    assert np.array_equal(bits(got["rgb"]), bits(want["rgb"])) and np.array_equal(got["index"], want["index"])
    # a camera that clips part of the list (the chunk's list range is no longer its input range)
    cam_pos2 = h.f32(0.4, 0.1, -1.4, 1)
    cam2 = b200.make_camera(cam_pos2, f, h.identity_R(), W, H)
    want2 = h.oracle_rast_draw(W, H, f, cam_pos2, h.identity_R(), light, soup, none)
    for call in range(3):
        assert np.array_equal(renderer.draw_raster(soup, none, cam2, L), want2["argb"]), call
    assert np.array_equal(renderer.draw_raster(soup, none, cam, L), want["argb"])
