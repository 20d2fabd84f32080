"""CPU tests: pin the plain-C rasteriser oracle against KAT #1, the committed
outputs of the compiled reference, and (when present) the compiled reference."""
import ctypes
import os

import numpy as np
import pytest

import helpers as h
from conftest import load_golden


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


# rasteriser/Instructions/instructions.pdf, "ComputePolygonRows ... should give
# the output" (the commented-out test at rasteriser/Source/skeleton.cpp:183-199)
KAT1 = [(10, 5, 10, 5), (9, 6, 10, 6), (8, 7, 11, 7), (7, 8, 11, 8), (6, 9, 12, 9), (5, 10, 12, 10),
        (7, 11, 13, 11), (9, 12, 13, 12), (11, 13, 14, 13), (13, 14, 14, 14), (15, 15, 15, 15)]


def test_kat1_compute_polygon_rows():
    lib = h.oracle()
    xy = np.array([10, 5, 5, 10, 15, 15], np.int32)
    y0, n = h.c_i(), h.c_i()
    lx, rx = np.zeros(64, np.int32), np.zeros(64, np.int32)
    assert lib.oracle_rast_polygon_rows_kat(h.ptr(xy), ctypes.byref(y0), ctypes.byref(n), h.ptr(lx), h.ptr(rx), 64) == 0
    got = [(int(lx[r]), y0.value + r, int(rx[r]), y0.value + r) for r in range(n.value)]
    assert got == KAT1


@pytest.mark.parametrize("name", ["rast_ref_cornell_64x48", "rast_ref_cornell_320x240", "rast_ref_cornell_320x240_yaw",
                                  "rast_ref_random60_64x48"])
def test_oracle_matches_committed_reference_outputs(name):
    g = load_golden(name + ".npz")
    W, H = int(g["W"]), int(g["H"])
    clipped = g["clipped"].view(h.RAST_TRI)
    o = h.oracle_rast_draw_clipped(W, H, float(g["focal"]), g["light_cam"], h.DEFAULT_RAST_LIGHT, clipped)
    for key in ("rgb", "depth", "low", "high", "screen_post"):
        if key in g.files:
            assert np.array_equal(bits(o[key]), bits(g[key])), key
    if "screen" in g.files and g["screen"].size:
        assert np.array_equal(bits(o["screen"]), bits(g["screen"]))
    assert np.array_equal(o["shadow"], g["shadow"])
    assert np.array_equal(o["index"], g["index"])
    if "argb" in g.files:
        assert np.array_equal(o["argb"], g["argb"])


def test_rows_vs_compiled_reference():
    if not h.have_ref(h.ref_rast_name(64, 48)):
        pytest.skip("oracle/_ref not built")
    ref = h.ref_lib(h.ref_rast_name(64, 48))
    lib = h.oracle()
    rng = np.random.default_rng(3)
    for _ in range(500):
        v = np.zeros((3, 4), np.float32)
        v[:, :2] = rng.uniform(-1.5, 1.5, (3, 2))
        v[:, 2] = rng.uniform(0.3, 3, 3)
        v[:, 3] = 1
        a = h.rows_call(ref.ref_rast_rows, 40.0, v)
        b = h.rows_call(lib.oracle_rast_rows, 40.0, v, dims=(64, 48))
        assert a[0] == b[0] and a[1].shape == b[1].shape
        assert np.array_equal(bits(a[1]), bits(b[1]))


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_oracle_vs_compiled_reference_random_lists(seed):
    if not h.have_ref(h.ref_rast_name(64, 48)):
        pytest.skip("oracle/_ref not built")
    W, H, f = 64, 48, 40.0
    tl = h.random_clipped_list(80 + 40 * seed, 50 + seed, W, H, f, size=0.3 + 0.3 * seed)
    lc = h.f32(0.1, -0.3, 1.2, 1.0)
    r = h.ref_rast_draw_clipped(W, H, f, lc, h.DEFAULT_RAST_LIGHT, tl)
    o = h.oracle_rast_draw_clipped(W, H, f, lc, h.DEFAULT_RAST_LIGHT, tl)
    for key in ("rgb", "depth", "low", "high", "screen"):
        assert np.array_equal(bits(o[key]), bits(r[key])), key
    assert np.array_equal(o["shadow"], r["shadow"]) and np.array_equal(o["index"], r["index"])
    assert np.array_equal(o["argb"], r["argb"])


@pytest.mark.parametrize("name", ["rast_ref_cornell_64x48", "rast_ref_cornell_320x240", "rast_ref_cornell_320x240_yaw"])
def test_geometry_matches_committed_clipped_lists(name):
    """Geometry stage (camera transform, shadow volumes, rotation, six-plane clip)
    against the clipped list the compiled reference built (committed)."""
    g = load_golden(name + ".npz")
    room, boxes = g["room"].view(h.RAST_TRI), g["boxes"].view(h.RAST_TRI)
    clipped, lc = h.oracle_rast_geometry(int(g["W"]), int(g["H"]), float(g["focal"]), g["cam"], g["R"],
                                         h.DEFAULT_RAST_LIGHT, room, boxes)
    assert h.clipped_equal(clipped, g["clipped"].view(h.RAST_TRI))
    assert np.array_equal(bits(lc), bits(g["light_cam"]))


@pytest.mark.parametrize("seed", range(8))
def test_geometry_vs_compiled_reference_random_poses(seed):
    """Cameras inside the room, yaw, moved lights: every clip case gets exercised."""
    if not h.have_ref(h.ref_rast_name(320, 240)):
        pytest.skip("oracle/_ref not built")
    W, H, f = (320, 240, 170.0) if seed % 2 else (64, 48, 36.0)
    rng = np.random.default_rng(200 + seed)
    room, boxes = h.ref_rast_testmodel(W, H)
    cam = h.f32(*rng.uniform(-0.9, 0.9, 2), rng.uniform(-3.5, 0.5), 1)
    R = h.yaw_R(float(rng.uniform(-1.2, 1.2)))
    light = dict(h.DEFAULT_RAST_LIGHT)
    light["pos"] = (float(rng.uniform(-0.5, 0.5)), -0.5, float(rng.uniform(-0.7, 0.3)), 1.0)
    r = h.ref_rast_draw(W, H, f, cam, R, light, room, boxes)
    clipped, lc = h.oracle_rast_geometry(W, H, f, cam, R, light, room, boxes)
    assert h.clipped_equal(clipped, r["clipped"])
    assert np.array_equal(bits(lc), bits(r["light_cam"]))
    o = h.oracle_rast_draw(W, H, f, cam, R, light, room, boxes)
    assert np.array_equal(bits(o["rgb"]), bits(r["rgb"])) and np.array_equal(o["shadow"], r["shadow"])


def test_whole_draw_default_config():
    """BASELINE config 2: 900x720, f = 512: 303 clipped triangles, the fragment count
    SURVEY.md quotes, and the oracle equal to the reference's whole Draw."""
    if not h.have_ref(h.ref_rast_name(900, 720)):
        pytest.skip("oracle/_ref not built")
    room, boxes = h.ref_rast_testmodel(900, 720)
    r = h.ref_rast_draw(900, 720, 512.0, h.DEFAULT_RAST_CAM, h.identity_R(), h.DEFAULT_RAST_LIGHT, room, boxes)
    assert len(r["clipped"]) == 303
    o = h.oracle_rast_draw_clipped(900, 720, 512.0, r["light_cam"], h.DEFAULT_RAST_LIGHT, r["clipped"])
    assert np.array_equal(bits(o["rgb"]), bits(r["rgb"])) and np.array_equal(o["argb"], r["argb"])
    assert np.array_equal(bits(o["depth"]), bits(r["depth"])) and np.array_equal(o["shadow"], r["shadow"])
    assert not o["rgb"][0].any() and not o["rgb"][:, 0].any()   # border never written


@pytest.mark.parametrize("entry", [0.15, 0.205, 0.0])
def test_indirect_entry_value_reaches_only_the_first_shaded_fragment(entry):
    """indirectLightPowerPerArea is a global that PixelShader leaves at 0.2 (:585): the value it
    has when Draw is entered (0.15 at start-up :54, 0.2 +- 0.005 after keys 1 / 2) is seen by
    the first shaded fragment only.  Oracle == the reference's own Draw, whole frame and
    every intermediate buffer; and the frame differs from the steady-state one in at most
    that fragment's pixel (before the post pass spreads it over its 5-tap neighbours)."""
    if not h.have_ref(h.ref_rast_name(64, 48)):
        pytest.skip("oracle/_ref not built")
    W, H, f = 64, 48, 36.0
    light = dict(h.DEFAULT_RAST_LIGHT, indirect=(entry, entry, entry))
    room, boxes = h.ref_rast_testmodel(W, H)
    r = h.ref_rast_draw(W, H, f, h.DEFAULT_RAST_CAM, h.identity_R(), light, room, boxes)
    o = h.oracle_rast_draw(W, H, f, h.DEFAULT_RAST_CAM, h.identity_R(), light, room, boxes)
    assert np.array_equal(bits(o["rgb"]), bits(r["rgb"])) and np.array_equal(o["argb"], r["argb"])
    assert np.array_equal(bits(o["low"]), bits(r["low"])) and np.array_equal(bits(o["high"]), bits(r["high"]))
    steady = h.oracle_rast_draw(W, H, f, h.DEFAULT_RAST_CAM, h.identity_R(), h.DEFAULT_RAST_LIGHT, room, boxes)
    assert np.count_nonzero((bits(o["screen"]) != bits(steady["screen"])).any(axis=-1)) <= 1
    # a random clipped list whose first triangle survives at its first fragment's pixel
    tl = h.random_clipped_list(40, 9, W, H, f, shadow_frac=0.2)
    tl["v0"][0, 2] = tl["v1"][0, 2] = tl["v2"][0, 2] = 0.3          # nearest: keeps its pixels
    for k in ("v0", "v1", "v2"):
        tl[k][0, 3] = tl[k][0, 2] / np.float32(f)
    tl["color"][0] = (0.4, 0.5, 0.6)
    lc = h.f32(0.1, -0.3, 1.2, 1.0)
    r = h.ref_rast_draw_clipped(W, H, f, lc, light, tl)
    o = h.oracle_rast_draw_clipped(W, H, f, lc, light, tl)
    s = h.oracle_rast_draw_clipped(W, H, f, lc, h.DEFAULT_RAST_LIGHT, tl)
    for key in ("rgb", "screen", "low", "high", "depth"):
        assert np.array_equal(bits(o[key]), bits(r[key])), key
    assert np.count_nonzero((bits(o["screen"]) != bits(s["screen"])).any(axis=-1)) == 1


# ---- texture branches (rasteriser/Source/skeleton.cpp:588-645, findU / findV :1756-1825) ----
@pytest.mark.parametrize("tag", ["a", "b"])
def test_oracle_textures_match_committed_reference_outputs(tag):
    """Whole textured Draw of the compiled reference (tests/golden/make_golden.py textured) on the
    synthetic images of helpers.synthetic_textures(seed)."""
    g = load_golden(f"rast_ref_cornell_tex_{tag}_64x48.npz")
    W, H = int(g["W"]), int(g["H"])
    tex = h.synthetic_textures(int(g["seed"]))
    room, boxes = g["room"].view(h.RAST_TRI), g["boxes"].view(h.RAST_TRI)
    assert set(np.unique(room["texture"])) | set(np.unique(boxes["texture"])) <= {1, 2, 3}
    try:
        h.oracle_rast_set_textures(tex, g["cam"], g["R"], float(g["yaw"]))
        o = h.oracle_rast_draw(W, H, float(g["focal"]), g["cam"], g["R"], h.DEFAULT_RAST_LIGHT, room, boxes)
    finally:
        h.oracle_rast_set_textures(None)
    for key in ("rgb", "depth", "low", "high", "screen_post"):
        assert np.array_equal(bits(o[key]), bits(g[key])), key
    assert np.array_equal(o["shadow"], g["shadow"])
    assert np.array_equal(o["argb"], g["argb"])
    assert np.count_nonzero(bits(g["rgb"])) > 1000


@pytest.mark.parametrize("setting,setting_boxes,cam,yaw,indirect", [
    (2, 1, h.DEFAULT_RAST_CAM, 0.0, 0.2), (1, 3, (0.1, -0.05, -2.6, 1.0), 0.174533, 0.2),
    (3, 2, h.DEFAULT_RAST_CAM, -0.349066, 0.2), (3, 3, (0.0, 0.0, -1.5, 1.0), 0.0, 0.15), (2, 2, h.DEFAULT_RAST_CAM, 0.0, 0.15)])
def test_oracle_textures_vs_compiled_reference(setting, setting_boxes, cam, yaw, indirect):
    """Every texture on room and boxes, the `yaw != 0` branch (glm::inverse(R)), holes that clear the
    depth (:619, :643) and the entry value of the indirect light behind holes, at 320x240."""
    W, H, f = 320, 240, 120.0
    if not h.have_ref(h.ref_rast_name(W, H)):
        pytest.skip("oracle/_ref not built")
    tex = h.synthetic_textures(11)
    R = h.yaw_R(yaw) if yaw != 0 else h.identity_R()
    room, boxes = h.ref_rast_testmodel_tex(setting, setting_boxes, W, H)
    light = dict(h.DEFAULT_RAST_LIGHT, indirect=(indirect,) * 3)
    h.ref_rast_set_textures(W, H, tex, cam, R, yaw)
    ref = h.ref_rast_draw(W, H, f, cam, R, light, room, boxes)
    try:
        h.oracle_rast_set_textures(tex, cam, R, yaw)
        o = h.oracle_rast_draw(W, H, f, cam, R, light, room, boxes)
    finally:
        h.oracle_rast_set_textures(None)
    for key in ("depth", "low", "high", "rgb", "screen_post"):
        assert np.array_equal(bits(ref[key]), bits(o[key])), key
    assert np.array_equal(ref["shadow"], o["shadow"])
    assert np.array_equal(ref["argb"], o["argb"])
    if setting_boxes in (2, 3):
        assert np.count_nonzero((o["depth"] == 0) & (o["index"] >= 0)) > 50   # colour kept under a cleared depth


def test_oracle_inverse_is_glm_inverse_on_rotations():
    """R stays a rotation about y (:387-396): inverse = transpose up to rounding; the restated cofactor
    expansion must at least invert it to float accuracy (its bit pattern is pinned by the tests above)."""
    lib = h.oracle()
    for yaw in (0.174533, -0.349066, 1.0, 2.5):
        R = h.yaw_R(yaw)
        inv = np.zeros(16, np.float32)
        lib.oracle_rast_inverse(h.ptr(R), h.ptr(inv))
        prod = R.reshape(4, 4).T.astype(np.float64) @ inv.reshape(4, 4).T.astype(np.float64)
        assert np.allclose(prod, np.eye(4), atol=1e-6)


@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("cam,yaw,indirect", [(h.DEFAULT_RAST_CAM, 0.0, 0.2), ((0.1, -0.05, -2.6, 1.0), 0.174533, 0.15)])
def test_oracle_colour_modes_vs_compiled_reference(mode, cam, yaw, indirect):
    """randColourSelect = 1 / 2 (:647-662): three rand() per accepted fragment in the order of the reference's
    loops, screenBuffer only, the entry value of the indirect light on every fragment.  Same seed, same
    pixels, and the C library's stream ends at the same place."""
    W, H, f = 320, 240, 120.0
    if not h.have_ref(h.ref_rast_name(W, H)):
        pytest.skip("oracle/_ref not built")
    R = h.yaw_R(yaw) if yaw else h.identity_R()
    room, boxes = h.ref_rast_testmodel(W, H)
    light = dict(h.DEFAULT_RAST_LIGHT, indirect=(indirect,) * 3)
    lib = h.ref_lib(h.ref_rast_name(W, H))
    try:
        lib.ref_rast_set_colour_mode(mode)
        h.srand(99)
        ref = h.ref_rast_draw(W, H, f, cam, R, light, room, boxes)
        next_ref = h.rand()
        h.oracle().oracle_rast_set_colour_mode(mode)
        h.srand(99)
        o = h.oracle_rast_draw(W, H, f, cam, R, light, room, boxes)
        next_o = h.rand()
    finally:
        lib.ref_rast_set_colour_mode(0)
        h.oracle().oracle_rast_set_colour_mode(0)
    for key in ("depth", "low", "high", "rgb", "screen_post"):
        assert np.array_equal(bits(ref[key]), bits(o[key])), key
    assert np.array_equal(ref["shadow"], o["shadow"]) and np.array_equal(ref["argb"], o["argb"])
    assert next_ref == next_o
    assert not np.any(o["low"]) and not np.any(o["high"])


@pytest.mark.parametrize("setting,setting_boxes,cam,yaw", [(2, 3, h.DEFAULT_RAST_CAM, 0.0), (3, 2, (0.1, -0.05, -2.6, 1.0), 0.174533),
                                                           (2, 1, h.DEFAULT_RAST_CAM, -0.349066)])
def test_oracle_textures_with_the_reference_repository_images(setting, setting_boxes, cam, yaw):
    """The same comparison on the images of the reference's own repository (metal grill, woven wood: decoded with
    cv2, grey + threshold like main() :148-155; committed as tests/golden/rast_reference_textures.npz): real hole
    patterns, real normal maps."""
    W, H, f = 320, 240, 120.0
    if not h.have_ref(h.ref_rast_name(W, H)):
        pytest.skip("oracle/_ref not built")
    tex = h.reference_textures()          # the committed decoded pixels ...
    assert set(np.unique(tex["grill_opacity"])) <= {0, 255} and tex["grill"].shape == (1024, 1024, 3)
    ref_dir = os.environ.get("REF")      # a checkout of the reference
    files = h.reference_textures(textures_dir=os.path.join(ref_dir, "rasteriser", "Textures")) if ref_dir else None
    if files is not None:                 # ... are what decoding the reference's files here gives
        for k in h.TEX_IMAGES:
            assert np.array_equal(tex[k], files[k]), k
    R = h.yaw_R(yaw) if yaw != 0 else h.identity_R()
    room, boxes = h.ref_rast_testmodel_tex(setting, setting_boxes, W, H)
    h.ref_rast_set_textures(W, H, tex, cam, R, yaw)
    ref = h.ref_rast_draw(W, H, f, cam, R, h.DEFAULT_RAST_LIGHT, room, boxes)
    try:
        h.oracle_rast_set_textures(tex, cam, R, yaw)
        o = h.oracle_rast_draw(W, H, f, cam, R, h.DEFAULT_RAST_LIGHT, room, boxes)
    finally:
        h.oracle_rast_set_textures(None)
    for key in ("depth", "low", "high", "rgb", "screen_post"):
        assert np.array_equal(bits(ref[key]), bits(o[key])), key
    assert np.array_equal(ref["shadow"], o["shadow"]) and np.array_equal(ref["argb"], o["argb"])
    holes = np.count_nonzero((o["depth"] == 0) & (o["index"] >= 0))
    assert holes > 0 or setting_boxes == 1
