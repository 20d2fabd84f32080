"""render_raytrace_samples, draw_raytrace_samples and rt_render_samples_device: Draw with the caller's own sample
offsets per pixel.  With the reference's nine offsets they give render_raytrace's frames bit for bit; with other
patterns they equal the plain-C oracle (oracle_rt_samples) and the composed rt_closest_hits -> rt_direct_light ->
accumulation chain, on the streaming, gridded and brute-force kernels."""
import ctypes

import numpy as np
import pytest

import helpers as h
import samples_helpers as sh
from conftest import load_golden

pytestmark = pytest.mark.gpu
EINVAL = -1
LIGHTS8 = [((0.3, 0.7, -0.4, 1.0), (3, 4, 5)), ((0.0, 0.0, 1.5, 1.0), (20, 20, 20)),
           ((0.0, -0.5, -0.7, 1.0), (14, 14, 14)), ((-0.3, 0.4, 0.2, 1.0), (2, 2, 2)),
           ((0.5, -0.9, 0.5, 1.0), (7, 1, 3)), ((-0.8, 0.8, -0.9, 1.0), (1, 9, 1)),
           ((0.0, 0.0, -2.0, 1.0), (30, 30, 30)), ((0.6, 0.2, -0.6, 1.0), (5, 5, 9))]
YAW_POSE = (h.f32(0.1, -0.05, -2.8, 1), h.yaw_R(0.3))
# (pattern, depth samples): S = 1, 2, 4, 5, 9 reordered, 10, 16, 64
PATTERNS = [("centre", (0,)), ("random2", (1,)), ("rgss", (0, 3)), ("random5", (2,)), ("nine_reordered", (4, 8)),
            ("random10", (9,)), ("strat4", (5,)), ("strat8", (0, 63))]


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def golden_scene(name):
    g = load_golden(f"rt_ref_{name}.npz")
    tris = g["tris"].view(h.RT_TRI).copy()
    sph = g["spheres"].view(h.RT_SPHERE).copy()
    cam = h.f32(*g["cam"])
    lights = [(tuple(l[:4]), tuple(l[4:])) for l in g["lights"].reshape(-1, 7)]
    return tris, (sph if len(sph) else None), int(g["W"]), int(g["H"]), float(g["focal"]), cam, g["R"].copy(), lights


def assert_frame_equal(got, want, what=""):
    assert np.array_equal(bits(got["rgb"]), bits(want["rgb"])), f"{what}: rgb"
    assert np.array_equal(bits(got["depth"]), bits(want["depth"])), f"{what}: depth"
    assert np.array_equal(got["index"], want["index"]), f"{what}: index"


def assert_oracle(got, o, what=""):
    assert np.array_equal(bits(got["rgb"]), bits(o["rgb"])), f"{what}: rgb"
    assert np.array_equal(bits(got["depth"]), bits(o["dist"])), f"{what}: depth"
    assert np.array_equal(got["index"], o["index"]), f"{what}: index"


@pytest.fixture
def options(b200, renderer):
    """Options set by a test go back to their defaults afterwards."""
    yield renderer
    for opt, v in ((b200.OPT_RT_BRUTEFORCE, 0), (b200.OPT_RT_GRID, 0), (b200.OPT_RT_INTERLEAVE_N, 1),
                   (b200.OPT_RT_PLAN, 1)):
        renderer.set_option(opt, v)


# ---- 1. the reference's pattern is render_raytrace --------------------------------------------
@pytest.mark.parametrize("name", ["cornell_default_160x128", "cornell_yaw_96x64", "random40_96x64"])
def test_reference_pattern_equals_render_raytrace(b200, renderer, name):
    tris, sph, W, H, f, cam, R, lights = golden_scene(name)
    c = b200.make_camera(cam, f, R, W, H)
    got = renderer.render_raytrace_samples(tris, sph, c, lights, sh.NINE, 4)
    want = renderer.render_raytrace(tris, sph, c, lights)
    assert_frame_equal(got, want, name)
    assert np.array_equal(renderer.draw_raytrace_samples(tris, sph, c, lights, sh.NINE, 4),
                          renderer.draw_raytrace(tris, sph, c, lights))


@pytest.mark.parametrize("n_lights", [0, 1, 3, 8])
def test_reference_pattern_any_light_count_yawed(b200, renderer, cornell_rt, n_lights):
    tris, sph = cornell_rt
    c = b200.make_camera(YAW_POSE[0], 100.0, YAW_POSE[1], 130, 90)
    lights = LIGHTS8[:n_lights]
    assert_frame_equal(renderer.render_raytrace_samples(tris, sph, c, lights, sh.NINE, 4),
                       renderer.render_raytrace(tris, sph, c, lights), f"{n_lights} lights")
    assert np.array_equal(renderer.draw_raytrace_samples(tris, sph, c, lights, sh.NINE, 4),
                          renderer.draw_raytrace(tris, sph, c, lights))


# ---- 2. other patterns: the oracle and the composed chain ---------------------------------------
@pytest.mark.parametrize("pat", range(len(PATTERNS)))
@pytest.mark.parametrize("scene", ["cornell", "random40"])
def test_patterns_equal_oracle(b200, renderer, cornell_rt, scene, pat):
    name, depth_samples = PATTERNS[pat]
    if scene == "cornell":
        tris, sph = cornell_rt
        W, H, f, (cam, R), lights = 72, 40, 60.0, YAW_POSE, LIGHTS8[:3]
    else:
        tris, sph, W, H, f, cam, R, lights = golden_scene("random40_96x64")
    off = sh.pattern(name, seed=pat)
    c = b200.make_camera(cam, f, R, W, H)
    L7 = h.lights_array(lights)
    for ds in depth_samples:
        got = renderer.render_raytrace_samples(tris, sph, c, lights, off, ds)
        st = renderer.stats()
        o = sh.oracle_rt_samples(W, H, f, cam, R, L7, tris, sph, off, ds)
        assert_oracle(got, o, f"{scene} {name} depth sample {ds}")
        assert st["primary_rays"] == W * H * len(off) == o["primary"]     # 5. stats
        assert st["shadow_rays"] == o["shadow"]
        assert np.array_equal(renderer.draw_raytrace_samples(tris, sph, c, lights, off, ds), o["argb"])


@pytest.mark.parametrize("name", ["rgss", "nine_reordered", "random10"])
def test_patterns_equal_composed_chain(b200, renderer, cornell_rt, name):
    tris, sph = cornell_rt
    W, H, f, (cam, R) = 64, 48, 50.0, YAW_POSE
    lights = LIGHTS8[:2]
    off = sh.pattern(name, seed=5)
    S = len(off)
    c = b200.make_camera(cam, f, R, W, H)
    got = renderer.render_raytrace_samples(tris, sph, c, lights, off, S - 1)
    hits = renderer.rt_closest_hits(tris, sph, sh.sample_rays(W, H, f, cam, R, off))
    power = renderer.rt_direct_light(tris, sph, hits, lights)
    arr = renderer._hits(hits)
    rgb = sh.accumulate(arr, power, tris, sph, S).reshape(H, W, 3)
    assert np.array_equal(bits(got["rgb"]), bits(rgb))


# ---- 3. gridded scenes: streaming, gridded, brute force and the oracle agree ---------------------
@pytest.mark.parametrize("scene", ["tess10", "cornell"])
def test_gridded_streaming_bruteforce_oracle(b200, options, cornell_rt, scene):
    r = options
    tris, sph = h.scene_cornell_rt_tessellated(10) if scene == "tess10" else cornell_rt
    if scene == "tess10":
        assert len(tris) == 2800
    W, H, f, (cam, R) = 56, 36, 48.0, YAW_POSE
    lights = LIGHTS8[:2]
    c = b200.make_camera(cam, f, R, W, H)
    for name, ds in (("rgss", 2), ("random10", 9)):
        off = sh.pattern(name, seed=11)
        frames = {}
        for mode, grid, brute in (("grid", 1, 0), ("stream", 2, 0), ("brute", 0, 1)):
            r.set_option(b200.OPT_RT_GRID, grid)
            r.set_option(b200.OPT_RT_BRUTEFORCE, brute)
            frames[mode] = r.render_raytrace_samples(tris, sph, c, lights, off, ds)
        r.set_option(b200.OPT_RT_BRUTEFORCE, 0)
        r.set_option(b200.OPT_RT_GRID, 0)
        o = sh.oracle_rt_samples(W, H, f, cam, R, h.lights_array(lights), tris, sph, off, ds)
        for mode, fr in frames.items():
            assert_oracle(fr, o, f"{scene} {name} {mode}")


# ---- 4. the device entry: its rows only, interleave classes --------------------------------------
@pytest.mark.parametrize("mode", ["stream", "grid"])
def test_device_entry_rows_and_interleave(b200, options, cornell_rt, mode):
    import torch
    r = options
    tris, sph = cornell_rt
    W, H, f = 150, 117, 100.0
    cam, R = YAW_POSE
    off = sh.pattern("random10", seed=2)
    c = b200.make_camera(cam, f, R, W, H)
    r.set_option(b200.OPT_RT_GRID, 1 if mode == "grid" else 2)
    full = r.render_raytrace_samples(tris, sph, c, h.DEFAULT_RT_LIGHTS, off, 3)
    argb_full = r.draw_raytrace_samples(tris, sph, c, h.DEFAULT_RT_LIGHTS, off, 3)
    r.rt_upload_scene(tris, sph)
    for row0, row1, il in ((5, 101, 1), (0, H, 2)):
        rgb = torch.full((H, W, 3), float("nan"), device="cuda")
        depth = torch.full((H, W), float("nan"), device="cuda")
        index = torch.full((H, W), 12345, dtype=torch.int32, device="cuda")
        argb = torch.full((H, W), 777, dtype=torch.int32, device="cuda")
        primary = 0
        for k in range(il):
            r.set_option(b200.OPT_RT_INTERLEAVE_N, il)
            r.set_option(b200.OPT_RT_INTERLEAVE_R, k)
            r.rt_render_samples_device(c, h.DEFAULT_RT_LIGHTS, off, 3, row0, row1, rgb.data_ptr(), depth.data_ptr(),
                                       index.data_ptr(), argb.data_ptr())
            primary += r.stats()["primary_rays"]
        r.set_option(b200.OPT_RT_INTERLEAVE_N, 1)
        rgb, depth, index = rgb.cpu().numpy(), depth.cpu().numpy(), index.cpu().numpy()
        argb = argb.cpu().numpy().view(np.uint32)
        assert np.array_equal(bits(rgb[row0:row1]), bits(full["rgb"][row0:row1]))
        assert np.array_equal(bits(depth[row0:row1]), bits(full["depth"][row0:row1]))
        assert np.array_equal(index[row0:row1], full["index"][row0:row1])
        assert np.array_equal(argb[row0:row1], argb_full[row0:row1])
        assert (index[:row0] == 12345).all() and (index[row1:] == 12345).all()
        assert (argb[:row0] == 777).all() and (argb[row1:] == 777).all()
        assert np.isnan(depth[:row0]).all() and np.isnan(depth[row1:]).all()
        assert primary == W * (row1 - row0) * len(off)


# ---- 6. a samples call leaves the context as it was --------------------------------------------
def test_context_state_unchanged(b200, options, cornell_rt):
    r = options
    tris, sph = cornell_rt
    c = b200.make_camera(h.f32(0, 0, -3, 1), 128.0, h.identity_R(), 160, 128)
    tess, tsph = h.scene_cornell_rt_tessellated(10)
    cg = b200.make_camera(YAW_POSE[0], 100.0, YAW_POSE[1], 200, 150)
    r.set_option(b200.OPT_RT_GRID, 1)
    r.render_raytrace(tess, tsph, cg, LIGHTS8[:2])
    before_grid = r.render_raytrace(tess, tsph, cg, LIGHTS8[:2])            # a planned frame
    r.set_option(b200.OPT_RT_GRID, 0)
    before = r.render_raytrace(tris, sph, c, h.DEFAULT_RT_LIGHTS)
    st_before = r.stats()
    r.set_option(b200.OPT_RT_GRID, 1)
    r.render_raytrace_samples(tess, tsph, cg, LIGHTS8[:2], sh.pattern("strat4"), 0)
    after_grid = r.render_raytrace(tess, tsph, cg, LIGHTS8[:2])
    r.set_option(b200.OPT_RT_GRID, 0)
    r.render_raytrace_samples(tris, sph, c, h.DEFAULT_RT_LIGHTS, sh.pattern("random16", seed=1), 7)
    after = r.render_raytrace(tris, sph, c, h.DEFAULT_RT_LIGHTS)
    st_after = r.stats()
    assert_frame_equal(after, before, "render_raytrace")
    assert_frame_equal(after_grid, before_grid, "gridded planned frame")
    for k in ("primary_rays", "shadow_rays", "exact_evals", "kernel_launches"):
        assert st_after[k] == st_before[k], k


# ---- 7. bad arguments --------------------------------------------------------------------------
def test_bad_arguments(b200, renderer, cornell_rt):
    tris, sph = cornell_rt
    lib = renderer.lib
    c = b200.make_camera(h.f32(0, 0, -3, 1), 64.0, h.identity_R(), 32, 32)
    la = b200.make_lights(h.DEFAULT_RT_LIGHTS)
    rgb = np.zeros((32, 32, 3), np.float32)
    argb = np.zeros((32, 32), np.uint32)

    def call(off, n, ds, cam=c, lights=la, n_lights=1, out=rgb):
        o = None if off is None else np.ascontiguousarray(off, np.float32)
        cam = ctypes.byref(cam)
        a = lib.render_raytrace_samples(renderer.ctx, h.ptr(tris), len(tris), h.ptr(sph), len(sph), cam, lights,
                                        n_lights, h.ptr(o), n, ds, h.ptr(out), None, None)
        d = lib.draw_raytrace_samples(renderer.ctx, h.ptr(tris), len(tris), h.ptr(sph), len(sph), cam, lights,
                                      n_lights, h.ptr(o), n, ds, h.ptr(argb))
        renderer.rt_upload_scene(tris, sph)
        v = lib.rt_render_samples_device(renderer.ctx, cam, lights, n_lights, h.ptr(o), n, ds, 0, 32, None, None,
                                         None, None)
        return a, d, v

    ok = sh.pattern("random4")
    assert call(ok, 4, 3) == (0, 0, 0)
    big = np.zeros((65, 2), np.float32)
    bad = []
    for v in (0.50000006, -0.50000006, 1.0, np.nan, np.inf, -np.inf):
        o = ok.copy()
        o[2, 1] = v
        bad.append((o, 4, 0))
    bad += [(ok, 0, 0), (big, 65, 0), (None, 4, 0), (ok, 4, 4), (ok, 4, -1), (big, 64, 64)]
    for o, n, ds in bad:
        assert call(o, n, ds) == (EINVAL, EINVAL, EINVAL), (o, n, ds)
    zero_cam = b200.make_camera(h.f32(0, 0, -3, 1), 64.0, h.identity_R(), 0, 32)
    assert call(ok, 4, 0, cam=zero_cam) == (EINVAL, EINVAL, EINVAL)
    assert call(ok, 4, 0, n_lights=9) == (EINVAL, EINVAL, EINVAL)
    assert call(ok, 4, 0, lights=None) == (EINVAL, EINVAL, EINVAL)
    assert lib.draw_raytrace_samples(renderer.ctx, h.ptr(tris), len(tris), h.ptr(sph), len(sph), ctypes.byref(c), la, 1,
                                     h.ptr(ok),
                                     4, 0, None) == EINVAL
    assert call(ok, 4, 3) == (0, 0, 0)   # the context still works


# ---- 8. a multi-GPU context ---------------------------------------------------------------------
def test_multi_context_equals_one_device(b200, renderer, cornell_rt):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two or more GPUs")
    tris, sph = cornell_rt
    c = b200.make_camera(YAW_POSE[0], 100.0, YAW_POSE[1], 150, 117)
    off = sh.pattern("random10", seed=4)
    m = b200.Renderer(n_gpus=min(torch.cuda.device_count(), 8))
    try:
        assert m.device_count() >= 2
        assert_frame_equal(m.render_raytrace_samples(tris, sph, c, LIGHTS8[:2], off, 2),
                           renderer.render_raytrace_samples(tris, sph, c, LIGHTS8[:2], off, 2), "multi")
        assert m.stats()["primary_rays"] == 150 * 117 * 10
        assert np.array_equal(m.draw_raytrace_samples(tris, sph, c, LIGHTS8[:2], off, 2),
                              renderer.draw_raytrace_samples(tris, sph, c, LIGHTS8[:2], off, 2))
        assert m.stats()["primary_rays"] == 150 * 117 * 10
        la = b200.make_lights(LIGHTS8[:2])
        o = np.ascontiguousarray(off)
        assert m.lib.rt_render_samples_device(m.ctx, ctypes.byref(c), la, 2, h.ptr(o), len(o), 0, 0, 117, None, None,
                                              None, None) == EINVAL
    finally:
        m.close()
