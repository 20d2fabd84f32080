"""Batched views: render_raytrace_views / draw_raytrace_views / rt_render_views_device render many cameras of one
scene in one call.  Every view must equal, bit for bit, the single-camera entry with that camera."""
import ctypes

import numpy as np
import pytest

import helpers as h
from conftest import load_golden

pytestmark = pytest.mark.gpu

VIEWS_PER_LAUNCH = 64     # RT_VIEWS_MAX (csrc/rt_filtered.cuh)


def bits(a):
    return a.view(np.uint32)


def cornell_poses(W, H):
    """Translation, yaw, focal changes, a camera inside the room and one far outside (|cam| ~ 50)."""
    f = float(W) * 0.8
    return [(h.f32(0, 0, -3, 1), f, h.identity_R()),
            (h.f32(0.3, -0.2, -2.7, 1), f, h.identity_R()),
            (h.f32(-0.1, 0.05, -3.1, 1), f, h.yaw_R(0.3)),
            (h.f32(0.05, 0.1, -2.9, 1), 0.5 * f, h.yaw_R(-0.2)),
            (h.f32(0.0, 0.2, -0.3, 1), 0.6 * f, h.yaw_R(0.7)),          # inside the room
            (h.f32(2.0, -1.5, -50.0, 1), 12.0 * f, h.yaw_R(0.04)),      # far outside: widens the shared bound
            (h.f32(0.1, -0.3, -2.2, 1), 1.7 * f, h.yaw_R(-0.5))]


def cams_of(b200, poses, W, H):
    return [b200.make_camera(p, f, R, W, H) for p, f, R in poses]


def check_views(got, singles, what, keys=("rgb", "depth", "index")):
    for k, s in enumerate(singles):
        for key in keys:
            if got[key] is None:
                continue
            nb = np.count_nonzero(bits(got[key][k]) != bits(s[key]) if got[key].dtype == np.float32 else got[key][k] != s[key])
            assert nb == 0, f"{what}: view {k}, {key} differs at {nb} values"


def singles_of(renderer, tris, sph, cams, lights):
    out = []
    for c in cams:
        out.append(renderer.render_raytrace(tris, sph, c, lights))
        out[-1]["stats"] = renderer.stats()
    return out


def test_cornell_poses_equal_single_view(b200, renderer, cornell_rt):
    tris, sph = cornell_rt
    W, H = 160, 128
    cams = cams_of(b200, cornell_poses(W, H), W, H)
    singles = singles_of(renderer, tris, sph, cams, h.DEFAULT_RT_LIGHTS)
    got = renderer.render_raytrace_views(tris, sph, cams, h.DEFAULT_RT_LIGHTS)
    st = renderer.stats()
    assert got["rgb"].shape == (len(cams), H, W, 3) and got["depth"].shape == (len(cams), H, W)
    check_views(got, singles, "cornell poses")
    assert st["primary_rays"] == len(cams) * W * H * 9
    assert st["shadow_rays"] == sum(s["stats"]["shadow_rays"] for s in singles)
    assert st["gpu_ms"] > 0
    # the packed frames against draw_raytrace, view by view
    argb = renderer.draw_raytrace_views(tris, sph, b200.make_cameras(cams), h.DEFAULT_RT_LIGHTS)
    assert renderer.stats()["primary_rays"] == len(cams) * W * H * 9
    assert argb.shape == (len(cams), H, W) and argb.dtype == np.uint32
    for k, c in enumerate(cams):
        assert np.array_equal(argb[k], renderer.draw_raytrace(tris, sph, c, h.DEFAULT_RT_LIGHTS)), f"argb view {k}"
    # a batch of one view (rendered by the single-view kernels)
    one = renderer.render_raytrace_views(tris, sph, cams[5:6], h.DEFAULT_RT_LIGHTS)
    check_views(one, singles[5:6], "one view")
    assert renderer.stats()["primary_rays"] == W * H * 9


def test_kat2_pose_in_a_batch_reproduces_the_screenshot(b200, renderer, cornell_rt):
    tris, sph = cornell_rt
    gold = load_golden("rt_screenshot_320x256.npz")["argb"]
    kat = h.f32(0, 0, np.float32(-3.0) + np.float32(0.1), 1)
    cams = [b200.make_camera(h.f32(0.2, 0, -2.8, 1), 256.0, h.yaw_R(0.2), 320, 256),
            b200.make_camera(kat, 256.0, h.identity_R(), 320, 256),
            b200.make_camera(h.f32(0, -0.1, -3.5, 1), 200.0, h.identity_R(), 320, 256)]
    argb = renderer.draw_raytrace_views(tris, sph, cams, h.DEFAULT_RT_LIGHTS)
    assert np.array_equal(argb[1], gold)


def test_oracle_three_views(b200, renderer, cornell_rt):
    tris, sph = cornell_rt
    W, H = 48, 40
    poses = cornell_poses(W, H)[1:4]
    got = renderer.render_raytrace_views(tris, sph, cams_of(b200, poses, W, H), h.DEFAULT_RT_LIGHTS)
    shadow = 0
    for k, (p, f, R) in enumerate(poses):
        want = h.oracle_rt_render(W, H, f, p, R, h.lights_array(h.DEFAULT_RT_LIGHTS), tris, sph)
        assert np.array_equal(got["index"][k], want["index"]), f"view {k} index"
        assert np.array_equal(bits(got["depth"][k]), bits(want["dist"])), f"view {k} distance"
        assert np.array_equal(bits(got["rgb"][k]), bits(want["rgb"])), f"view {k} colour"
        shadow += want["shadow"]
    assert renderer.stats()["shadow_rays"] == shadow


def test_random_scene_spheres_three_lights(b200, renderer):
    tris, sph = h.random_rt_scene(45, 11, n_spheres=2)
    lights = [((0.2, -1.4, -1.5, 1.0), (9, 9, 9)), ((-1.1, 0.4, -1.8, 1.0), (4, 5, 6)), ((0.9, 0.9, -2.0, 1.0), (3, 2, 1))]
    W, H = 64, 48
    poses = [(h.f32(0, 0, -3, 1), 50.0, h.identity_R()), (h.f32(0.4, -0.3, -2.6, 1), 40.0, h.yaw_R(0.25)),
             (h.f32(-0.5, 0.2, -3.4, 1), 70.0, h.yaw_R(-0.35)), (h.f32(0.1, 0.1, -4.0, 1), 55.0, h.yaw_R(0.1))]
    cams = cams_of(b200, poses, W, H)
    singles = singles_of(renderer, tris, sph, cams, lights)
    got = renderer.render_raytrace_views(tris, sph, cams, lights)
    check_views(got, singles, "random scene, 3 lights")
    assert renderer.stats()["shadow_rays"] == sum(s["stats"]["shadow_rays"] for s in singles)


def test_frames_not_multiples_of_16(b200, renderer, cornell_rt):
    tris, sph = cornell_rt
    W, H = 37, 21
    cams = cams_of(b200, cornell_poses(W, H), W, H)
    got = renderer.render_raytrace_views(tris, sph, cams, h.DEFAULT_RT_LIGHTS)
    check_views(got, singles_of(renderer, tris, sph, cams, h.DEFAULT_RT_LIGHTS), "37x21")


def test_host_entry_with_some_outputs_null(b200, renderer, cornell_rt):
    tris, sph = cornell_rt
    W, H = 64, 48
    cams = cams_of(b200, cornell_poses(W, H)[:4], W, H)
    singles = singles_of(renderer, tris, sph, cams, h.DEFAULT_RT_LIGHTS)
    for want in (("depth",), ("rgb", "index"), ("index",)):
        got = renderer.render_raytrace_views(tris, sph, cams, h.DEFAULT_RT_LIGHTS, want=want)
        for key in ("rgb", "depth", "index"):
            assert (got[key] is None) == (key not in want)
        check_views(got, singles, f"outputs {want}")


def test_device_entry_leaves_the_extra_view_untouched(b200, renderer, cornell_rt):
    import torch
    tris, sph = cornell_rt
    W, H = 80, 64
    cams = cams_of(b200, cornell_poses(W, H)[:5], W, H)
    K = len(cams)
    singles = singles_of(renderer, tris, sph, cams, h.DEFAULT_RT_LIGHTS)
    argbs = [renderer.draw_raytrace(tris, sph, c, h.DEFAULT_RT_LIGHTS) for c in cams]
    sentinel = 0x7F7F7F7F
    rgb = torch.full(((K + 1) * H * W * 3,), sentinel, dtype=torch.int32, device="cuda")
    depth = torch.full(((K + 1) * H * W,), sentinel, dtype=torch.int32, device="cuda")
    index = torch.full(((K + 1) * H * W,), sentinel, dtype=torch.int32, device="cuda")
    argb = torch.full(((K + 1) * H * W,), sentinel, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    renderer.rt_upload_scene(tris, sph)
    renderer.rt_render_views_device(cams, h.DEFAULT_RT_LIGHTS, rgb.data_ptr(), depth.data_ptr(), index.data_ptr(),
                                    argb.data_ptr())
    renderer.synchronize()
    st = renderer.stats()
    assert st["primary_rays"] == K * W * H * 9
    rgb, depth, index, argb = (t.cpu().numpy() for t in (rgb, depth, index, argb))
    got = dict(rgb=rgb[: K * H * W * 3].view(np.float32).reshape(K, H, W, 3),
               depth=depth[: K * H * W].view(np.float32).reshape(K, H, W), index=index[: K * H * W].reshape(K, H, W))
    check_views(got, singles, "device entry")
    assert np.array_equal(argb[: K * H * W].view(np.uint32).reshape(K, H, W), np.stack(argbs))
    for t, n in ((rgb, 3), (depth, 1), (index, 1), (argb, 1)):
        assert np.all(t[K * H * W * n:] == sentinel), "the view past the batch was written"


def test_batch_larger_than_one_launch(b200, renderer, cornell_rt):
    tris, sph = cornell_rt
    W, H = 16, 12
    K = VIEWS_PER_LAUNCH + 3
    rng = np.random.default_rng(5)
    poses = [(h.f32(*rng.uniform(-0.4, 0.4, 2), rng.uniform(-3.4, -2.2), 1), float(rng.uniform(8, 20)),
              h.yaw_R(float(rng.uniform(-0.4, 0.4)))) for _ in range(K)]
    poses[K - 1] = (h.f32(1.0, 2.0, -48.0, 1), 160.0, h.identity_R())   # in the last launch only
    cams = cams_of(b200, poses, W, H)
    singles = singles_of(renderer, tris, sph, cams, h.DEFAULT_RT_LIGHTS)
    got = renderer.render_raytrace_views(tris, sph, cams, h.DEFAULT_RT_LIGHTS)
    st = renderer.stats()
    check_views(got, singles, f"{K} views")
    assert st["primary_rays"] == K * W * H * 9
    assert st["shadow_rays"] == sum(s["stats"]["shadow_rays"] for s in singles)
    assert st["kernel_launches"] >= 4     # scene preparation + two launches of (planes, render)


def test_bruteforce_equals_filtered_batch(b200, renderer, cornell_rt):
    tris, sph = cornell_rt
    W, H = 48, 32
    cams = cams_of(b200, cornell_poses(W, H)[:4], W, H)
    filtered = renderer.render_raytrace_views(tris, sph, cams, h.DEFAULT_RT_LIGHTS)
    sh = renderer.stats()["shadow_rays"]
    renderer.set_option(b200.OPT_RT_BRUTEFORCE, 1)
    try:
        brute = renderer.render_raytrace_views(tris, sph, cams, h.DEFAULT_RT_LIGHTS)
        st = renderer.stats()
    finally:
        renderer.set_option(b200.OPT_RT_BRUTEFORCE, 0)
    check_views(brute, [{k: filtered[k][i] for k in ("rgb", "depth", "index")} for i in range(len(cams))], "bruteforce")
    assert st["shadow_rays"] == sh and st["primary_rays"] == len(cams) * W * H * 9


def test_gridded_scenes_view_by_view(b200, renderer, cornell_rt):
    tris, sph = b200.scene_cornell_rt_tessellated(7)
    assert len(tris) == 1372
    W, H = 64, 48
    cams = cams_of(b200, cornell_poses(W, H)[:3], W, H)
    singles = singles_of(renderer, tris, sph, cams, h.DEFAULT_RT_LIGHTS)
    got = renderer.render_raytrace_views(tris, sph, cams, h.DEFAULT_RT_LIGHTS)
    check_views(got, singles, "tessellated 1372, grids")
    assert renderer.stats()["shadow_rays"] == sum(s["stats"]["shadow_rays"] for s in singles)
    # the Cornell box forced onto the grid kernels equals its streamed batch
    ctris, csph = cornell_rt
    ccams = cams_of(b200, cornell_poses(W, H), W, H)
    streamed = renderer.render_raytrace_views(ctris, csph, ccams, h.DEFAULT_RT_LIGHTS)
    renderer.set_option(b200.OPT_RT_GRID, 1)
    try:
        gridded = renderer.render_raytrace_views(ctris, csph, ccams, h.DEFAULT_RT_LIGHTS)
    finally:
        renderer.set_option(b200.OPT_RT_GRID, 0)
    check_views(gridded, [{k: streamed[k][i] for k in ("rgb", "depth", "index")} for i in range(len(ccams))],
                "cornell, B200_OPT_RT_GRID = 1")


def test_invalid_arguments(b200, renderer, cornell_rt):
    tris, sph = cornell_rt
    lib = renderer.lib
    W, H = 32, 24
    good = cams_of(b200, cornell_poses(W, H)[:3], W, H)
    la = b200.make_lights(h.DEFAULT_RT_LIGHTS)
    out = np.zeros(3 * W * H, np.uint32)
    P = b200._ptr

    def draw(cams, n_views, lights=la, n_lights=1):
        return lib.draw_raytrace_views(renderer.ctx, P(tris), len(tris), P(sph), len(sph), cams, int(n_views), lights,
                                       int(n_lights), P(out))

    want = renderer.draw_raytrace_views(tris, sph, good, h.DEFAULT_RT_LIGHTS)
    mismatched = list(good[:2]) + [b200.make_camera(h.f32(0, 0, -3, 1), 20.0, h.identity_R(), W, H + 1)]
    bad_res = list(good[:2]) + [b200.make_camera(h.f32(0, 0, -3, 1), 20.0, h.identity_R(), 0, H)]
    nine = b200.make_lights(h.DEFAULT_RT_LIGHTS * 9)
    cases = [("n_views = 0", lambda: draw(b200.make_cameras(good), 0)),
             ("n_views < 0", lambda: draw(b200.make_cameras(good), -2)),
             ("null cameras", lambda: draw(None, 3)),
             ("mismatched sizes", lambda: draw(b200.make_cameras(mismatched), 3)),
             ("bad resolution", lambda: draw(b200.make_cameras(bad_res), 3)),
             ("9 lights", lambda: draw(b200.make_cameras(good), 3, nine, 9)),
             ("null lights", lambda: draw(b200.make_cameras(good), 3, None, 1)),
             ("render, n_views = 0", lambda: lib.render_raytrace_views(renderer.ctx, P(tris), len(tris), P(sph), len(sph),
                                                                        b200.make_cameras(good), 0, la, 1, None, None, None)),
             ("device, null cameras", lambda: lib.rt_render_views_device(renderer.ctx, None, 3, la, 1, None, None, None, None))]
    for what, call in cases:
        assert call() == b200.B200_EINVAL, what
        assert lib.b200_last_error(renderer.ctx), what
        # the context stays usable
        assert np.array_equal(renderer.draw_raytrace_views(tris, sph, good, h.DEFAULT_RT_LIGHTS), want), what


def test_device_entry_refused_on_a_multi_gpu_context(b200, renderer, cornell_rt):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    m = b200.Renderer(n_gpus=2)
    try:
        cams = b200.make_cameras(cams_of(b200, cornell_poses(16, 16)[:2], 16, 16))
        la = b200.make_lights(h.DEFAULT_RT_LIGHTS)
        assert m.lib.rt_render_views_device(m.ctx, cams, 2, la, 1, None, None, None, None) == b200.B200_EINVAL
        tris, sph = cornell_rt
        assert m.draw_raytrace_views(tris, sph, cams, h.DEFAULT_RT_LIGHTS).shape == (2, 16, 16)   # still usable
    finally:
        m.close()


def test_multi_gpu_context_equals_single_device(b200, renderer, cornell_rt):
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs 2 GPUs")
    tris, sph = cornell_rt
    W, H = 96, 64
    cams = cams_of(b200, cornell_poses(W, H), W, H)          # 7 views: uneven runs, some devices may get none
    want = renderer.render_raytrace_views(tris, sph, cams, h.DEFAULT_RT_LIGHTS)
    want_st = renderer.stats()
    want_argb = renderer.draw_raytrace_views(tris, sph, cams, h.DEFAULT_RT_LIGHTS)
    m = b200.Renderer(n_gpus=min(n, 8))
    try:
        got = m.render_raytrace_views(tris, sph, cams, h.DEFAULT_RT_LIGHTS)
        st = m.stats()
        check_views(got, [{k: want[k][i] for k in ("rgb", "depth", "index")} for i in range(len(cams))], "multi-GPU")
        assert st["primary_rays"] == want_st["primary_rays"] and st["shadow_rays"] == want_st["shadow_rays"]
        assert np.array_equal(m.draw_raytrace_views(tris, sph, cams, h.DEFAULT_RT_LIGHTS), want_argb)
    finally:
        m.close()


def test_make_cameras_layout(b200):
    cams = b200.make_cameras([b200.make_camera((1, 2, 3, 1), 7.0, h.identity_R(), 5, 4), ((0, 0, -3, 1), 9.0, h.yaw_R(0.1), 5, 4)])
    assert len(cams) == 2 and ctypes.sizeof(cams) == 2 * ctypes.sizeof(b200.Camera)
    assert cams[0].pos[2] == 3.0 and cams[1].focal == 9.0 and cams[1].width == 5
