"""Ray queries (rt_closest_hits, rt_occluded and their _device variants) against the plain-C oracle, bit for bit:
position (all four components), distance, both indices and the occlusion flag."""
import ctypes

import numpy as np
import pytest

import helpers as h
import rays_helpers as rh

pytestmark = pytest.mark.gpu
FLT_MAX = np.finfo(np.float32).max
EINVAL = -1


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_hits_equal(got, want, what=""):
    """got: dict of Renderer.rt_closest_hits; want: RT_INTERSECTION array of the oracle."""
    for f in ("position", "distance"):
        g, w = bits(got[f]), bits(want[f])
        assert g.size == w.size, f"{what}: {f} has {g.size} values, want {w.size}"
        bad = np.nonzero((g != w).reshape(len(want), -1).any(axis=1))[0] if len(want) else []
        assert len(bad) == 0, f"{what}: {f} differs for {len(bad)} rays, first {bad[:5]}"
    for f in ("triangle_index", "sphere_index"):
        bad = np.nonzero(got[f] != want[f])[0]
        assert len(bad) == 0, f"{what}: {f} differs for {len(bad)} rays, first {bad[:5]}"


def check_closest(renderer, tris, sph, rays, what=""):
    got = renderer.rt_closest_hits(tris, sph, rays)
    assert_hits_equal(got, rh.oracle_rt_closest(tris, sph, rays), what)
    return got


def check_occluded(renderer, tris, sph, rays, md, what=""):
    got = renderer.rt_occluded(tris, sph, rays, md)
    want = rh.oracle_rt_occluded(tris, sph, rays, md).astype(bool)
    bad = np.nonzero(got != want)[0]
    assert len(bad) == 0, f"{what}: occlusion differs for {len(bad)} rays, first {bad[:5]}"
    return got


POSES = [(h.f32(0, 0, -3, 1), h.identity_R()), (h.f32(0.13, -0.21, -2.4, 1), h.identity_R()),
         (h.f32(0.1, 0, -2.8, 1), h.yaw_R(0.3))]


@pytest.mark.parametrize("pose", range(3))
def test_cornell_camera_rays_equal_frame_and_oracle(b200, renderer, cornell_rt, pose):
    tris, sph = cornell_rt
    cam, R = POSES[pose]
    W, H, f = 160, 128, 128.0
    rays = rh.camera_rays(W, H, f, cam, R)
    got = check_closest(renderer, tris, sph, rays, f"pose {pose}")
    frame = renderer.render_raytrace(tris, sph, b200.make_camera(cam, f, R, W, H), h.DEFAULT_RT_LIGHTS)
    hit = got["distance"] < FLT_MAX
    depth = np.where(hit, got["distance"], np.float32(np.inf)).astype(np.float32)
    assert np.array_equal(bits(depth), bits(frame["depth"].reshape(-1)))
    idx = np.where(got["triangle_index"] != -1, got["triangle_index"], -1 - got["sphere_index"])
    assert np.array_equal(np.where(hit, idx, h.INDEX_MISS), frame["index"].reshape(-1))


def nine_sample_hits(cornell_rt):
    tris, sph = cornell_rt
    rays = rh.camera_rays(64, 48, 48.0, h.f32(0, 0, -3, 1), h.identity_R(), rh.NINE_SAMPLES)
    return rays, rh.oracle_rt_closest(tris, sph, rays)


def test_nine_samples_and_their_shadow_rays(renderer, cornell_rt):
    tris, sph = cornell_rt
    rays, want = nine_sample_hits(cornell_rt)
    assert_hits_equal(renderer.rt_closest_hits(tris, sph, rays), want, "nine samples")
    light = h.DEFAULT_RT_LIGHTS[0][0]
    srays, r_mag, _ = rh.shadow_rays(want, tris, sph, light)
    assert len(srays) > 20000
    occ = check_occluded(renderer, tris, sph, srays, r_mag, "shadow rays")
    assert occ.any() and not occ.all()
    check_closest(renderer, tris, sph, srays, "shadow rays, closest")


def adversarial_rays(tris, sph, seed=3):
    rng = np.random.default_rng(seed)
    f = np.float32
    out = []

    def add(start, d):
        r = np.zeros(1, rh.RT_RAY)
        r["start"][0] = np.asarray(start, np.float32)
        r["dir"][0] = np.asarray(d, np.float32)
        out.append(r)

    starts = [(0, 0, -3, 1), (0.31, -0.47, -0.2, 1), (-0.9, 0.9, 0.9, 1), (0.0, 0.0, 0.0, 1)]
    for s in starts:
        s3 = np.asarray(s[:3], np.float32)
        for t in tris:   # vertices and edge midpoints: shared by neighbouring triangles (ties)
            for p in (t["v0"][:3], t["v1"][:3], t["v2"][:3], ((t["v0"][:3] + t["v1"][:3]) * f(0.5)).astype(np.float32),
                      ((t["v1"][:3] + t["v2"][:3]) * f(0.5)).astype(np.float32)):
                add(s, list((p - s3).astype(np.float32)) + [0.0])
    for t in tris[::3]:
        v0, e1, e2 = t["v0"][:3], (t["v1"][:3] - t["v0"][:3]).astype(np.float32), (t["v2"][:3] - t["v0"][:3]).astype(np.float32)
        on = (v0 + (e1 * f(0.25)).astype(np.float32) + (e2 * f(0.25)).astype(np.float32)).astype(np.float32)
        nrm = t["normal"][:3]
        add(list(on) + [1], list(e1) + [0])                                   # in the plane
        add(list(v0) + [1], list(e2) + [0])                                   # along an edge
        add(list((on + nrm * f(0.1)).astype(np.float32)) + [1], list(e1) + [0])   # parallel to the plane
        for _ in range(3):                                                   # starts exactly on the triangle
            add(list(on) + [1], list(rng.normal(size=3).astype(np.float32)) + [0])
        add(list(on) + [1], list(-nrm) + [0])
        add(list(on) + [1], list(nrm) + [0])
    base = rng.normal(size=(12, 3)).astype(np.float32)
    for d in base:
        for scale in (0.0, 1e-30, 1e-20, 1e20, 1e30):
            add((0.1, 0.2, -0.5, 1), list((d * f(scale)).astype(np.float32)) + [0])
    for s, d in [((-0.0, 0.0, -3.0, -0.0), (-0.0, -0.0, 1.0, 0.0)), ((0, -0.0, -0.0, 1), (0.0, 1.0, -0.0, 0.0)),
                 ((np.nan, 0, 0, 1), (0, 0, 1, 0)), ((0, 0, -3, 1), (np.nan, 0, 1, 0)),
                 ((np.inf, 0, 0, 1), (-1, 0, 0, 0)), ((0, 0, -3, 1), (0, np.inf, 1, 0)),
                 ((0, 0, -3, 1), (np.inf, np.inf, np.inf, 0)), ((-np.inf, 0, 0, 1), (np.inf, 0, 0, 0)),
                 ((0, 0, -3, np.nan), (0, 0, 1, np.nan)), ((0, 0, -3, 1e30), (0.01, 0.02, 1, -7))]:
        add(s, d)
    for s_ in sph:   # inside the sphere, and rays that graze it
        c, r = s_["centre"].astype(np.float32), f(s_["radius"])
        for _ in range(8):
            add(list(c) + [1], list(rng.normal(size=3).astype(np.float32)) + [0])
        for eps in (0.0, 1e-7, -1e-7, 1e-4, -1e-4):
            st = (c + np.array([r * f(1 + eps), 0, -2], np.float32)).astype(np.float32)
            add(list(st) + [1], [0, 0, 1, 0])
    rays = np.concatenate(out)
    rays["start"][::7, 3] = rng.normal(size=len(rays[::7])).astype(np.float32)   # arbitrary w
    rays["dir"][::5, 3] = rng.normal(size=len(rays[::5])).astype(np.float32)
    return rays


def test_adversarial_rays(renderer, cornell_rt):
    tris, sph = cornell_rt
    rays = adversarial_rays(tris, sph)
    got = check_closest(renderer, tris, sph, rays, "adversarial")
    assert (got["distance"] < FLT_MAX).sum() > len(rays) // 2
    for md in (np.full(len(rays), np.inf, np.float32), np.full(len(rays), 1.0, np.float32),
               np.ascontiguousarray(got["distance"])):
        check_occluded(renderer, tris, sph, rays, md, "adversarial")


def random_rays(n, seed, extent=1.5):
    rng = np.random.default_rng(seed)
    rays = np.zeros(n, rh.RT_RAY)
    rays["start"][:, :3] = rng.uniform(-extent, extent, (n, 3)).astype(np.float32)
    rays["start"][:, 3] = 1.0
    rays["dir"][:, :3] = rng.normal(size=(n, 3)).astype(np.float32)
    return rays


@pytest.mark.parametrize("n_sph", [0, 1, 3])
@pytest.mark.parametrize("n_tris", [1, 7, 64, 65, 200])
def test_random_scenes_incoherent_rays(renderer, n_tris, n_sph):
    tris, sph = h.random_rt_scene(n_tris, 1000 + 7 * n_tris + n_sph, n_spheres=n_sph)
    rays = random_rays(3001, n_tris + n_sph)
    got = check_closest(renderer, tris, sph if n_sph else None, rays, f"random {n_tris}/{n_sph}")
    md = np.random.default_rng(n_tris).uniform(0, 2, len(rays)).astype(np.float32)
    check_occluded(renderer, tris, sph if n_sph else None, rays, md, f"random {n_tris}/{n_sph}")
    check_occluded(renderer, tris, sph if n_sph else None, rays, np.ascontiguousarray(got["distance"]), "at distance")


def test_tessellated_box_many_tiles(b200, renderer):
    tris, sph = h.scene_cornell_rt_tessellated(20)
    assert len(tris) == 11200
    rays = random_rays(20000, 11, extent=0.9)
    check_closest(renderer, tris, sph, rays, "tessellated")
    md = np.random.default_rng(2).uniform(0, 1, len(rays)).astype(np.float32)
    check_occluded(renderer, tris, sph, rays, md, "tessellated")
    big = np.concatenate([rh.camera_rays(1000, 1000, 800.0, h.f32(0, 0, -3, 1), h.identity_R()), random_rays(3, 5)])
    assert len(big) == 1000003
    mdb = np.full(len(big), 3.5, np.float32)
    filt, filt_occ = renderer.rt_closest_hits(tris, sph, big), renderer.rt_occluded(tris, sph, big, mdb)
    renderer.set_option(b200.OPT_RT_BRUTEFORCE, 1)
    try:
        brute, brute_occ = renderer.rt_closest_hits(tris, sph, big), renderer.rt_occluded(tris, sph, big, mdb)
    finally:
        renderer.set_option(b200.OPT_RT_BRUTEFORCE, 0)
    for f in brute:
        assert np.array_equal(np.ascontiguousarray(filt[f]).view(np.uint32 if filt[f].dtype == np.float32 else filt[f].dtype),
                              np.ascontiguousarray(brute[f]).view(np.uint32 if brute[f].dtype == np.float32 else brute[f].dtype)), f
    assert np.array_equal(filt_occ, brute_occ)


@pytest.mark.parametrize("n", [0, 1, 31, 33])
@pytest.mark.parametrize("scene", ["cornell", "empty", "spheres", "triangles"])
def test_batch_sizes_and_scenes(renderer, cornell_rt, n, scene):
    tris, sph = cornell_rt
    t, s = {"cornell": (tris, sph), "empty": (tris[:0], None), "spheres": (tris[:0], sph),
            "triangles": (tris, None)}[scene]
    rays = rh.camera_rays(8, 8, 8.0, h.f32(0, 0, -3, 1), h.identity_R())
    rays = np.resize(np.concatenate([rays, random_rays(64, n)]), n) if n else rays[:0]
    got = check_closest(renderer, t, s, rays, scene)
    if scene == "empty":
        assert np.all(got["distance"] == FLT_MAX) and np.all(got["triangle_index"] == -1)
    check_occluded(renderer, t, s, rays, np.full(n, 10.0, np.float32), scene)


def test_max_distance_edges(renderer, cornell_rt):
    tris, sph = cornell_rt
    rays = rh.camera_rays(48, 32, 32.0, h.f32(0, 0, -3, 1), h.identity_R())
    want = rh.oracle_rt_closest(tris, sph, rays)
    d = want["distance"]
    hit = d < FLT_MAX
    n = len(rays)
    with np.errstate(over="ignore"):
        up = np.nextafter(d, np.float32(np.inf))
    for name, md in [("zero", np.zeros(n)), ("negative", -np.ones(n)), ("nan", np.full(n, np.nan)),
                     ("inf", np.full(n, np.inf)), ("equal", d), ("next float", up)]:
        got = check_occluded(renderer, tris, sph, rays, np.ascontiguousarray(md, np.float32), name)
        if name == "equal":
            assert not got.any()
        if name == "next float":
            assert np.array_equal(got, hit)


def test_device_entries_equal_host_entries(renderer, cornell_rt):
    import torch
    tris, sph = cornell_rt
    rays, _ = nine_sample_hits(cornell_rt)
    srays, r_mag, _ = rh.shadow_rays(rh.oracle_rt_closest(tris, sph, rays), tris, sph, h.DEFAULT_RT_LIGHTS[0][0])
    host = renderer.rt_closest_hits(tris, sph, rays)
    host_occ = renderer.rt_occluded(tris, sph, srays, r_mag)
    renderer.rt_upload_scene(tris, sph)
    d_rays = torch.from_numpy(rays.view(np.uint8).copy()).cuda()
    d_srays = torch.from_numpy(srays.view(np.uint8).copy()).cuda()
    d_md = torch.from_numpy(r_mag.copy()).cuda()
    for _ in range(2):   # a second identical call gives identical results
        d_out = torch.full((len(rays) * 28,), 0xAB, dtype=torch.uint8, device="cuda")
        d_occ = torch.full((len(srays),), 7, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        renderer.rt_closest_hits_device(d_rays.data_ptr(), len(rays), d_out.data_ptr())
        renderer.rt_occluded_device(d_srays.data_ptr(), d_md.data_ptr(), len(srays), d_occ.data_ptr())
        renderer.synchronize()
        out = d_out.cpu().numpy().view(rh.RT_INTERSECTION)
        assert_hits_equal(host, out, "device entry")
        assert np.array_equal(d_occ.cpu().numpy().astype(bool), host_occ)


def test_query_leaves_frames_alone(b200, renderer, cornell_rt):
    """A gridded frame, a query, the same frame: bit-identical frames.  A pipelined raster frame in flight around a
    query still verifies."""
    tris, sph = cornell_rt
    cam = b200.make_camera(h.f32(0, 0, -3, 1), 96.0, h.identity_R(), 128, 96)
    renderer.set_option(b200.OPT_RT_GRID, 1)
    try:
        a = renderer.render_raytrace(tris, sph, cam, h.DEFAULT_RT_LIGHTS)
        renderer.rt_closest_hits(tris, sph, random_rays(5000, 1))
        renderer.rt_occluded(tris, sph, random_rays(5000, 2), np.ones(5000, np.float32))
        b = renderer.render_raytrace(tris, sph, cam, h.DEFAULT_RT_LIGHTS)
    finally:
        renderer.set_option(b200.OPT_RT_GRID, 0)
    for k in a:
        assert np.array_equal(np.ascontiguousarray(a[k]).view(np.uint32), np.ascontiguousarray(b[k]).view(np.uint32)), k

    import torch
    room, boxes = b200.scene_cornell_rast()
    W, H = 96, 64
    rcam = b200.make_camera(h.DEFAULT_RAST_CAM, 64.0, h.identity_R(), W, H)
    L = b200.make_rast_light(**h.DEFAULT_RAST_LIGHT)
    want = renderer.render_raster(room, boxes, rcam, L)
    renderer.rast_upload_scene(room, boxes)
    renderer.set_option(b200.OPT_RAST_PIPELINED, 1)
    try:
        rgb = torch.zeros(H * W * 3, dtype=torch.float32, device="cuda")
        depth = torch.zeros(H * W, dtype=torch.float32, device="cuda")
        index = torch.zeros(H * W, dtype=torch.int32, device="cuda")
        for _ in range(3):
            renderer.rast_draw_device(rcam, L, 0, H, rgb.data_ptr(), depth.data_ptr(), index.data_ptr())
            q = renderer.rt_closest_hits(tris, sph, random_rays(777, 3))
            assert_hits_equal(q, rh.oracle_rt_closest(tris, sph, random_rays(777, 3)), "query between raster frames")
            renderer.synchronize()
            assert np.array_equal(rgb.cpu().numpy().view(np.uint32), want["rgb"].reshape(-1).view(np.uint32))
            assert np.array_equal(index.cpu().numpy(), want["index"].reshape(-1))
    finally:
        renderer.set_option(b200.OPT_RAST_PIPELINED, 0)


def test_stats(b200, renderer, cornell_rt):
    tris, sph = cornell_rt
    rays = rh.camera_rays(320, 256, 256.0, h.f32(0, 0, -3, 1), h.identity_R())
    n = len(rays)
    renderer.rt_closest_hits(tris, sph, rays)
    st = renderer.stats()
    assert st["primary_rays"] == n and st["shadow_rays"] == 0
    assert st["prim_tests"] == n * (len(tris) + len(sph))
    assert st["kernel_launches"] >= 1 and st["gpu_ms"] > 0
    # the cull runs: coherent camera rays leave well under a quarter of the ray/triangle pairs to the exact test
    assert 0 < st["exact_evals"] < n * len(tris) // 4, st
    renderer.rt_occluded(tris, sph, rays, np.full(n, 2.0, np.float32))
    st = renderer.stats()
    assert st["primary_rays"] == 0 and st["shadow_rays"] == n and st["prim_tests"] == n * (len(tris) + len(sph))
    renderer.set_option(b200.OPT_RT_BRUTEFORCE, 1)
    try:
        renderer.rt_closest_hits(tris, sph, rays)
        assert renderer.stats()["exact_evals"] == n * len(tris)
    finally:
        renderer.set_option(b200.OPT_RT_BRUTEFORCE, 0)


def test_invalid_arguments(b200, renderer, cornell_rt):
    tris, sph = cornell_rt
    lib, ctx = renderer.lib, renderer.ctx
    rays = rh.camera_rays(4, 4, 4.0, h.f32(0, 0, -3, 1), h.identity_R())
    md = np.ones(len(rays), np.float32)
    out = np.zeros(len(rays), rh.RT_INTERSECTION)
    occ = np.zeros(len(rays), np.uint8)
    P = h.ptr
    nt, ns = len(tris), len(sph)
    assert lib.rt_closest_hits(ctx, P(tris), nt, P(sph), ns, P(rays), -1, P(out)) == EINVAL
    assert lib.rt_closest_hits(ctx, P(tris), nt, P(sph), ns, None, len(rays), P(out)) == EINVAL
    assert lib.rt_closest_hits(ctx, P(tris), nt, P(sph), ns, P(rays), len(rays), None) == EINVAL
    assert lib.rt_closest_hits(ctx, None, nt, P(sph), ns, P(rays), len(rays), P(out)) == EINVAL
    assert lib.rt_closest_hits(ctx, P(tris), -1, P(sph), ns, P(rays), len(rays), P(out)) == EINVAL
    assert lib.rt_closest_hits(ctx, P(tris), nt, None, ns, P(rays), len(rays), P(out)) == EINVAL
    assert lib.rt_occluded(ctx, P(tris), nt, P(sph), ns, P(rays), None, len(rays), P(occ)) == EINVAL
    assert lib.rt_occluded(ctx, P(tris), nt, P(sph), ns, P(rays), P(md), len(rays), None) == EINVAL
    assert lib.rt_occluded(ctx, P(tris), nt, P(sph), -2, P(rays), P(md), len(rays), P(occ)) == EINVAL
    assert lib.rt_closest_hits_device(ctx, None, 5, None) == EINVAL
    assert lib.rt_closest_hits_device(ctx, None, -1, None) == EINVAL
    assert lib.rt_occluded_device(ctx, None, None, 3, None) == EINVAL
    assert lib.rt_closest_hits(None, P(tris), nt, P(sph), ns, P(rays), len(rays), P(out)) == EINVAL
    # n_rays == 0: OK, nothing written
    out[:] = np.frombuffer(b"\xab" * out.nbytes, rh.RT_INTERSECTION)
    before = out.tobytes()
    assert lib.rt_closest_hits(ctx, P(tris), nt, P(sph), ns, None, 0, None) == 0
    assert lib.rt_closest_hits(ctx, P(tris), nt, P(sph), ns, P(rays), 0, P(out)) == 0
    assert lib.rt_occluded(ctx, P(tris), nt, P(sph), ns, None, None, 0, None) == 0
    assert lib.rt_closest_hits_device(ctx, None, 0, None) == 0
    assert lib.rt_occluded_device(ctx, None, None, 0, None) == 0
    assert out.tobytes() == before


def test_multi_gpu_context(b200, cornell_rt):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    tris, sph = cornell_rt
    rays = np.concatenate([rh.camera_rays(200, 150, 150.0, h.f32(0, 0, -3, 1), h.yaw_R(0.2)), random_rays(1001, 9)])
    md = np.random.default_rng(4).uniform(0, 3, len(rays)).astype(np.float32)
    one = b200.Renderer(0)
    multi = b200.Renderer(n_gpus=min(torch.cuda.device_count(), 4))
    try:
        a, b = one.rt_closest_hits(tris, sph, rays), multi.rt_closest_hits(tris, sph, rays)
        for f in a:
            assert np.array_equal(np.ascontiguousarray(a[f]).tobytes(), np.ascontiguousarray(b[f]).tobytes()), f
        assert np.array_equal(one.rt_occluded(tris, sph, rays, md), multi.rt_occluded(tris, sph, rays, md))
        assert multi.stats()["primary_rays"] == 0 and multi.stats()["shadow_rays"] == len(rays)
        d = torch.zeros(64, dtype=torch.uint8, device="cuda")
        assert multi.lib.rt_closest_hits_device(multi.ctx, ctypes.c_void_p(d.data_ptr()), 1,
                                                ctypes.c_void_p(d.data_ptr())) == EINVAL
        assert multi.lib.rt_occluded_device(multi.ctx, ctypes.c_void_p(d.data_ptr()), ctypes.c_void_p(d.data_ptr()), 1,
                                            ctypes.c_void_p(d.data_ptr())) == EINVAL
    finally:
        one.close()
        multi.close()
