"""rt_direct_light and rt_direct_light_device: DirectLight for caller-supplied hits and lights, bit for bit against
the plain-C oracle (under the NaN rule of the header) and, composed with rt_closest_hits in Draw's order, against
whole frames of render_raytrace and the compiled reference."""
import ctypes

import numpy as np
import pytest

import helpers as h
import direct_light_helpers as dh
import rays_helpers as rh
from conftest import load_golden
from test_rt_rays_gpu import POSES

pytestmark = pytest.mark.gpu
FLT_MAX = np.finfo(np.float32).max
EINVAL = -1
X86_NAN = 0xFFC00000


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def lights7(lights):
    return h.lights_array(lights).reshape(-1, 7)


def as_array(hits):
    out = np.zeros(len(hits["distance"]), rh.RT_INTERSECTION)
    for f in rh.RT_INTERSECTION.names:
        out[f] = hits[f]
    return out


def assert_power_equal(got, want, nan_payload=True, what=""):
    """Bits equal; where the oracle's value is NaN the device must give NaN, and with nan_payload the x86 NaN."""
    g, w = bits(got).reshape(-1), bits(want).reshape(-1)
    wn = np.isnan(np.asarray(want, np.float32).reshape(-1))
    assert not np.any(g[~wn] != w[~wn]), f"{what}: {np.count_nonzero(g[~wn] != w[~wn])} components differ"
    assert np.all(np.isnan(np.asarray(got, np.float32).reshape(-1)[wn])), f"{what}: NaN expected"
    if nan_payload:
        assert np.all(g[wn] == X86_NAN) and np.all(w[wn] == X86_NAN), f"{what}: NaN bits"


def check_direct(renderer, tris, sph, hits, lights, nan_payload=True, what=""):
    got = renderer.rt_direct_light(tris, sph, hits, lights)
    want, _ = dh.oracle_rt_direct_light(tris, sph, as_array(hits) if isinstance(hits, dict) else hits, lights7(lights))
    assert got.shape == want.shape
    assert_power_equal(got, want, nan_payload, what)
    return got


MORE_LIGHTS = [((0.3, 0.7, -0.4, 1.0), (3, 4, 5)),        # inside the short box
               ((0.0, 0.0, 1.5, 1.0), (20, 20, 20)),       # behind the back wall
               ((0.0, -0.5, -0.7, 1.0), (14, 14, 14)),
               ((-0.3, 0.4, 0.2, 1.0), (2, 2, 2)),         # inside the tall box
               ((0.5, -0.9, 0.5, 1.0), (7, 1, 3)),
               ((-0.8, 0.8, -0.9, 1.0), (1, 9, 1)),
               ((0.0, 0.0, -2.0, 1.0), (30, 30, 30)),
               ((0.9, 0.0, 0.0, 0.0), (5, 5, 0.5))]


def composed_frame(renderer, tris, sph, W, H, f, cam, R, lights):
    rays = rh.camera_rays(W, H, f, cam, R, rh.NINE_SAMPLES)
    hits = as_array(renderer.rt_closest_hits(tris, sph, rays))
    power = renderer.rt_direct_light(tris, sph, hits, lights)
    return dh.draw_accumulate(hits, power, tris, sph).reshape(H, W, 3)


@pytest.mark.parametrize("name", ["cornell_default_160x128", "cornell_yaw_96x64", "random40_96x64"])
def test_composed_frame_equals_golden_and_render(b200, renderer, name):
    g = load_golden(f"rt_ref_{name}.npz")
    tris, sph = g["tris"].view(h.RT_TRI).copy(), g["spheres"].view(h.RT_SPHERE).copy()
    sph = sph if len(sph) else None
    W, H, f = int(g["W"]), int(g["H"]), float(g["focal"])
    L = g["lights"].reshape(-1, 7)
    lights = [(l[:4], l[4:]) for l in L]
    rgb = composed_frame(renderer, tris, sph, W, H, f, g["cam"], g["R"], lights)
    assert np.array_equal(bits(rgb), bits(g["rgb"]))
    frame = renderer.render_raytrace(tris, sph, b200.make_camera(g["cam"], f, g["R"], W, H), lights)
    assert np.array_equal(bits(rgb), bits(frame["rgb"]))


@pytest.mark.parametrize("n_lights", [1, 2, 5, 8])
@pytest.mark.parametrize("pose", range(3))
def test_composed_frame_equals_render_poses_and_lights(b200, renderer, cornell_rt, pose, n_lights):
    tris, sph = cornell_rt
    cam, R = POSES[pose]
    W, H, f = 96, 64, 64.0
    lights = h.DEFAULT_RT_LIGHTS if n_lights == 1 else MORE_LIGHTS[:n_lights]
    rgb = composed_frame(renderer, tris, sph, W, H, f, cam, R, lights)
    frame = renderer.render_raytrace(tris, sph, b200.make_camera(cam, f, R, W, H), lights)
    assert np.array_equal(bits(rgb), bits(frame["rgb"])), f"pose {pose}, {n_lights} lights"


def adversarial_hits(tris, sph, seed=7):
    """Entries and lights aimed at DirectLight's corners; returns (hits, lights, finite), finite = no NaN input."""
    rng = np.random.default_rng(seed)
    f = np.float32
    out = []

    def add(pos, ti=-1, si=-1, dist=1.0):
        e = np.zeros(1, rh.RT_INTERSECTION)
        e["position"][0] = np.asarray(list(pos)[:3] + [1.0], np.float32)
        e["distance"], e["triangle_index"], e["sphere_index"] = dist, ti, si
        out.append(e)

    for k, t in enumerate(tris):   # vertices and edge midpoints: ties between neighbouring triangles
        for p in (t["v0"][:3], t["v1"][:3], t["v2"][:3], ((t["v0"][:3] + t["v1"][:3]) * f(0.5)).astype(f),
                  ((t["v1"][:3] + t["v2"][:3]) * f(0.5)).astype(f)):
            add(p, ti=k)
    for _ in range(200):           # positions on no surface
        add(rng.uniform(-1.2, 1.2, 3).astype(f), ti=int(rng.integers(len(tris))))
        add(rng.uniform(-1.2, 1.2, 3).astype(f), si=0)
    for s_ in range(len(sph)):     # on, inside and at the centre of the sphere
        c, r = sph["centre"][s_].astype(f), f(sph["radius"][s_])
        add(c, si=s_)
        for _ in range(20):
            d = rng.normal(size=3).astype(f)
            d = (d / f(np.linalg.norm(d))).astype(f)
            add((c + d * r).astype(f), si=s_)
            add((c + d * (r * f(0.5))).astype(f), si=s_)
    for scale in (1e-30, 1e-10, 1e10, 1e30):   # magnitudes
        add((np.array([0.3, -0.2, 0.5], f) * f(scale)).astype(f), ti=3)
        add((np.array([0.3, -0.2, 0.5], f) * f(scale)).astype(f), si=0)
    add((np.inf, 0, 0), ti=2); add((0, -np.inf, 0.5), si=0)
    for ti, si in [(-1, -1), (len(tris), -1), (-2, 0), (-1, len(sph)), (-1, -5), (10**9, 0)]:   # name nothing
        add((0.1, 0.2, 0.3), ti=ti, si=si, dist=FLT_MAX if ti == -1 and si == -1 else 1.0)
    hits = np.concatenate(out)
    t0 = tris[8]   # back wall
    on_wall = ((t0["v0"][:3] + t0["v1"][:3] + t0["v2"][:3]) / f(3)).astype(f)
    add(on_wall, ti=8)
    lights = [((0.0, -0.5, -0.7, 1.0), (14, 14, 14)),
              (tuple(on_wall) + (1.0,), (9, 9, 9)),                 # in the wall's plane, and exactly at a hit
              ((0.2, 0.1, 1.7, 1.0), (5, 6, 7)),                    # behind the wall
              ((0.3, 0.7, -0.4, 1.0), (3, 3, 3)),
              ((1e30, 0.0, 0.0, 1.0), (1, 1, 1)),
              (tuple(sph["centre"][0]) + (1.0,), (2, 2, 2))]        # at the sphere's centre
    return np.concatenate(out), lights


def test_adversarial_entries_against_oracle(renderer, cornell_rt):
    tris, sph = cornell_rt
    hits, lights = adversarial_hits(tris, sph)
    got = check_direct(renderer, tris, sph, hits, lights, what="adversarial")
    assert np.isnan(got).any() and (got > 0).any() and (got == 0).any()
    named = (hits["triangle_index"] != -1) & (hits["triangle_index"] >= 0) & (hits["triangle_index"] < len(tris)) | \
        (hits["triangle_index"] == -1) & (hits["sphere_index"] >= 0) & (hits["sphere_index"] < len(sph))
    assert np.all(bits(got[~named]) == 0)
    # NaN inputs: positions and lights; only NaN-ness is compared
    nan_hits = hits.copy()
    nan_hits["position"][::5, 0] = np.nan
    nan_lights = lights[:2] + [((np.nan, 0.0, 0.0, 1.0), (1, 1, 1)), ((0.0, 0.0, 0.0, 1.0), (np.nan, 1, 1))]
    check_direct(renderer, tris, sph, nan_hits, nan_lights, nan_payload=False, what="NaN inputs")


@pytest.mark.parametrize("n_tris", [1, 64, 65, 200])
def test_random_scenes_against_oracle(renderer, n_tris):
    tris, sph = h.random_rt_scene(n_tris, 77 + n_tris, n_spheres=2)
    rays = rh.camera_rays(48, 32, 32.0, h.f32(0, 0, -3, 1), h.identity_R(), rh.NINE_SAMPLES[:3])
    hits = as_array(renderer.rt_closest_hits(tris, sph, rays))
    check_direct(renderer, tris, sph, hits, MORE_LIGHTS[:3], what=f"random {n_tris}")


def test_bruteforce_identical_and_culls(b200, renderer, cornell_rt):
    tris, sph = cornell_rt
    hits, lights = adversarial_hits(tris, sph)
    rays = rh.camera_rays(160, 128, 128.0, h.f32(0, 0, -3, 1), h.identity_R(), rh.NINE_SAMPLES)
    frame_hits = as_array(renderer.rt_closest_hits(tris, sph, rays))
    res = {}
    for brute in (0, 1):
        renderer.set_option(b200.OPT_RT_BRUTEFORCE, brute)
        try:
            a = renderer.rt_direct_light(tris, sph, hits, lights)
            b = renderer.rt_direct_light(tris, sph, frame_hits, MORE_LIGHTS[:5])
            res[brute] = (a, b, renderer.stats())
        finally:
            renderer.set_option(b200.OPT_RT_BRUTEFORCE, 0)
    assert np.array_equal(bits(res[0][0]), bits(res[1][0]))
    assert np.array_equal(bits(res[0][1]), bits(res[1][1]))
    assert res[0][2]["shadow_rays"] == res[1][2]["shadow_rays"] > 0
    assert res[1][2]["exact_evals"] == res[1][2]["shadow_rays"] * len(tris)
    assert res[0][2]["exact_evals"] < res[1][2]["exact_evals"] // 3, (res[0][2], res[1][2])


def device_chain(renderer, tris, sph, rays, lights):
    import torch
    renderer.rt_upload_scene(tris, sph)
    d_rays = torch.from_numpy(rays.view(np.uint8).copy()).cuda()
    d_hits = torch.full((len(rays) * 28,), 0xAB, dtype=torch.uint8, device="cuda")
    d_power = torch.full((len(rays) * len(lights) * 3,), float("nan"), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    renderer.rt_closest_hits_device(d_rays.data_ptr(), len(rays), d_hits.data_ptr())
    renderer.rt_direct_light_device(d_hits.data_ptr(), len(rays), lights, d_power.data_ptr())
    renderer.synchronize()
    return d_hits.cpu().numpy().view(rh.RT_INTERSECTION), d_power.cpu().numpy().reshape(len(rays), len(lights), 3)


def test_device_chain_equals_host_entry(renderer, cornell_rt):
    tris, sph = cornell_rt
    rays = rh.camera_rays(64, 48, 48.0, h.f32(0.1, 0, -2.8, 1), h.yaw_R(0.3), rh.NINE_SAMPLES)
    lights = MORE_LIGHTS[:4]
    hits, power = device_chain(renderer, tris, sph, rays, lights)
    host = renderer.rt_direct_light(tris, sph, hits, lights)
    assert np.array_equal(bits(power), bits(host))
    want, _ = dh.oracle_rt_direct_light(tris, sph, hits, lights7(lights))
    assert_power_equal(power, want, what="device chain")


def test_device_chain_tessellated_box(b200, renderer):
    tris, sph = h.scene_cornell_rt_tessellated(60)
    assert len(tris) == 100800
    rays = rh.camera_rays(50, 40, 40.0, h.f32(0, 0, -3, 1), h.identity_R())
    assert len(rays) == 2000
    lights = MORE_LIGHTS[2:4]
    hits, power = device_chain(renderer, tris, sph, rays, lights)
    want_hits = rh.oracle_rt_closest(tris, sph, rays)
    assert hits.tobytes() == want_hits.tobytes()
    want, _ = dh.oracle_rt_direct_light(tris, sph, want_hits, lights7(lights))
    assert_power_equal(power, want, what="tessellated")
    assert np.array_equal(bits(power), bits(renderer.rt_direct_light(tris, sph, hits, lights)))


def test_stats_and_context_state(b200, renderer, cornell_rt):
    tris, sph = cornell_rt
    hits, lights = adversarial_hits(tris, sph)
    renderer.rt_direct_light(tris, sph, hits, lights)
    st = renderer.stats()
    _, n_shadow = dh.oracle_rt_direct_light(tris, sph, hits, lights7(lights))
    ti, si = hits["triangle_index"], hits["sphere_index"]
    named = np.where(ti != -1, (ti >= 0) & (ti < len(tris)), (si >= 0) & (si < len(sph)))
    assert st["shadow_rays"] == named.sum() * len(lights) == n_shadow
    assert st["primary_rays"] == 0
    assert st["prim_tests"] == st["shadow_rays"] * (len(tris) + len(sph))
    assert st["kernel_launches"] >= 1 and st["gpu_ms"] > 0 and st["exact_evals"] > 0

    cam = b200.make_camera(h.f32(0, 0, -3, 1), 96.0, h.identity_R(), 128, 96)
    renderer.set_option(b200.OPT_RT_GRID, 1)
    try:
        a = renderer.render_raytrace(tris, sph, cam, h.DEFAULT_RT_LIGHTS)
        renderer.rt_direct_light(tris, sph, hits, lights)
        b = renderer.render_raytrace(tris, sph, cam, h.DEFAULT_RT_LIGHTS)
    finally:
        renderer.set_option(b200.OPT_RT_GRID, 0)
    for k in a:
        assert np.array_equal(np.ascontiguousarray(a[k]).view(np.uint32), np.ascontiguousarray(b[k]).view(np.uint32)), k


def test_invalid_arguments(b200, renderer, cornell_rt):
    tris, sph = cornell_rt
    lib, ctx, P = renderer.lib, renderer.ctx, h.ptr
    nt, ns = len(tris), len(sph)
    hits = as_array(renderer.rt_closest_hits(tris, sph, rh.camera_rays(4, 4, 4.0, h.f32(0, 0, -3, 1), h.identity_R())))
    n = len(hits)
    la = b200.make_lights(MORE_LIGHTS)
    out = np.zeros(n * 8 * 3, np.float32)
    assert lib.rt_direct_light(ctx, P(tris), nt, P(sph), ns, P(hits), -1, la, 1, P(out)) == EINVAL
    assert lib.rt_direct_light(ctx, P(tris), nt, P(sph), ns, P(hits), n, la, -1, P(out)) == EINVAL
    assert lib.rt_direct_light(ctx, P(tris), nt, P(sph), ns, P(hits), n, la, 9, P(out)) == EINVAL
    assert lib.rt_direct_light(ctx, P(tris), nt, P(sph), ns, None, n, la, 1, P(out)) == EINVAL
    assert lib.rt_direct_light(ctx, P(tris), nt, P(sph), ns, P(hits), n, la, 1, None) == EINVAL
    assert lib.rt_direct_light(ctx, P(tris), nt, P(sph), ns, P(hits), n, None, 1, P(out)) == EINVAL
    assert lib.rt_direct_light(ctx, P(tris), nt, P(sph), ns, P(hits), 0, None, 1, P(out)) == EINVAL
    assert lib.rt_direct_light(ctx, None, nt, P(sph), ns, P(hits), n, la, 1, P(out)) == EINVAL
    assert lib.rt_direct_light(ctx, P(tris), -1, P(sph), ns, P(hits), n, la, 1, P(out)) == EINVAL
    assert lib.rt_direct_light(ctx, P(tris), nt, None, ns, P(hits), n, la, 1, P(out)) == EINVAL
    assert lib.rt_direct_light(None, P(tris), nt, P(sph), ns, P(hits), n, la, 1, P(out)) == EINVAL
    assert lib.rt_direct_light_device(ctx, None, -1, la, 1, None) == EINVAL
    assert lib.rt_direct_light_device(ctx, None, 5, la, 1, None) == EINVAL
    assert lib.rt_direct_light_device(ctx, None, 5, la, 9, None) == EINVAL
    assert lib.rt_direct_light_device(ctx, None, 5, None, 2, None) == EINVAL
    # n_hits == 0 or n_lights == 0: OK, a poisoned output untouched
    out[:] = np.frombuffer(b"\xab" * out.nbytes, np.float32)
    before = out.tobytes()
    assert lib.rt_direct_light(ctx, P(tris), nt, P(sph), ns, None, 0, la, 3, None) == 0
    assert lib.rt_direct_light(ctx, P(tris), nt, P(sph), ns, P(hits), 0, la, 3, P(out)) == 0
    assert lib.rt_direct_light(ctx, P(tris), nt, P(sph), ns, P(hits), n, None, 0, P(out)) == 0
    assert lib.rt_direct_light(ctx, P(tris), nt, P(sph), ns, None, n, la, 0, None) == 0
    assert lib.rt_direct_light_device(ctx, None, 0, la, 2, None) == 0
    assert lib.rt_direct_light_device(ctx, None, 7, None, 0, None) == 0
    assert out.tobytes() == before


def test_multi_gpu_context(b200, cornell_rt):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    tris, sph = cornell_rt
    hits, lights = adversarial_hits(tris, sph)
    one = b200.Renderer(0)
    multi = b200.Renderer(n_gpus=min(torch.cuda.device_count(), 4))
    try:
        a, b = one.rt_direct_light(tris, sph, hits, lights), multi.rt_direct_light(tris, sph, hits, lights)
        assert a.tobytes() == b.tobytes()
        assert multi.stats()["shadow_rays"] == one.stats()["shadow_rays"] and multi.stats()["primary_rays"] == 0
        d = torch.zeros(64, dtype=torch.uint8, device="cuda")
        assert multi.lib.rt_direct_light_device(multi.ctx, ctypes.c_void_p(d.data_ptr()), 1, b200.make_lights(lights), 1,
                                                ctypes.c_void_p(d.data_ptr())) == EINVAL
    finally:
        one.close()
        multi.close()
