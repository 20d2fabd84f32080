"""Frames whose sample rays form a half-pixel lattice run rt_lattice_kernel, which traces each ray that neighbouring
pixels share once per 16x16 block; every other frame runs rt_filtered_kernel.  Each case is compared with the oracle
bit for bit (colour, distance, index and the ray counts), and the launch timeline (B200_TIMELINE) shows which kernel
rendered it.  Which one it must be follows from the rule restated here in float32: R[1] = R[4] = 0, and sample 2 of
each pixel has the bits of sample 0 of its right (lower) neighbour."""
import os
import re

import numpy as np
import pytest

import helpers as h
from test_rt_gpu import bits, check_equal

pytestmark = pytest.mark.gpu

TL = re.compile(r"^\[b200 timeline\] (.+?)\s+-?[0-9.]+ us$")


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


def launched(capfd):
    names = []
    for line in capfd.readouterr().err.splitlines():
        m = TL.match(line.strip())
        if m and m.group(1) != "frame":
            names.append(m.group(1))
    return names


def lattice_exact(W, H, focal, R, row0, row1):
    """The host's rule, in the kernel's float32 arithmetic (numpy rounds every operation)."""
    R = np.asarray(R, np.float32)
    f32 = np.float32
    if R[1] != 0 or R[4] != 0:
        return False

    def d(r, x, y):
        return (R[r] * f32(x) + R[4 + r] * f32(y)) + (R[8 + r] * f32(focal) + R[12 + r] * f32(1.0))

    with np.errstate(all="ignore"):
        for r, lo, hi in ((0, 0, W), (1, row0, row1)):
            c = np.arange(lo, hi)
            dd = d(0, (c - W // 2).astype(np.float32), row0 - H // 2) if r == 0 else \
                d(1, -(W // 2), (c - H // 2).astype(np.float32))
            s0, s1, s2 = dd + f32(-0.5), dd + f32(0.0), dd + f32(0.5)
            if not (np.isfinite(s0).all() and np.isfinite(s1).all() and np.isfinite(s2).all()):
                return False
            if not np.array_equal(s0[1:].view(np.uint32), s2[:-1].view(np.uint32)):
                return False
    return True


def render_and_check(b200, r, capfd, tris, sph, W, H, focal, cam, R, lights, what, row0=0, row1=None, kernel=None):
    row1 = H if row1 is None else row1
    expect = "rt_lattice_kernel" if len(lights) <= 1 and lattice_exact(W, H, focal, R, row0, row1) else "rt_filtered_kernel"
    if kernel is not None:
        assert expect == kernel, f"{what}: the case was meant for {kernel}"
    want = h.oracle_rt_render(W, H, focal, cam, R, h.lights_array(lights), tris, sph, row0, row1)
    c = b200.make_camera(cam, focal, R, W, H)
    capfd.readouterr()
    got = r.render_raytrace(tris, sph, c, lights, row0, row1)
    st = r.stats()
    names = launched(capfd)
    assert expect in names, f"{what}: {expect} missing from the launches {names}"
    other = "rt_filtered_kernel" if expect == "rt_lattice_kernel" else "rt_lattice_kernel"
    assert other not in names, f"{what}: {other} in the launches {names}"
    check_equal(got, {k: (v[row0:row1] if isinstance(v, np.ndarray) else v) for k, v in want.items()}, what)
    assert st["primary_rays"] == want["primary"] and st["shadow_rays"] == want["shadow"], (what, st, want["primary"], want["shadow"])
    return got, want, st


def translated(x, y):
    R = h.identity_R()
    R[12], R[13] = np.float32(x), np.float32(y)
    return R


CAM = h.f32(0, 0, -3, 1)


@pytest.mark.parametrize("W,H,focal,row0,row1", [
    (83, 45, 60.0, 0, 45),        # odd width and height: partial blocks on the right and at the bottom
    (160, 128, 128.0, 0, 128),
    (83, 45, 60.0, 5, 37),        # a band whose first row is not a multiple of 16
    (97, 70, 64.0, 19, 20),       # one row
    (1, 1, 1.0, 0, 1),
])
def test_identity_camera(b200, tl_renderer, capfd, cornell_rt, W, H, focal, row0, row1):
    tris, sph = cornell_rt
    render_and_check(b200, tl_renderer, capfd, tris, sph, W, H, focal, CAM, h.identity_R(), h.DEFAULT_RT_LIGHTS,
                     f"{W}x{H} rows {row0}-{row1}", row0, row1, kernel="rt_lattice_kernel")


def test_sphere_in_view(b200, tl_renderer, capfd, cornell_rt):
    tris, sph = cornell_rt
    _, want, _ = render_and_check(b200, tl_renderer, capfd, tris, sph, 120, 96, 96.0, h.f32(0.1, 0.05, -2.6, 1),
                                  h.identity_R(), h.DEFAULT_RT_LIGHTS, "sphere in view", kernel="rt_lattice_kernel")
    assert (want["index"] == -1).sum() > 100          # sphere 0 is hit


@pytest.mark.parametrize("x,y", [(7.0, -4.0), (-31.0, 12.0), (2.5, -1.5), (-0.5, 0.5)])
def test_integer_and_half_integer_translation(b200, tl_renderer, capfd, cornell_rt, x, y):
    """Windows of a larger frame, as bench.window_R makes them."""
    tris, sph = cornell_rt
    render_and_check(b200, tl_renderer, capfd, tris, sph, 75, 50, 64.0, CAM, translated(x, y), h.DEFAULT_RT_LIGHTS,
                     f"translation {x}, {y}", kernel="rt_lattice_kernel")


def test_translation_that_breaks_the_lattice(b200, tl_renderer, capfd, cornell_rt):
    """dir0 + 0.5 and dir0(u + 1) - 0.5 round differently for some u: the per-pixel kernel renders it."""
    tris, sph = cornell_rt
    R = translated(0.1, 0.0)
    assert not lattice_exact(75, 50, 64.0, R, 0, 50)
    render_and_check(b200, tl_renderer, capfd, tris, sph, 75, 50, 64.0, CAM, R, h.DEFAULT_RT_LIGHTS,
                     "translation 0.1", kernel="rt_filtered_kernel")


def test_yaw_falls_back(b200, tl_renderer, capfd, cornell_rt):
    tris, sph = cornell_rt
    render_and_check(b200, tl_renderer, capfd, tris, sph, 75, 50, 64.0, CAM, h.yaw_R(0.2), h.DEFAULT_RT_LIGHTS,
                     "yaw", kernel="rt_filtered_kernel")


def test_light_count(b200, tl_renderer, capfd, cornell_rt):
    """No light: colour only, on the lattice.  Two lights: the per-pixel kernel."""
    tris, sph = cornell_rt
    render_and_check(b200, tl_renderer, capfd, tris, sph, 75, 50, 64.0, CAM, h.identity_R(), [], "no light",
                     kernel="rt_lattice_kernel")
    two = [((0.2, -0.4, -0.9, 1), (10, 12, 14)), ((-0.5, 0.3, -1.2, 1), (3, 2, 1))]
    render_and_check(b200, tl_renderer, capfd, tris, sph, 75, 50, 64.0, CAM, h.identity_R(), two, "two lights",
                     kernel="rt_filtered_kernel")


def test_light_on_a_wall_plane(b200, tl_renderer, capfd, cornell_rt):
    """A light within 1e-4 / 3e-6 of the largest triangle's plane (as in test_rt_self_shadow_gpu): the sign of the
    self pair's D is not known there, the reference arithmetic decides."""
    tris, sph = cornell_rt
    v0, v1, v2 = (tris[k][:, :3].astype(np.float64) for k in ("v0", "v1", "v2"))
    i = int(np.linalg.norm(np.cross(v1 - v0, v2 - v0), axis=1).argmax())
    n = np.cross(v1[i] - v0[i], v2[i] - v0[i])
    n /= np.linalg.norm(n)
    centre = (v0[i] + v1[i] + v2[i]) / 3.0
    inward = n if np.dot(n, -centre) > 0 else -n
    for d in (1e-4, 3e-6, 0.0):
        pos = (centre + d * inward).astype(np.float32)
        lights = [((float(pos[0]), float(pos[1]), float(pos[2]), 1.0), (14, 14, 14))]
        render_and_check(b200, tl_renderer, capfd, tris, sph, 96, 80, 80.0, CAM, h.identity_R(), lights,
                         f"light {d} from a wall plane", kernel="rt_lattice_kernel")


def test_tilted_and_flipped_normals(b200, tl_renderer, capfd, cornell_rt):
    """The self-pair scenes of test_rt_self_shadow_gpu: the shadow ray's own triangle occludes it, or the normal
    points away from the light."""
    tris, sph = cornell_rt
    L = np.array(h.DEFAULT_RT_LIGHTS[0][0][:3], np.float64)
    t = tris.copy()
    v0, v1, v2 = (t[k][:, :3].astype(np.float64) for k in ("v0", "v1", "v2"))
    N = np.cross(v1 - v0, v2 - v0)
    N /= np.linalg.norm(N, axis=1, keepdims=True)
    to_l = L - (v0 + v1 + v2) / 3.0
    N *= np.sign(np.einsum("ij,ij->i", to_l, N))[:, None]
    along = to_l - np.einsum("ij,ij->i", to_l, N)[:, None] * N
    along /= np.linalg.norm(along, axis=1, keepdims=True)
    t["normal"][:, :3] = (50.0 * (along - 0.05 * N)).astype(np.float32)
    render_and_check(b200, tl_renderer, capfd, t, sph, 96, 80, 80.0, CAM, h.identity_R(), h.DEFAULT_RT_LIGHTS,
                     "tilted normals", kernel="rt_lattice_kernel")
    t = tris.copy()
    t["normal"][::2, :3] *= np.float32(-1.0)
    t["normal"][1::3, :3] *= np.float32(57.0)
    t["normal"][::5, :3] *= np.float32(0.02)
    render_and_check(b200, tl_renderer, capfd, t, sph, 96, 80, 80.0, CAM, h.identity_R(), h.DEFAULT_RT_LIGHTS,
                     "flipped and scaled normals", kernel="rt_lattice_kernel")


def test_interleaved_launches(b200, tl_renderer, capfd, cornell_rt):
    """OPT_RT_INTERLEAVE_N/R: three launches of every third 16-row block of a band fill the oracle's frame."""
    import torch
    tris, sph = cornell_rt
    r = tl_renderer
    W, H, focal = 150, 117, 100.0
    c = b200.make_camera(CAM, focal, h.identity_R(), W, H)
    r.rt_upload_scene(tris, sph)
    try:
        for row0, row1 in ((0, H), (5, 101)):
            assert lattice_exact(W, H, focal, h.identity_R(), row0, row1)
            want = h.oracle_rt_render(W, H, focal, CAM, h.identity_R(), h.lights_array(h.DEFAULT_RT_LIGHTS), tris, sph,
                                      row0, row1)
            rgb = torch.full((H, W, 3), float("nan"), device="cuda")
            depth = torch.full((H, W), float("nan"), device="cuda")
            index = torch.full((H, W), 12345, dtype=torch.int32, device="cuda")
            primary = shadow = 0
            for k in range(3):
                r.set_option(b200.OPT_RT_INTERLEAVE_N, 3)
                r.set_option(b200.OPT_RT_INTERLEAVE_R, k)
                capfd.readouterr()
                r.rt_render_device(c, h.DEFAULT_RT_LIGHTS, row0, row1, rgb.data_ptr(), depth.data_ptr(), index.data_ptr())
                st = r.stats()
                names = launched(capfd)
                assert "rt_lattice_kernel" in names and "rt_filtered_kernel" not in names, names
                primary += st["primary_rays"]; shadow += st["shadow_rays"]
            got = dict(rgb=rgb.cpu().numpy()[row0:row1], depth=depth.cpu().numpy()[row0:row1],
                       index=index.cpu().numpy()[row0:row1])
            check_equal(got, {k: (v[row0:row1] if isinstance(v, np.ndarray) else v) for k, v in want.items()},
                        f"interleaved rows {row0}-{row1}")
            assert (index.cpu().numpy()[:row0] == 12345).all() and (index.cpu().numpy()[row1:] == 12345).all()
            assert np.isnan(bits(rgb.cpu().numpy()[:row0]).view(np.float32)).all()
            assert primary == want["primary"] and shadow == want["shadow"]
    finally:
        r.set_option(b200.OPT_RT_INTERLEAVE_N, 1)
        r.set_option(b200.OPT_RT_INTERLEAVE_R, 0)
