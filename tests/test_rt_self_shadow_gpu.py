"""The shadow ray against the triangle it starts on.  The render kernel decides that pair from the
sign of the reference's D, known per (light, triangle) from the frame's preparation, and Dt formed
inline in the reference's arithmetic; every other case runs the reference arithmetic.  These frames
reach each branch and are compared with the oracle bit for bit."""
import numpy as np
import pytest

import helpers as h
from test_rt_gpu import check_equal, run_both

pytestmark = pytest.mark.gpu


def test_self_pairs_skip_the_exact_call(b200, renderer, cornell_rt):
    """Most shadow rays start on a surface that faces the light: their own triangle no longer runs the
    reference arithmetic.  Each primary hit needs at least one exact evaluation (its distance) and, with
    one light, starts one shadow ray; with every self pair exact, exact_evals was at least twice
    shadow_rays."""
    tris, sph = cornell_rt
    _, _, st = run_both(b200, renderer, tris, sph, 320, 256, 256.0, h.f32(0, 0, -3, 1), h.identity_R(),
                        h.DEFAULT_RT_LIGHTS, "cornell 320x256", brute=False)
    assert st["shadow_rays"] > 0
    assert st["exact_evals"] < 1.6 * st["shadow_rays"], (st["exact_evals"], st["shadow_rays"])


def test_surfaces_facing_away_from_the_light(b200, renderer, cornell_rt):
    """Lights outside the room and behind the boxes: many visible faces have the light behind them,
    so the pair can occlude and the reference arithmetic decides it."""
    tris, sph = cornell_rt
    for lights in ([((0.0, -0.5, 1.6, 1.0), (14, 14, 14))],
                   [((0.7, 0.3, 0.6, 1.0), (9, 9, 9)), ((-1.4, -0.2, -0.4, 1.0), (4, 5, 6))]):
        run_both(b200, renderer, tris, sph, 96, 80, 80.0, h.f32(0.05, -0.1, -2.8, 1), h.yaw_R(0.15), lights,
                 f"lights behind surfaces {lights[0][0]}", brute=False)


def test_light_close_to_a_wall_plane(b200, renderer, cornell_rt):
    """A light within 1e-4 of the plane of the largest triangle: the sign of D is not known for the
    triangles of that plane, which fall back to the reference arithmetic."""
    tris, sph = cornell_rt
    v0, v1, v2 = (tris[k][:, :3].astype(np.float64) for k in ("v0", "v1", "v2"))
    area = np.linalg.norm(np.cross(v1 - v0, v2 - v0), axis=1)
    i = int(area.argmax())
    n = np.cross(v1[i] - v0[i], v2[i] - v0[i])
    n /= np.linalg.norm(n)
    centre = (v0[i] + v1[i] + v2[i]) / 3.0
    inward = n if np.dot(n, -centre) > 0 else -n          # towards the middle of the room
    for d in (1e-4, 3e-6):
        pos = (centre + d * inward).astype(np.float32)
        lights = [((float(pos[0]), float(pos[1]), float(pos[2]), 1.0), (14, 14, 14))]
        run_both(b200, renderer, tris, sph, 96, 80, 80.0, h.f32(0, 0, -3, 1), h.identity_R(), lights,
                 f"light {d} from a wall plane", brute=False)


def test_flipped_and_scaled_normals(b200, renderer, cornell_rt):
    """Caller-supplied normals that point away from the light or are far from unit length: the start
    offset 1e-5 * normal moves to the other side of the plane, and n_scale > 1 widens the bounds."""
    tris, sph = cornell_rt
    tris = tris.copy()
    tris["normal"][::2, :3] *= np.float32(-1.0)
    tris["normal"][1::3, :3] *= np.float32(57.0)
    tris["normal"][::5, :3] *= np.float32(0.02)
    run_both(b200, renderer, tris, sph, 96, 80, 80.0, h.f32(0, 0, -3, 1), h.identity_R(), h.DEFAULT_RT_LIGHTS,
             "flipped and scaled normals", brute=False)


def test_tilted_normals_make_the_own_triangle_occlude(b200, renderer, cornell_rt):
    """Caller-supplied normals tilted far from the geometric normal: mostly along the wall towards the light,
    a little into the wall.  The start hit + 1e-5 * normal then lies behind the triangle's plane, the shadow
    ray crosses its own triangle and the reference turns the pixel's direct light off, while normal . r > 0
    would have lit it.  A self pair decided with the wrong sign of D changes these pixels."""
    tris, sph = cornell_rt
    tris = tris.copy()
    L = np.array(h.DEFAULT_RT_LIGHTS[0][0][:3], np.float64)
    v0, v1, v2 = (tris[k][:, :3].astype(np.float64) for k in ("v0", "v1", "v2"))
    N = np.cross(v1 - v0, v2 - v0)
    N /= np.linalg.norm(N, axis=1, keepdims=True)
    to_l = L - (v0 + v1 + v2) / 3.0
    N *= np.sign(np.einsum("ij,ij->i", to_l, N))[:, None]                 # towards the light
    along = to_l - np.einsum("ij,ij->i", to_l, N)[:, None] * N
    along /= np.linalg.norm(along, axis=1, keepdims=True)
    tris["normal"][:, :3] = (50.0 * (along - 0.05 * N)).astype(np.float32)
    got, want, _ = run_both(b200, renderer, tris, sph, 96, 80, 80.0, h.f32(0, 0, -3, 1), h.identity_R(),
                            h.DEFAULT_RT_LIGHTS, "tilted normals", brute=False)
    # the scene does what it is for: most triangle hits are in their own shadow, which the lit colour would not be
    plain = renderer.render_raytrace(cornell_rt[0], sph, b200.make_camera(h.f32(0, 0, -3, 1), 80.0, h.identity_R(), 96, 80),
                                     h.DEFAULT_RT_LIGHTS)
    tri_hit = want["index"] >= 0
    darker = (want["rgb"].sum(axis=-1) < plain["rgb"].sum(axis=-1)) & tri_hit
    assert darker.sum() > 0.25 * tri_hit.sum()


def test_tessellated_100k_rows_match_the_oracle(b200, renderer):
    """The 100 800-triangle box through the direction grids (which decide every self pair with the reference
    arithmetic and get no self-pair signs), a band of rows against the oracle."""
    tris, sph = b200.scene_cornell_rt_tessellated(60)
    W, H, f, r0, r1 = 64, 48, 48.0, 20, 24
    cam = h.f32(0.013, -0.021, -3.02, 1)
    c = b200.make_camera(cam, f, h.identity_R(), W, H)
    want = h.oracle_rt_render(W, H, f, cam, h.identity_R(), h.lights_array(h.DEFAULT_RT_LIGHTS), tris, sph, r0, r1)
    want = {k: (v[r0:r1] if isinstance(v, np.ndarray) else v) for k, v in want.items()}
    renderer.set_option(b200.OPT_RT_GRID, 1)
    try:
        for frame in range(2):
            got = renderer.render_raytrace(tris, sph, c, h.DEFAULT_RT_LIGHTS, r0, r1)
            check_equal(got, want, f"tessellated 100800, rows {r0}-{r1}, frame {frame}")
            assert renderer.stats()["shadow_rays"] == want["shadow"]
    finally:
        renderer.set_option(b200.OPT_RT_GRID, 0)
