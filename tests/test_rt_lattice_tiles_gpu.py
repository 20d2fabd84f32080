"""rt_lattice_kernel streams the plane records through a ring of 64-record tiles, so scenes of more than 64 triangles
take several rounds of the ring in both the primary and the shadow phase (the light's records start a whole number of
256-record units after the camera's).  Random scenes just below, at and above the tile edges, up to the largest scene
that is still streamed whole, with and without a sphere and a light; each frame is compared with the oracle bit for
bit (colour, distance, index and the ray counts), and the launch timeline shows that the lattice kernel rendered it."""
import numpy as np
import pytest

import helpers as h
from test_rt_lattice_gpu import CAM, render_and_check, tl_renderer  # noqa: F401  (tl_renderer: fixture)

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n_tris", [63, 64, 65, 129, 1000])
@pytest.mark.parametrize("n_spheres", [0, 1])
@pytest.mark.parametrize("n_lights", [1, 0])
def test_scene_over_several_tiles(b200, tl_renderer, capfd, n_tris, n_spheres, n_lights):
    tris, sph = h.random_rt_scene(n_tris, seed=1000 + n_tris, n_spheres=n_spheres)
    lights = h.DEFAULT_RT_LIGHTS[:n_lights]
    W, H, focal = 48, 40, 40.0
    _, want, _ = render_and_check(b200, tl_renderer, capfd, tris, sph, W, H, focal, CAM, h.identity_R(), lights,
                                  f"{n_tris} triangles, {n_spheres} spheres, {n_lights} lights", kernel="rt_lattice_kernel")
    idx = want["index"]
    assert (idx >= 0).sum() > W * H // 4, "the scene should cover a good part of the frame"
    if n_tris > 64:   # hits on triangles of a later tile than the first
        assert (idx >= 64).any()
    if n_spheres:
        assert (idx == -1).any()
