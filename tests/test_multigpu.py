"""Needs >= 2 GPUs (skipped otherwise): bands rendered by different GPUs, assembled on
rank 0 by peer stores and by an NCCL gather, equal the single-GPU frame bit for bit."""
import os
import subprocess
import sys

import pytest

import helpers as h

pytestmark = pytest.mark.gpu


def test_two_gpu_bands_equal_single_gpu_frame():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29533",
                          os.path.join(h.ROOT, "tests", "multigpu_check.py")],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "MULTIGPU_OK" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]


def _multi(b200):
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs 2 GPUs")
    return b200.Renderer(n_gpus=min(n, 8))


def test_library_multi_context_raytracer(b200, renderer):
    """b200_init_multi: the host-pointer entries share the frame among the devices by row bands
    (adaptive from the second frame on); every frame equals the single-device frame bit for bit."""
    import numpy as np
    m = _multi(b200)
    try:
        assert m.device_count() >= 2
        tris, sph = h.golden_cornell_rt()
        cam = b200.make_camera((0, 0, -3, 1), 200.0, h.identity_R(), 352, 200)
        want = renderer.render_raytrace(tris, sph, cam, h.DEFAULT_RT_LIGHTS)
        want_argb = renderer.draw_raytrace(tris, sph, cam, h.DEFAULT_RT_LIGHTS)
        for frame in range(3):
            got = m.render_raytrace(tris, sph, cam, h.DEFAULT_RT_LIGHTS)
            for k in ("rgb", "depth", "index"):
                assert np.array_equal(got[k].view(np.uint32), want[k].view(np.uint32)), (frame, k)
            assert np.array_equal(m.draw_raytrace(tris, sph, cam, h.DEFAULT_RT_LIGHTS), want_argb), frame
        st, st1 = m.stats(), renderer.stats()
        assert st["primary_rays"] == 352 * 200 * 9
        # a large scene (direction grids), a band of the frame only
        big, sph = h.scene_cornell_rt_tessellated(12)
        a = renderer.render_raytrace(big, sph, cam, h.DEFAULT_RT_LIGHTS, row_begin=40, row_end=171)
        b = m.render_raytrace(big, sph, cam, h.DEFAULT_RT_LIGHTS, row_begin=40, row_end=171)
        for k in ("rgb", "depth", "index"):
            assert np.array_equal(a[k].view(np.uint32), b[k].view(np.uint32)), k
        # the camera and row checks of a single context
        wide = b200.make_camera((0, 0, -3, 1), 200.0, h.identity_R(), 40000, 200)
        for c, r0, r1 in ((cam, 10, 5), (cam, 0, 201), (wide, 0, 200)):
            with pytest.raises(b200.B200Error):
                m.render_raytrace(tris, sph, c, h.DEFAULT_RT_LIGHTS, row_begin=r0, row_end=r1, want=())
        with pytest.raises(b200.B200Error):
            m.rt_upload_scene(tris, sph)          # device-pointer entries exist per device only
    finally:
        m.close()


def test_library_multi_context_rasteriser(b200, renderer):
    """Scene slices uploaded by different devices and all-gathered over NVLink, bands rendered
    concurrently, geometry culled to the band: equal to the single-device frame bit for bit."""
    import numpy as np
    m = _multi(b200)
    try:
        none = np.zeros(0, h.RAST_TRI)
        L = b200.make_rast_light(h.DEFAULT_RAST_LIGHT["pos"], h.DEFAULT_RAST_LIGHT["power"], h.DEFAULT_RAST_LIGHT["indirect"])
        L15 = b200.make_rast_light(h.DEFAULT_RAST_LIGHT["pos"], h.DEFAULT_RAST_LIGHT["power"], (0.15, 0.15, 0.15))
        room, boxes = b200.scene_cornell_rast()
        soup = b200.scene_soup_rast(40000, edge=0.03)            # 3.4 MB: takes the all-gather path
        for (rm, bx, W, H, f, light) in ((room, boxes, 320, 240, 170.0, L), (room, boxes, 320, 240, 170.0, L15),
                                         (soup, none, 640, 360, 256.0, L), (soup, none, 640, 360, 256.0, L15),
                                         (soup, boxes, 320, 200, 140.0, L)):
            cam = b200.make_camera(h.DEFAULT_RAST_CAM, f, h.identity_R(), W, H)
            want = renderer.render_raster(rm, bx, cam, light)
            want_argb = renderer.draw_raster(rm, bx, cam, light)
            for frame in range(3):                                # pipelined frames from the second on
                got = m.render_raster(rm, bx, cam, light)
                for k in ("rgb", "depth", "index"):
                    assert np.array_equal(got[k].view(np.uint32), want[k].view(np.uint32)), (len(rm), frame, k)
                assert np.array_equal(m.draw_raster(rm, bx, cam, light), want_argb), (len(rm), frame)
        assert m.stats()["fragments"] >= renderer.stats()["fragments"]      # bands overlap by their 2-row halos
        with pytest.raises(b200.B200Error):
            m.render_raster(room, boxes, cam, L, want=(), row_begin=10, row_end=5)
    finally:
        m.close()


def test_library_multi_context_textures_and_colour_modes(b200, renderer):
    """rast_set_textures on a multi-GPU context copies the images to every device; textured frames are
    shared by row bands like any other, colour-mode frames (whole-frame fragment ordinals) are drawn by
    the first device.  Equal to the single-device frames bit for bit."""
    import numpy as np
    m = _multi(b200)
    tex = h.synthetic_textures(3)
    try:
        room, boxes = h.golden_cornell_rast()
        room["texture"] = 2
        boxes["texture"] = 3
        L = b200.make_rast_light(h.DEFAULT_RAST_LIGHT["pos"], h.DEFAULT_RAST_LIGHT["power"], h.DEFAULT_RAST_LIGHT["indirect"])
        cam = b200.make_camera((0.1, -0.05, -2.6, 1.0), 170.0, h.yaw_R(0.174533), 320, 240)
        renderer.set_textures(tex)
        m.set_textures(tex)
        want = renderer.render_raster(room, boxes, cam, L)
        for frame in range(3):
            got = m.render_raster(room, boxes, cam, L)
            for k in ("rgb", "depth", "index"):
                assert np.array_equal(got[k].view(np.uint32), want[k].view(np.uint32)), (frame, k)
        for mode in (1, 2):
            renderer.set_option(b200.OPT_RAST_COLOUR_MODE, mode)
            m.set_option(b200.OPT_RAST_COLOUR_MODE, mode)
            h.srand(5)
            want = renderer.render_raster(room, boxes, cam, L)
            h.srand(5)
            got = m.render_raster(room, boxes, cam, L)
            for k in ("rgb", "depth", "index"):
                assert np.array_equal(got[k].view(np.uint32), want[k].view(np.uint32)), (mode, k)
    finally:
        renderer.set_option(b200.OPT_RAST_COLOUR_MODE, 0)
        renderer.set_textures(None)
        m.close()
