"""Generates the committed golden fixtures under tests/golden/.

Run in the development container, where /root/reference exists and the
unmodified reference has been compiled into oracle/_ref/ (oracle/refbuild/
build_ref.sh).  The GPU box has neither, so everything the `-m gpu` tests and
the oracle tests need from the reference is frozen here as small .npz files:

  rt_screenshot_320x256.npz  the reference's own golden image
                             raytracer/screenshot.bmp (KAT #2), as the uint32
                             ARGB pixel array top-down
  rt_cornell.npz             bytes of the reference's LoadTestModel scene
                             (28 triangles + 1 sphere)
  rt_ref_*.npz               outputs of the compiled reference (Draw float colour,
                             centre-sample distance / index) on seeded inputs
  rast_*.npz                 the same for the rasteriser (see make_rast below)
"""
import os
import struct
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import helpers as h  # noqa: E402

REF = os.environ.get("REF", "/root/reference")


def read_bmp32(path):
    b = open(path, "rb").read()
    off = struct.unpack_from("<I", b, 10)[0]
    w, hgt = struct.unpack_from("<ii", b, 18)
    bpp = struct.unpack_from("<H", b, 28)[0]
    assert bpp == 32
    px = np.frombuffer(b, np.uint32, count=w * abs(hgt), offset=off).reshape(abs(hgt), w)
    return px[::-1].copy() if hgt > 0 else px.copy()


def make_rt():
    px = read_bmp32(os.path.join(REF, "raytracer", "screenshot.bmp"))
    np.savez_compressed(os.path.join(HERE, "rt_screenshot_320x256.npz"), argb=px)
    tris, sph = h.ref_rt_testmodel()
    np.savez_compressed(os.path.join(HERE, "rt_cornell.npz"), tris=tris.view(np.uint8), spheres=sph.view(np.uint8))
    L = h.lights_array(h.DEFAULT_RT_LIGHTS)
    cases = {
        # name: (W, H, focal, cam, R, scene)
        "cornell_default_160x128": (160, 128, 128.0, h.f32(0, 0, -3, 1), h.identity_R(), None),
        "cornell_yaw_96x64": (96, 64, 64.0, h.f32(0.1, 0, -2.9, 1), h.yaw_R(-0.174533), None),
        "random40_96x64": (96, 64, 80.0, h.f32(0.1, -0.2, -2.5, 1), h.yaw_R(0.3), h.random_rt_scene(40, 7, n_spheres=2)),
    }
    for name, (W, H, f, cam, R, scene) in cases.items():
        t, s = scene if scene is not None else (None, None)
        d = h.ref_rt_draw(W, H, f, cam, R, L, t, s)
        tr = h.ref_rt_trace(W, H, f, cam, R, t, s)
        np.savez_compressed(os.path.join(HERE, f"rt_ref_{name}.npz"), W=W, H=H, focal=f, cam=cam, R=R,
                            lights=L, rgb=d["rgb"], argb=d["argb"], dist=tr["dist"], index=tr["index"],
                            tris=(t if t is not None else tris).view(np.uint8),
                            spheres=(s if s is not None else sph).view(np.uint8))
    print("rt goldens written")




def make_rast():
    """Rasteriser goldens: the compiled reference's whole Draw on its own Cornell
    box (untextured), with the clipped list it built and its buffers."""
    for (W, H, f, yaw, keys) in [(64, 48, 36.0, 0.0, ("rgb", "argb", "depth", "low", "high", "shadow", "screen_post")),
                                 (320, 240, 170.0, 0.0, ("rgb", "depth", "shadow")),
                                 (320, 240, 170.0, -0.174533, ("rgb", "depth", "shadow"))]:
        room, boxes = h.ref_rast_testmodel(W, H)
        R = h.yaw_R(yaw) if yaw else h.identity_R()
        r = h.ref_rast_draw(W, H, f, h.DEFAULT_RAST_CAM, R, h.DEFAULT_RAST_LIGHT, room, boxes)
        r2 = h.ref_rast_draw_clipped(W, H, f, r["light_cam"], h.DEFAULT_RAST_LIGHT, r["clipped"])
        assert np.array_equal(r2["rgb"].view(np.uint32), r["rgb"].view(np.uint32))
        out = {k: r[k] for k in keys}
        name = f"rast_ref_cornell_{W}x{H}" + ("_yaw" if yaw else "")
        np.savez_compressed(os.path.join(HERE, name + ".npz"), W=W, H=H, focal=f, cam=h.f32(*h.DEFAULT_RAST_CAM),
                            R=R, light_cam=r["light_cam"], clipped=r["clipped"].view(np.uint8),
                            room=room.view(np.uint8), boxes=boxes.view(np.uint8), index=r2["index"],
                            screen=r2["screen"] if W == 64 else np.zeros(0, np.float32), **out)
    # a random clipped list with shadow triangles, equal depths and off-screen parts
    W, H, f = 64, 48, 40.0
    tl = h.random_clipped_list(60, 5, W, H, f)
    lc = h.f32(0.1, -0.3, 1.2, 1.0)
    r = h.ref_rast_draw_clipped(W, H, f, lc, h.DEFAULT_RAST_LIGHT, tl)
    np.savez_compressed(os.path.join(HERE, "rast_ref_random60_64x48.npz"), W=W, H=H, focal=f, light_cam=lc,
                        clipped=tl.view(np.uint8), rgb=r["rgb"], argb=r["argb"], depth=r["depth"],
                        screen=r["screen"], low=r["low"], high=r["high"], shadow=r["shadow"], index=r["index"])
    print("rast goldens written")


def make_rast_textured():
    """The compiled reference's whole Draw with its texture branches (skeleton.cpp:588-645) on the
    synthetic images of helpers.synthetic_textures(seed): the settings the reference ships with (2, 1)
    straight on, and (3, 2) through the `yaw != 0` branch of findU / findV."""
    W, H, f, seed = 64, 48, 30.0, 7
    tex = h.synthetic_textures(seed)
    for tag, setting, setting_boxes, cam, yaw in [("a", 2, 1, h.DEFAULT_RAST_CAM, 0.0),
                                                  ("b", 3, 2, (0.1, -0.05, -2.6, 1.0), 0.174533)]:
        R = h.yaw_R(yaw) if yaw else h.identity_R()
        room, boxes = h.ref_rast_testmodel_tex(setting, setting_boxes, W, H)
        h.ref_rast_set_textures(W, H, tex, cam, R, yaw)
        r = h.ref_rast_draw(W, H, f, cam, R, h.DEFAULT_RAST_LIGHT, room, boxes)
        np.savez_compressed(os.path.join(HERE, f"rast_ref_cornell_tex_{tag}_{W}x{H}.npz"), W=W, H=H, focal=f, seed=seed,
                            cam=h.f32(*cam), R=R, yaw=yaw, room=room.view(np.uint8), boxes=boxes.view(np.uint8),
                            **{k: r[k] for k in ("rgb", "argb", "depth", "low", "high", "shadow", "screen_post")})
    print("textured rast goldens written")


def make_reference_textures():
    """The decoded pixels of the texture files in the reference's repository (rasteriser/Textures: metal grill and
    woven wood; cv2 = the decoder cv::imread uses; the two opacity maps grey + thresholded like main() :148-155), so
    that the GPU box -- which has neither the files nor /root/reference -- can draw with the real images
    (helpers.reference_textures).  The opacity maps whole, the other images thinned (helpers.coarse_texture):
    0.3 MB compressed."""
    tex = h.reference_textures(textures_dir=os.path.join(REF, "rasteriser", "Textures"))
    assert tex is not None, "the reference's texture files (or cv2) are not here"
    s = h.REF_TEX_STEP
    np.savez_compressed(os.path.join(HERE, "rast_reference_textures.npz"),
                        **{k: tex[k] if k.endswith("opacity") else tex[k][::s, ::s] for k in h.TEX_IMAGES if k != "marble"})
    print("reference textures written")


if __name__ == "__main__":
    if "textures" in sys.argv[1:]:
        make_reference_textures()
    elif "textured" in sys.argv[1:]:
        make_rast_textured()
    else:
        make_rt()
        make_rast()
        make_rast_textured()
        make_reference_textures()
