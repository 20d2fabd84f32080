"""Python plumbing over the B200 renderer's C ABI (``include/b200render.h``).

The product is ``libb200render.so`` (hand-written CUDA for sm_100a behind an
``extern "C"`` boundary).  This module only loads it with ctypes and moves numpy
buffers across; tests and ``bench.py`` go through it so that everything they
exercise crosses the same ABI a C/C++ caller of the reference would bind.

There is no fallback of any kind: if the library is missing, or there is no CUDA
device, loading / ``Renderer()`` raises.

Import with ``importlib.import_module("computer-graphics_b200")`` (the directory
name is not a valid identifier).
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200render.so")

B200_OK, B200_EINVAL, B200_ECUDA, B200_ENOMEM, B200_ENODEV = 0, -1, -2, -3, -4
INDEX_MISS = -2147483648
OPT_RT_BRUTEFORCE = 1
OPT_RAST_TILE_LOG2 = 2
OPT_RAST_PATH = 3
OPT_RAST_PIPELINED = 4
OPT_RT_GRID = 5
OPT_RT_INTERLEAVE_N = 6
OPT_RT_INTERLEAVE_R = 7
OPT_RAST_BAND_CULL = 8
OPT_RAST_COLOUR_MODE = 9
OPT_RT_PLAN = 10

RT_TRI = np.dtype([("v0", "<f4", 4), ("v1", "<f4", 4), ("v2", "<f4", 4),
                   ("normal", "<f4", 4), ("color", "<f4", 3)])
RT_SPHERE = np.dtype([("radius", "<f4"), ("radius2", "<f4"), ("centre", "<f4", 3),
                      ("color", "<f4", 3), ("normal", "<f4", 3)])
RAST_TRI = np.dtype([("v0", "<f4", 4), ("v1", "<f4", 4), ("v2", "<f4", 4),
                     ("normal", "<f4", 4), ("color", "<f4", 3),
                     ("texture", "<i4"), ("index", "<i4")])


class Camera(ctypes.Structure):
    _fields_ = [("pos", ctypes.c_float * 4), ("focal", ctypes.c_float),
                ("R", ctypes.c_float * 16), ("width", ctypes.c_int32), ("height", ctypes.c_int32)]


class Light(ctypes.Structure):
    _fields_ = [("pos", ctypes.c_float * 4), ("colour", ctypes.c_float * 3)]


class RastLight(ctypes.Structure):
    _fields_ = [("pos", ctypes.c_float * 4), ("power", ctypes.c_float * 3),
                ("indirect", ctypes.c_float * 3)]


class RastImage(ctypes.Structure):
    _fields_ = [("data", ctypes.c_void_p), ("rows", ctypes.c_int32), ("cols", ctypes.c_int32), ("step", ctypes.c_int32)]


class RastTextures(ctypes.Structure):
    """rast_textures_t (include/b200render.h): the decoded images of the reference's texture globals."""
    _fields_ = [("marble", RastImage), ("marble_noise", ctypes.c_void_p), ("marble_noise_len", ctypes.c_int64),
                ("grill", RastImage), ("grill_opacity", RastImage), ("grill_normal", RastImage),
                ("woven", RastImage), ("woven_occlusion", RastImage), ("woven_opacity", RastImage),
                ("woven_normal", RastImage)]


class RtRay(ctypes.Structure):
    """rt_ray: the (start, dir) arguments of ClosestIntersection (32 bytes)."""
    _fields_ = [("start", ctypes.c_float * 4), ("dir", ctypes.c_float * 4)]


class RtIntersection(ctypes.Structure):
    """rt_intersection: the reference's `struct Intersection` (28 bytes, offsets 0 / 16 / 20 / 24)."""
    _fields_ = [("position", ctypes.c_float * 4), ("distance", ctypes.c_float),
                ("triangle_index", ctypes.c_int32), ("sphere_index", ctypes.c_int32)]


# numpy views of the same layouts
RT_RAY = np.dtype([("start", "<f4", 4), ("dir", "<f4", 4)])
RT_INTERSECTION = np.dtype([("position", "<f4", 4), ("distance", "<f4"), ("triangle_index", "<i4"),
                            ("sphere_index", "<i4")])


class Stats(ctypes.Structure):
    _fields_ = [("primary_rays", ctypes.c_uint64), ("shadow_rays", ctypes.c_uint64),
                ("prim_tests", ctypes.c_uint64), ("exact_evals", ctypes.c_uint64),
                ("kernel_launches", ctypes.c_uint64), ("fragments", ctypes.c_uint64),
                ("bin_entries", ctypes.c_uint64), ("respeculated", ctypes.c_uint64),
                ("gpu_ms", ctypes.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# Every symbol include/b200render.h declares; tests check they are all exported.
ABI_SYMBOLS = [
    "b200_init", "b200_init_multi", "b200_device_count", "b200_destroy", "b200_last_error", "b200_stream", "b200_synchronize",
    "b200_set_stream", "b200_set_option", "b200_get_stats",
    "b200_scene_cornell_rt", "b200_scene_cornell_rt_tessellated", "b200_scene_cornell_rast",
    "b200_scene_soup_rast",
    "render_raytrace", "render_raytrace_band", "draw_raytrace", "draw_raytrace_band",
    "b200_measure_fp32_peak", "rt_upload_scene", "rt_render_device",
    "render_raytrace_views", "draw_raytrace_views", "rt_render_views_device",
    "rt_closest_hits", "rt_occluded", "rt_closest_hits_device", "rt_occluded_device",
    "render_raster_clipped", "render_raster", "render_raster_band", "draw_raster", "raster_read_buffers",
    "raster_read_clipped", "rast_upload_clipped", "rast_render_device", "draw_raster_band",
    "rast_upload_scene", "rast_draw_device", "rast_set_textures",
    "b200_quantise", "b200_save_bmp",
]

_lib = None


def load_library():
    """Loads libb200render.so; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `make -C {_HERE}` "
                "(or __graft_entry__.build()); there is no fallback path")
        _lib = ctypes.CDLL(LIB_PATH)
        _lib.b200_last_error.restype = ctypes.c_char_p
        _lib.b200_stream.restype = ctypes.c_void_p
        vp, i32 = ctypes.c_void_p, ctypes.c_int
        _lib.rt_closest_hits.argtypes = [vp, vp, i32, vp, i32, vp, i32, vp]
        _lib.rt_occluded.argtypes = [vp, vp, i32, vp, i32, vp, vp, i32, vp]
        _lib.rt_closest_hits_device.argtypes = [vp, vp, i32, vp]
        _lib.rt_occluded_device.argtypes = [vp, vp, vp, i32, vp]
    return _lib


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, int):
        return ctypes.c_void_p(a)
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(ctypes.c_void_p)


def make_camera(pos, focal, R, width, height):
    c = Camera()
    c.pos[:] = [float(x) for x in pos]
    c.focal = float(focal)
    c.R[:] = [float(x) for x in np.asarray(R, np.float32).reshape(-1)]
    c.width, c.height = int(width), int(height)
    return c


def make_cameras(cams):
    """[Camera or (pos, focal, R, width, height), ...] -> ctypes array of camera_t (one per view)."""
    arr = (Camera * max(1, len(cams)))()
    for i, c in enumerate(cams):
        arr[i] = c if isinstance(c, Camera) else make_camera(*c)
    return arr


def _cameras(cams):
    """(ctypes array of camera_t, number of views) for a list of cameras or an array from make_cameras."""
    if isinstance(cams, ctypes.Array):
        return cams, len(cams)
    return make_cameras(cams), len(cams)


def make_lights(lights):
    """[(pos4, colour3), ...] -> ctypes array of light_t."""
    arr = (Light * max(1, len(lights)))()
    for i, (p, col) in enumerate(lights):
        arr[i].pos[:] = [float(x) for x in p]
        arr[i].colour[:] = [float(x) for x in col]
    return arr


def make_rast_light(pos, power, indirect):
    l = RastLight()
    l.pos[:] = [float(x) for x in pos]
    l.power[:] = [float(x) for x in power]
    l.indirect[:] = [float(x) for x in indirect]
    return l


class B200Error(RuntimeError):
    pass


class Renderer:
    """One context on one GPU (one process per GPU: pass LOCAL_RANK), or -- n_gpus given -- one
    context that shares every host-pointer frame among the first n_gpus devices of the box."""

    def __init__(self, device=0, n_gpus=None):
        self.lib = load_library()
        self.ctx = ctypes.c_void_p()
        if n_gpus is not None:
            rc = self.lib.b200_init_multi(int(n_gpus), ctypes.byref(self.ctx))
        else:
            rc = self.lib.b200_init(int(device), ctypes.byref(self.ctx))
        if rc != B200_OK:
            raise B200Error(f"b200_init(device={device}, n_gpus={n_gpus}) failed with code {rc} "
                            "(no CUDA device? there is no CPU fallback)")

    def device_count(self):
        return int(self.lib.b200_device_count(self.ctx))

    def close(self):
        if self.ctx:
            self.lib.b200_destroy(self.ctx)
            self.ctx = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != B200_OK:
            msg = self.lib.b200_last_error(self.ctx)
            raise B200Error(f"{what} failed with code {rc}: {msg.decode() if msg else ''}")

    def set_option(self, option, value):
        self._check(self.lib.b200_set_option(self.ctx, int(option), int(value)), "b200_set_option")

    def stats(self):
        s = Stats()
        self._check(self.lib.b200_get_stats(self.ctx, ctypes.byref(s)), "b200_get_stats")
        return s.as_dict()

    def stream(self):
        return self.lib.b200_stream(self.ctx)

    def set_stream(self, cuda_stream):
        self._check(self.lib.b200_set_stream(self.ctx, ctypes.c_void_p(cuda_stream or 0)), "b200_set_stream")

    def synchronize(self):
        self._check(self.lib.b200_synchronize(self.ctx), "b200_synchronize")

    # ---- RT ------------------------------------------------------------------
    def render_raytrace(self, tris, spheres, cam, lights, row_begin=0, row_end=None,
                        want=("rgb", "depth", "index")):
        W, H = cam.width, cam.height
        row_end = H if row_end is None else row_end
        rows = row_end - row_begin
        rgb = np.zeros((rows, W, 3), np.float32) if "rgb" in want else None
        depth = np.zeros((rows, W), np.float32) if "depth" in want else None
        index = np.zeros((rows, W), np.int32) if "index" in want else None
        la = make_lights(lights)
        rc = self.lib.render_raytrace_band(
            self.ctx, _ptr(tris), len(tris), _ptr(spheres), 0 if spheres is None else len(spheres),
            ctypes.byref(cam), la, len(lights), int(row_begin), int(row_end),
            _ptr(rgb), _ptr(depth), _ptr(index))
        self._check(rc, "render_raytrace_band")
        return dict(rgb=rgb, depth=depth, index=index)

    def draw_raytrace(self, tris, spheres, cam, lights, out=None):
        argb = np.zeros((cam.height, cam.width), np.uint32) if out is None else out
        la = make_lights(lights)
        rc = self.lib.draw_raytrace(self.ctx, _ptr(tris), len(tris), _ptr(spheres),
                                    0 if spheres is None else len(spheres), ctypes.byref(cam), la,
                                    len(lights), _ptr(argb))
        self._check(rc, "draw_raytrace")
        return argb

    def draw_raytrace_band(self, tris, spheres, cam, lights, row_begin, row_end, out_ptr):
        """out_ptr: host address (e.g. pinned memory) of a band-sized uint32 buffer."""
        la = make_lights(lights)
        rc = self.lib.draw_raytrace_band(self.ctx, _ptr(tris), len(tris), _ptr(spheres),
                                         0 if spheres is None else len(spheres), ctypes.byref(cam), la,
                                         len(lights), int(row_begin), int(row_end), _ptr(out_ptr))
        self._check(rc, "draw_raytrace_band")

    def measure_fp32_peak(self):
        v = ctypes.c_float(0)
        self._check(self.lib.b200_measure_fp32_peak(self.ctx, ctypes.byref(v)), "b200_measure_fp32_peak")
        return float(v.value)

    def rt_upload_scene(self, tris, spheres):
        rc = self.lib.rt_upload_scene(self.ctx, _ptr(tris), len(tris), _ptr(spheres),
                                      0 if spheres is None else len(spheres))
        self._check(rc, "rt_upload_scene")

    def rt_render_device(self, cam, lights, row_begin, row_end, d_rgb=None, d_depth=None,
                         d_index=None, d_argb=None):
        """Device pointers (ints) addressed as full frames; asynchronous."""
        la = make_lights(lights)
        rc = self.lib.rt_render_device(self.ctx, ctypes.byref(cam), la, len(lights), int(row_begin),
                                       int(row_end), _ptr(d_rgb), _ptr(d_depth), _ptr(d_index),
                                       _ptr(d_argb))
        self._check(rc, "rt_render_device")

    def render_raytrace_views(self, tris, spheres, cams, lights, want=("rgb", "depth", "index")):
        """Whole frames of every camera in `cams` (same width and height) in one call: arrays of shape
        (K, H, W, 3) / (K, H, W), view k equal to render_raytrace with cams[k]."""
        ca, k = _cameras(cams)
        W, H = (ca[0].width, ca[0].height) if k else (0, 0)
        rgb = np.zeros((k, H, W, 3), np.float32) if "rgb" in want else None
        depth = np.zeros((k, H, W), np.float32) if "depth" in want else None
        index = np.zeros((k, H, W), np.int32) if "index" in want else None
        la = make_lights(lights)
        rc = self.lib.render_raytrace_views(
            self.ctx, _ptr(tris), len(tris), _ptr(spheres), 0 if spheres is None else len(spheres),
            ca, int(k), la, len(lights), _ptr(rgb), _ptr(depth), _ptr(index))
        self._check(rc, "render_raytrace_views")
        return dict(rgb=rgb, depth=depth, index=index)

    def draw_raytrace_views(self, tris, spheres, cams, lights, out=None):
        """Packed frames of every camera in `cams`: (K, H, W) uint32."""
        ca, k = _cameras(cams)
        W, H = (ca[0].width, ca[0].height) if k else (0, 0)
        argb = np.zeros((k, H, W), np.uint32) if out is None else out
        la = make_lights(lights)
        rc = self.lib.draw_raytrace_views(self.ctx, _ptr(tris), len(tris), _ptr(spheres),
                                          0 if spheres is None else len(spheres), ca, int(k), la, len(lights),
                                          _ptr(argb))
        self._check(rc, "draw_raytrace_views")
        return argb

    def rt_render_views_device(self, cams, lights, d_rgb=None, d_depth=None, d_index=None, d_argb=None):
        """Every camera in `cams` on the uploaded scene into device pointers (ints) holding K whole frames
        back to back; asynchronous."""
        ca, k = _cameras(cams)
        la = make_lights(lights)
        rc = self.lib.rt_render_views_device(self.ctx, ca, int(k), la, len(lights), _ptr(d_rgb), _ptr(d_depth),
                                             _ptr(d_index), _ptr(d_argb))
        self._check(rc, "rt_render_views_device")

    # ---- RT, ray queries --------------------------------------------------------
    @staticmethod
    def _rays(rays):
        """rays: an RT_RAY array, or (n, 8) float32 (start xyzw, dir xyzw)."""
        rays = np.ascontiguousarray(rays)
        if rays.dtype != RT_RAY:
            rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 8).view(RT_RAY).reshape(-1)
        return rays

    def rt_closest_hits(self, tris, spheres, rays):
        """ClosestIntersection for every ray: dict of numpy arrays position (n, 4), distance, triangle_index and
        sphere_index (distance < FLT_MAX iff the ray hit something)."""
        rays = self._rays(rays)
        out = np.zeros(len(rays), RT_INTERSECTION)
        rc = self.lib.rt_closest_hits(self.ctx, _ptr(tris), 0 if tris is None else len(tris), _ptr(spheres),
                                      0 if spheres is None else len(spheres), _ptr(rays), len(rays), _ptr(out))
        self._check(rc, "rt_closest_hits")
        return dict(position=out["position"].copy(), distance=out["distance"].copy(),
                    triangle_index=out["triangle_index"].copy(), sphere_index=out["sphere_index"].copy())

    def rt_occluded(self, tris, spheres, rays, max_distance):
        """DirectLight's shadow test for every ray: bool array, ClosestIntersection && distance < max_distance."""
        rays = self._rays(rays)
        md = np.ascontiguousarray(max_distance, np.float32).reshape(-1)
        if len(md) != len(rays):
            raise ValueError("one max_distance per ray")
        out = np.zeros(len(rays), np.uint8)
        rc = self.lib.rt_occluded(self.ctx, _ptr(tris), 0 if tris is None else len(tris), _ptr(spheres),
                                  0 if spheres is None else len(spheres), _ptr(rays), _ptr(md), len(rays), _ptr(out))
        self._check(rc, "rt_occluded")
        return out.astype(bool)

    def rt_closest_hits_device(self, d_rays, n_rays, d_out):
        """Device pointers (ints): n_rays rt_ray in, rt_intersection out; the scene of rt_upload_scene; asynchronous."""
        self._check(self.lib.rt_closest_hits_device(self.ctx, _ptr(d_rays), int(n_rays), _ptr(d_out)),
                    "rt_closest_hits_device")

    def rt_occluded_device(self, d_rays, d_max_distance, n_rays, d_out):
        """Device pointers (ints): rt_ray and float limits in, one byte per ray out; asynchronous."""
        self._check(self.lib.rt_occluded_device(self.ctx, _ptr(d_rays), _ptr(d_max_distance), int(n_rays),
                                                _ptr(d_out)), "rt_occluded_device")

    # ---- RAST ----------------------------------------------------------------
    def render_raster_clipped(self, clipped, cam, light, want=("rgb", "depth", "index")):
        W, H = cam.width, cam.height
        rgb = np.zeros((H, W, 3), np.float32) if "rgb" in want else None
        depth = np.zeros((H, W), np.float32) if "depth" in want else None
        index = np.zeros((H, W), np.int32) if "index" in want else None
        rc = self.lib.render_raster_clipped(self.ctx, _ptr(clipped), len(clipped), ctypes.byref(cam),
                                            ctypes.byref(light), _ptr(rgb), _ptr(depth), _ptr(index))
        self._check(rc, "render_raster_clipped")
        return dict(rgb=rgb, depth=depth, index=index)

    def render_raster(self, room, boxes, cam, light, want=("rgb", "depth", "index"), row_begin=0, row_end=None):
        W, H = cam.width, cam.height
        row_end = H if row_end is None else row_end
        rows = row_end - row_begin
        rgb = np.zeros((rows, W, 3), np.float32) if "rgb" in want else None
        depth = np.zeros((rows, W), np.float32) if "depth" in want else None
        index = np.zeros((rows, W), np.int32) if "index" in want else None
        rc = self.lib.render_raster_band(self.ctx, _ptr(room), len(room), _ptr(boxes), len(boxes),
                                         ctypes.byref(cam), ctypes.byref(light), int(row_begin), int(row_end),
                                         _ptr(rgb), _ptr(depth), _ptr(index))
        self._check(rc, "render_raster_band")
        return dict(rgb=rgb, depth=depth, index=index)

    def draw_raster(self, room, boxes, cam, light, out=None):
        argb = np.zeros((cam.height, cam.width), np.uint32) if out is None else out
        rc = self.lib.draw_raster(self.ctx, _ptr(room), len(room), _ptr(boxes), len(boxes),
                                  ctypes.byref(cam), ctypes.byref(light), _ptr(argb))
        self._check(rc, "draw_raster")
        return argb

    def raster_read_buffers(self, W, H):
        screen = np.zeros((H, W, 3), np.float32)
        low = np.zeros((H, W, 3), np.float32)
        high = np.zeros((H, W, 3), np.float32)
        shadow = np.zeros((H, W), np.int32)
        rc = self.lib.raster_read_buffers(self.ctx, _ptr(screen), _ptr(low), _ptr(high), _ptr(shadow))
        self._check(rc, "raster_read_buffers")
        return dict(screen=screen, low=low, high=high, shadow=shadow)

    def raster_read_clipped(self, cap=1 << 22):
        n = ctypes.c_int(0)
        self._check(self.lib.raster_read_clipped(self.ctx, None, 0, ctypes.byref(n)), "raster_read_clipped")
        out = np.zeros(min(cap, n.value), RAST_TRI)
        self._check(self.lib.raster_read_clipped(self.ctx, _ptr(out), len(out), ctypes.byref(n)),
                    "raster_read_clipped")
        return out

    def set_textures(self, tex):
        """tex: dict of (rows, cols, channels) uint8 arrays named like rast_textures_t's images plus
        'marble_noise' ((n, 4) float32), or None to switch textures off (rast_set_textures)."""
        if tex is None:
            self._check(self.lib.rast_set_textures(self.ctx, None), "rast_set_textures")
            return
        t = RastTextures()
        keep = []
        for name in ("marble", "grill", "grill_opacity", "grill_normal", "woven", "woven_occlusion", "woven_opacity",
                     "woven_normal"):
            im = np.ascontiguousarray(tex[name], np.uint8)
            keep.append(im)
            setattr(t, name, RastImage(im.ctypes.data, im.shape[0], im.shape[1], im.shape[1] * (im.shape[2] if im.ndim == 3 else 1)))
        noise = np.ascontiguousarray(tex["marble_noise"], np.float32).reshape(-1, 4)
        t.marble_noise = noise.ctypes.data
        t.marble_noise_len = len(noise)
        self._check(self.lib.rast_set_textures(self.ctx, ctypes.byref(t)), "rast_set_textures")

    def rast_upload_clipped(self, clipped):
        self._check(self.lib.rast_upload_clipped(self.ctx, _ptr(clipped), len(clipped)), "rast_upload_clipped")

    def rast_upload_scene(self, room, boxes):
        self._check(self.lib.rast_upload_scene(self.ctx, _ptr(room), len(room), _ptr(boxes), len(boxes)),
                    "rast_upload_scene")

    def rast_draw_device(self, cam, light, row_begin, row_end, d_rgb=None, d_depth=None,
                         d_index=None, d_argb=None):
        rc = self.lib.rast_draw_device(self.ctx, ctypes.byref(cam), ctypes.byref(light),
                                       int(row_begin), int(row_end), _ptr(d_rgb), _ptr(d_depth),
                                       _ptr(d_index), _ptr(d_argb))
        self._check(rc, "rast_draw_device")

    def draw_raster_band(self, room, boxes, cam, light, row_begin, row_end, out_ptr):
        rc = self.lib.draw_raster_band(self.ctx, _ptr(room), len(room), _ptr(boxes), len(boxes),
                                       ctypes.byref(cam), ctypes.byref(light), int(row_begin),
                                       int(row_end), _ptr(out_ptr))
        self._check(rc, "draw_raster_band")

    def rast_render_device(self, cam, light, row_begin, row_end, d_rgb=None, d_depth=None,
                           d_index=None, d_argb=None):
        rc = self.lib.rast_render_device(self.ctx, ctypes.byref(cam), ctypes.byref(light),
                                         int(row_begin), int(row_end), _ptr(d_rgb), _ptr(d_depth),
                                         _ptr(d_index), _ptr(d_argb))
        self._check(rc, "rast_render_device")


def scene_cornell_rt():
    lib = load_library()
    tris, sph = np.zeros(28, RT_TRI), np.zeros(1, RT_SPHERE)
    nt, ns = ctypes.c_int(), ctypes.c_int()
    assert lib.b200_scene_cornell_rt(_ptr(tris), 28, _ptr(sph), 1, ctypes.byref(nt), ctypes.byref(ns)) == 0
    return tris, sph


def scene_cornell_rt_tessellated(n):
    lib = load_library()
    nt = ctypes.c_int()
    assert lib.b200_scene_cornell_rt_tessellated(int(n), None, 0, ctypes.byref(nt)) == 0
    tris = np.zeros(nt.value, RT_TRI)
    assert lib.b200_scene_cornell_rt_tessellated(int(n), _ptr(tris), len(tris), ctypes.byref(nt)) == 0
    return tris, scene_cornell_rt()[1]


def scene_cornell_rast():
    lib = load_library()
    room, boxes = np.zeros(10, RAST_TRI), np.zeros(20, RAST_TRI)
    a, b = ctypes.c_int(), ctypes.c_int()
    assert lib.b200_scene_cornell_rast(_ptr(room), 10, _ptr(boxes), 20, ctypes.byref(a), ctypes.byref(b)) == 0
    return room, boxes


def scene_soup_rast(n, seed=0x5EED, edge=0.01):
    lib = load_library()
    tris = np.zeros(int(n), RAST_TRI)
    assert lib.b200_scene_soup_rast(int(n), ctypes.c_uint32(seed), ctypes.c_float(edge), _ptr(tris)) == 0
    return tris


def quantise(rgb):
    lib = load_library()
    rgb = np.ascontiguousarray(rgb, np.float32)
    out = np.zeros(rgb.shape[:-1], np.uint32)
    lib.b200_quantise(_ptr(rgb), ctypes.c_size_t(out.size), _ptr(out))
    return out


def save_bmp(path, argb):
    lib = load_library()
    argb = np.ascontiguousarray(argb, np.uint32)
    rc = lib.b200_save_bmp(path.encode(), _ptr(argb), argb.shape[1], argb.shape[0])
    if rc != B200_OK:
        raise B200Error(f"b200_save_bmp({path}) failed with code {rc}")
