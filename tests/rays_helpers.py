"""Test plumbing of the RT ray queries: the numpy layouts of rt_ray / rt_intersection, the plain-C oracle's
ray-query entries (oracle/rays/oracle_rt_rays.c, which includes oracle/oracle_rt.c and calls its
closest_intersection unchanged), and the rays of the reference's Draw and DirectLight.

Nothing here is product code.
"""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from helpers import ORACLE_DIR, c_i, ptr

RAYS_SRC = os.path.join(ORACLE_DIR, "rays", "oracle_rt_rays.c")
# oracle/Makefile's flags: one IEEE rounding per operation, like the reference's own build
CFLAGS = ["-O2", "-std=gnu11", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-shared"]
_lib = None


def rays_oracle():
    """liboracle_rays.so, compiled on first use into the temporary directory (the tree may be read-only), named
    by a hash of the sources and flags."""
    global _lib
    if _lib is None:
        key = hashlib.sha256()
        for p in (RAYS_SRC, os.path.join(ORACLE_DIR, "oracle_rt.c")):
            key.update(open(p, "rb").read())
        key.update(" ".join(CFLAGS).encode())
        path = os.path.join(tempfile.gettempdir(), f"liboracle_rays_{key.hexdigest()[:16]}_{os.getuid()}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.check_call([os.environ.get("CC", "gcc"), *CFLAGS, "-o", tmp, RAYS_SRC, "-lm"])
            os.replace(tmp, path)
        _lib = ctypes.CDLL(path)
    return _lib


RT_RAY = np.dtype([("start", "<f4", 4), ("dir", "<f4", 4)])
RT_INTERSECTION = np.dtype([("position", "<f4", 4), ("distance", "<f4"), ("triangle_index", "<i4"),
                            ("sphere_index", "<i4")])
assert RT_RAY.itemsize == 32 and RT_INTERSECTION.itemsize == 28


def as_rays(rays):
    """RT_RAY array from an RT_RAY array or (n, 8) float32 (start xyzw, dir xyzw)."""
    rays = np.ascontiguousarray(rays)
    if rays.dtype != RT_RAY:
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 8).view(RT_RAY).reshape(-1)
    return rays


def oracle_rt_closest(tris, spheres, rays):
    """RT_INTERSECTION per ray (position 0 and both indices -1 on a miss)."""
    rays = as_rays(rays)
    out = np.zeros(len(rays), RT_INTERSECTION)
    rc = rays_oracle().oracle_rt_closest(ptr(rays), c_i(len(rays)), ptr(tris), c_i(0 if tris is None else len(tris)),
                                    ptr(spheres), c_i(0 if spheres is None else len(spheres)), ptr(out))
    assert rc == 0
    return out


def oracle_rt_occluded(tris, spheres, rays, max_distance):
    """uint8 per ray: ClosestIntersection && distance < max_distance."""
    rays = as_rays(rays)
    md = np.ascontiguousarray(max_distance, np.float32).reshape(-1)
    out = np.zeros(len(rays), np.uint8)
    rc = rays_oracle().oracle_rt_occluded(ptr(rays), ptr(md), c_i(len(rays)), ptr(tris),
                                     c_i(0 if tris is None else len(tris)), ptr(spheres),
                                     c_i(0 if spheres is None else len(spheres)), ptr(out))
    assert rc == 0
    return out


def camera_rays(W, H, focal, cam, R, offsets=((0, 0),)):
    """The sample rays of Draw (raytracer skeleton.cpp:126-137) for every pixel, in pixel order and, per pixel, in
    the order of `offsets` (i, j): dir = R * vec4(u - W/2, v - H/2, f, 1) with glm's pairwise mat4*vec4 sums, then
    (dir.x + 0.5 i, dir.y + 0.5 j, f, 1).  All float32, one rounding per operation."""
    f = np.float32
    R = np.asarray(R, np.float32).reshape(-1)
    u = np.arange(W, dtype=np.int64)[None, :] - W // 2
    v = np.arange(H, dtype=np.int64)[:, None] - H // 2
    x = np.broadcast_to(u.astype(np.float32), (H, W))
    y = np.broadcast_to(v.astype(np.float32), (H, W))
    fl = f(focal)
    dirs = []
    for r in range(2):
        a = (R[0 + r] * x).astype(np.float32) + (R[4 + r] * y).astype(np.float32)
        b = f(R[8 + r] * fl) + f(R[12 + r] * f(1.0))
        dirs.append((a.astype(np.float32) + b).astype(np.float32))
    rays = np.zeros((H, W, len(offsets)), RT_RAY)
    for k, (i, j) in enumerate(offsets):
        rays["start"][:, :, k] = np.asarray(cam, np.float32)
        rays["dir"][:, :, k, 0] = (dirs[0] + f(f(0.5) * f(i))).astype(np.float32)
        rays["dir"][:, :, k, 1] = (dirs[1] + f(f(0.5) * f(j))).astype(np.float32)
        rays["dir"][:, :, k, 2] = fl
        rays["dir"][:, :, k, 3] = 1.0
    return rays.reshape(-1)


NINE_SAMPLES = tuple((i, j) for i in (-1, 0, 1) for j in (-1, 0, 1))


def shadow_rays(hits, tris, spheres, light_pos):
    """DirectLight's shadow rays (raytracer skeleton.cpp:366-397) for the hits among `hits` (RT_INTERSECTION):
    start = p + n * 1e-5 (n the triangle's normal or Sphere::getNormal), dir = light - p, and
    max_distance = r_mag = |light - p| summed and rooted in double.  Returns (rays, max_distance, which)."""
    f = np.float32
    which = np.nonzero(hits["distance"] < np.finfo(np.float32).max)[0]
    h = hits[which]
    p = h["position"].astype(np.float32)
    L = np.asarray(light_pos, np.float32)
    r = (L[None, :] - p).astype(np.float32)
    r_mag = np.sqrt((r[:, 0].astype(np.float64) * r[:, 0]) + (r[:, 1].astype(np.float64) * r[:, 1])
                    + (r[:, 2].astype(np.float64) * r[:, 2])).astype(np.float32)
    n = np.zeros((len(h), 4), np.float32)
    ti = h["triangle_index"]
    tri_hit = ti >= 0
    n[tri_hit] = tris["normal"][ti[tri_hit]]
    on_sph = np.nonzero(~tri_hit)[0]
    if len(on_sph):
        a = (p[on_sph, :3] - spheres["centre"][h["sphere_index"][on_sph]]).astype(np.float32)
        d = ((a[:, 0] * a[:, 0]).astype(f) + (a[:, 1] * a[:, 1]).astype(f)).astype(f)
        d = (d + (a[:, 2] * a[:, 2]).astype(f)).astype(f)
        inv = (f(1.0) / np.sqrt(d, dtype=np.float32)).astype(f)
        n[on_sph, :3] = (a * inv[:, None]).astype(f)
        n[on_sph, 3] = 0.0
    rays = np.zeros(len(h), RT_RAY)
    rays["start"] = (p + (n * f(0.00001)).astype(np.float32)).astype(np.float32)
    rays["dir"] = r
    return rays, r_mag, which
