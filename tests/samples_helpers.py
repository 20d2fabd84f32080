"""Test plumbing of render_raytrace_samples: the plain-C oracle's Draw with the caller's own sample offsets
(oracle/rays/oracle_rt_samples.c, which includes oracle_rt_rays.c and oracle_rt.c and calls closest_intersection
and direct_light unchanged), the sample rays of such a pattern, and a set of patterns.

Nothing here is product code.
"""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from helpers import ORACLE_DIR, c_i, ptr
from rays_helpers import CFLAGS, RT_RAY

SRC = os.path.join(ORACLE_DIR, "rays", "oracle_rt_samples.c")
_lib = None

# The reference's pattern (skeleton.cpp:134-137): 0.5 * (i, j), i = -1..1 outer, j = -1..1 inner; its centre is 4
NINE = np.array([(0.5 * i, 0.5 * j) for i in (-1, 0, 1) for j in (-1, 0, 1)], np.float32)


def samples_oracle():
    """liboracle_samples.so, compiled on first use into the temporary directory (the tree may be read-only), named
    by a hash of the sources and flags."""
    global _lib
    if _lib is None:
        key = hashlib.sha256()
        for p in (SRC, os.path.join(ORACLE_DIR, "rays", "oracle_rt_rays.c"), os.path.join(ORACLE_DIR, "oracle_rt.c")):
            key.update(open(p, "rb").read())
        key.update(" ".join(CFLAGS).encode())
        path = os.path.join(tempfile.gettempdir(), f"liboracle_samples_{key.hexdigest()[:16]}_{os.getuid()}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.check_call([os.environ.get("CC", "gcc"), *CFLAGS, "-o", tmp, SRC, "-lm"])
            os.replace(tmp, path)
        _lib = ctypes.CDLL(path)
    return _lib


def oracle_rt_samples(W, H, focal, cam, R, lights7, tris, spheres, offsets, depth_sample, row0=0, row1=None):
    """Draw with sample k of every pixel along (dir.x + offsets[k, 0], dir.y + offsets[k, 1], f): dict of rgb, dist,
    index, argb (full frames; rows outside [row0, row1) zero) and the primary / shadow rays traced."""
    row1 = H if row1 is None else row1
    off = np.ascontiguousarray(offsets, np.float32).reshape(-1, 2)
    L = np.ascontiguousarray(lights7, np.float32).reshape(-1)
    rgb = np.zeros((H, W, 3), np.float32)
    dist = np.zeros((H, W), np.float32)
    index = np.zeros((H, W), np.int32)
    argb = np.zeros((H, W), np.uint32)
    counts = np.zeros(2, np.uint64)
    rc = samples_oracle().oracle_rt_samples(
        c_i(W), c_i(H), ctypes.c_float(focal), ptr(np.ascontiguousarray(cam, np.float32)),
        ptr(np.ascontiguousarray(R, np.float32)), ptr(L), c_i(len(L) // 7), ptr(tris),
        c_i(0 if tris is None else len(tris)), ptr(spheres), c_i(0 if spheres is None else len(spheres)), ptr(off),
        c_i(len(off)), c_i(depth_sample), c_i(row0), c_i(row1), ptr(rgb), ptr(dist), ptr(index), ptr(argb),
        ptr(counts))
    assert rc == 0
    return dict(rgb=rgb, dist=dist, index=index, argb=argb, primary=int(counts[0]), shadow=int(counts[1]))


def sample_rays(W, H, focal, cam, R, offsets):
    """The sample rays of the pattern for every pixel, in pixel order and, per pixel, in the pattern's order:
    dir = R * vec4(u - W/2, v - H/2, f, 1) with glm's pairwise sums, then (dir.x + o.x, dir.y + o.y, f, 1), float32
    with one rounding per operation."""
    f = np.float32
    R = np.asarray(R, np.float32).reshape(-1)
    x = np.broadcast_to((np.arange(W, dtype=np.int64)[None, :] - W // 2).astype(np.float32), (H, W))
    y = np.broadcast_to((np.arange(H, dtype=np.int64)[:, None] - H // 2).astype(np.float32), (H, W))
    fl = f(focal)
    dirs = []
    for r in range(2):
        a = (R[0 + r] * x).astype(np.float32) + (R[4 + r] * y).astype(np.float32)
        b = f(R[8 + r] * fl) + f(R[12 + r] * f(1.0))
        dirs.append((a.astype(np.float32) + b).astype(np.float32))
    off = np.asarray(offsets, np.float32).reshape(-1, 2)
    rays = np.zeros((H, W, len(off)), RT_RAY)
    for k, (ox, oy) in enumerate(off):
        rays["start"][:, :, k] = np.asarray(cam, np.float32)
        rays["dir"][:, :, k, 0] = (dirs[0] + ox).astype(np.float32)
        rays["dir"][:, :, k, 1] = (dirs[1] + oy).astype(np.float32)
        rays["dir"][:, :, k, 2] = fl
        rays["dir"][:, :, k, 3] = 1.0
    return rays.reshape(-1)


def accumulate(hits, power, tris, spheres, n_samples):
    """Draw's pixel loop over n_samples consecutive hits per pixel (as direct_light_helpers.draw_accumulate), the
    pixel divided by (float)n_samples.  Returns (pixels, 3) float32."""
    f = np.float32
    hit = (hits["distance"] < np.finfo(np.float32).max).reshape(-1, n_samples)
    power = np.asarray(power, np.float32).reshape(hit.shape[0], n_samples, -1, 3)
    ti = hits["triangle_index"].reshape(-1, n_samples)
    si = hits["sphere_index"].reshape(-1, n_samples)
    pix = np.zeros((hit.shape[0], 3), np.float32)
    for k in range(n_samples):
        h = hit[:, k]
        add = pix.copy()
        for l in range(power.shape[2]):
            add = (add + power[:, k, l]).astype(f)
        col = np.zeros((len(pix), 3), np.float32)
        on_tri = h & (ti[:, k] != -1)
        on_sph = h & (ti[:, k] == -1)
        col[on_tri] = tris["color"][ti[on_tri, k]]
        if on_sph.any():
            col[on_sph] = spheres["color"][si[on_sph, k]]
        add = (add + (col * f(0.5)).astype(f)).astype(f)
        pix = np.where(h[:, None], add, pix)
    valid = hit.any(axis=1)
    return np.where(valid[:, None], (pix / f(n_samples)).astype(f), f(0.0)).astype(np.float32)


def pattern(name, seed=0):
    """(S, 2) float32 offsets: 'centre' (1), 'rgss' (4, a rotated grid), 'strat4' (16, 4x4 stratified), 'strat8'
    (64, 8x8), 'nine_reordered' (the reference's nine in another order), or 'random<S>' (uniform in [-0.5, 0.5] with
    +-0.5, +-0 and subnormal offsets mixed in)."""
    if name == "centre":
        return np.zeros((1, 2), np.float32)
    if name == "rgss":
        return np.array([(-0.125, -0.375), (0.375, -0.125), (0.125, 0.375), (-0.375, 0.125)], np.float32)
    if name.startswith("strat"):
        n = int(name[5:])
        g = (np.arange(n, dtype=np.float32) - np.float32((n - 1) / 2)) / np.float32(n)
        return np.array([(a, b) for a in g for b in g], np.float32)
    if name == "nine_reordered":
        return NINE[np.random.default_rng(seed).permutation(9)].copy()
    assert name.startswith("random")
    n = int(name[6:])
    rng = np.random.default_rng(seed)
    o = rng.uniform(-0.5, 0.5, (n, 2)).astype(np.float32)
    special = np.array([0.5, -0.5, 0.0, -0.0, 1e-40, -1e-40, np.float32(2.0 ** -149), 0.49999997], np.float32)
    k = min(n * 2, len(special))
    flat = o.reshape(-1)
    flat[rng.permutation(2 * n)[:k]] = special[:k]
    return o
