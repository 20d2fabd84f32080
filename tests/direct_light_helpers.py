"""Test plumbing of rt_direct_light: the plain-C oracle's DirectLight entry (oracle/rays/oracle_rt_direct_light.c,
which includes oracle_rt_rays.c and oracle_rt.c and calls direct_light unchanged), and Draw's pixel accumulation
over samples the caller traced.

Nothing here is product code.
"""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from helpers import ORACLE_DIR, c_i, ptr
from rays_helpers import CFLAGS, RT_INTERSECTION

SRC = os.path.join(ORACLE_DIR, "rays", "oracle_rt_direct_light.c")
_lib = None


def direct_light_oracle():
    """liboracle_direct_light.so, compiled on first use into the temporary directory (the tree may be read-only),
    named by a hash of the sources and flags."""
    global _lib
    if _lib is None:
        key = hashlib.sha256()
        for p in (SRC, os.path.join(ORACLE_DIR, "rays", "oracle_rt_rays.c"), os.path.join(ORACLE_DIR, "oracle_rt.c")):
            key.update(open(p, "rb").read())
        key.update(" ".join(CFLAGS).encode())
        path = os.path.join(tempfile.gettempdir(), f"liboracle_direct_light_{key.hexdigest()[:16]}_{os.getuid()}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.check_call([os.environ.get("CC", "gcc"), *CFLAGS, "-o", tmp, SRC, "-lm"])
            os.replace(tmp, path)
        _lib = ctypes.CDLL(path)
    return _lib


def oracle_rt_direct_light(tris, spheres, hits, lights7):
    """DirectLight per (entry, light): (n_hits, n_lights, 3) float32, and the shadow rays traced.  lights7: (n, 7)
    float32 (pos xyzw, colour rgb).  An entry naming no primitive gives 0."""
    hits = np.ascontiguousarray(hits, RT_INTERSECTION)
    L = np.ascontiguousarray(lights7, np.float32).reshape(-1, 7)
    out = np.zeros((len(hits), len(L), 3), np.float32)
    n_shadow = ctypes.c_uint64(0)
    rc = direct_light_oracle().oracle_rt_direct_light(
        ptr(hits), c_i(len(hits)), ptr(tris), c_i(0 if tris is None else len(tris)), ptr(spheres),
        c_i(0 if spheres is None else len(spheres)), ptr(L), c_i(len(L)), ptr(out), ctypes.byref(n_shadow))
    assert rc == 0
    return out, int(n_shadow.value)


def draw_accumulate(hits, power, tris, spheres, n_samples=9):
    """Draw's pixel loop (raytracer skeleton.cpp:138-166) over samples the caller traced: hits (RT_INTERSECTION) and
    power (n, n_lights, 3) hold n_samples consecutive entries per pixel.  Per hit sample: pix += power[l] for each
    light in order, then pix += colour * 0.5f; at the end pix / 9.0f if any sample hit, else 0.  float32, one rounding
    per operation.  Returns (pixels, 3)."""
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
    return np.where(valid[:, None], (pix / f(9.0)).astype(f), f(0.0)).astype(np.float32)
