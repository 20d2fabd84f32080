"""CPU tests of the ray-query ABI layouts and of the oracle's ray-query exports (oracle_rt_closest,
oracle_rt_occluded): pinned on the committed outputs of the compiled reference."""
import ctypes
import importlib
import os
import sys

import numpy as np
import pytest

import helpers as h
import rays_helpers as rh
from conftest import load_golden

FLT_MAX = np.finfo(np.float32).max


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def index_encoding(out):
    """RT_INTERSECTION -> the `index` planes of the goldens: triangle, -1 - sphere, INT32_MIN on a miss."""
    hit = out["distance"] < FLT_MAX
    idx = np.where(out["triangle_index"] != -1, out["triangle_index"], -1 - out["sphere_index"])
    return np.where(hit, idx, h.INDEX_MISS).astype(np.int32)


def test_layouts_match_header():
    sys.path.insert(0, h.ROOT)
    b200 = importlib.import_module("computer-graphics_b200")
    assert ctypes.sizeof(b200.RtRay) == 32 and rh.RT_RAY.itemsize == 32 and b200.RT_RAY.itemsize == 32
    assert ctypes.sizeof(b200.RtIntersection) == 28 and rh.RT_INTERSECTION.itemsize == 28
    assert b200.RT_INTERSECTION.itemsize == 28
    offs = [getattr(b200.RtIntersection, f).offset for f in ("position", "distance", "triangle_index", "sphere_index")]
    assert offs == [0, 16, 20, 24]
    assert [rh.RT_INTERSECTION.fields[f][1] for f in ("position", "distance", "triangle_index", "sphere_index")] == offs
    header = open(os.path.join(h.ROOT, "include", "b200render.h")).read()
    for name in ("rt_closest_hits", "rt_occluded", "rt_closest_hits_device", "rt_occluded_device"):
        assert f"\nint {name}(" in header and name in b200.ABI_SYMBOLS


@pytest.mark.parametrize("name", ["cornell_default_160x128", "cornell_yaw_96x64", "random40_96x64"])
def test_closest_matches_committed_reference_outputs(name):
    """The centre-sample rays of ref_rt_trace (oracle/refbuild/ref_rt_harness.cpp), through oracle_rt_closest ==
    the compiled reference's distance and index planes, bit for bit."""
    g = load_golden(f"rt_ref_{name}.npz")
    tris = g["tris"].view(h.RT_TRI)
    sph = g["spheres"].view(h.RT_SPHERE)
    W, H = int(g["W"]), int(g["H"])
    rays = rh.camera_rays(W, H, float(g["focal"]), g["cam"], g["R"])
    out = rh.oracle_rt_closest(tris, sph if len(sph) else None, rays)
    hit = out["distance"] < FLT_MAX
    dist = np.where(hit, out["distance"], np.float32(np.inf)).astype(np.float32).reshape(H, W)
    assert np.array_equal(bits(dist), bits(g["dist"]))
    assert np.array_equal(index_encoding(out).reshape(H, W), g["index"])
    # misses: position 0, both indices -1; hits: exactly one index set
    assert np.all(out["position"][~hit] == 0) and np.all(out["triangle_index"][~hit] == -1)
    assert np.all(out["sphere_index"][~hit] == -1)
    assert np.all((out["triangle_index"][hit] == -1) != (out["sphere_index"][hit] == -1))


def test_closest_position_is_start_plus_t_dir(cornell_rt):
    """position.w = start.w + 0 (-0 becomes +0) and position.xyz on the ray."""
    tris, sph = cornell_rt
    rays = rh.camera_rays(32, 24, 24.0, h.f32(0, 0, -3, -0.0), h.identity_R())
    out = rh.oracle_rt_closest(tris, sph, rays)
    hit = out["distance"] < FLT_MAX
    assert hit.sum() > len(rays) // 2
    assert np.all(bits(out["position"][hit, 3]) == 0)


def test_occluded_is_closest_then_limit(cornell_rt):
    rng = np.random.default_rng(5)
    tris, sph = cornell_rt
    n = 4000
    rays = np.zeros(n, rh.RT_RAY)
    rays["start"][:, :3] = rng.uniform(-1.2, 1.2, (n, 3)).astype(np.float32)
    rays["start"][:, 3] = 1.0
    rays["dir"][:, :3] = rng.normal(size=(n, 3)).astype(np.float32)
    closest = rh.oracle_rt_closest(tris, sph, rays)
    d = closest["distance"]
    with np.errstate(over="ignore"):
        up = np.nextafter(d, np.float32(np.inf))
    limits = [rng.uniform(0, 3, n).astype(np.float32), np.zeros(n, np.float32), -np.ones(n, np.float32),
              np.full(n, np.nan, np.float32), np.full(n, np.inf, np.float32), d, up]
    for md in limits:
        md = np.ascontiguousarray(md, np.float32)
        want = ((d < FLT_MAX) & (d < md)).astype(np.uint8)
        got = rh.oracle_rt_occluded(tris, sph, rays, md)
        assert np.array_equal(got, want)
    hit = d < FLT_MAX
    assert hit.any() and (~hit).any()
    assert not rh.oracle_rt_occluded(tris, sph, rays, d)[hit].any()        # exactly the hit's distance: 0
    assert rh.oracle_rt_occluded(tris, sph, rays, up)[hit].all()           # the next float above it: 1
