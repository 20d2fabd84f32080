"""CPU tests of the oracle's Draw with the caller's own sample offsets (oracle_rt_samples): with the reference's nine
offsets it is oracle_rt_render and the committed frames of the compiled reference, bit for bit; with other patterns
it is the composition oracle_rt_closest -> oracle_rt_direct_light -> Draw's accumulation / S."""
import ctypes
import importlib
import os
import sys

import numpy as np
import pytest

import helpers as h
import direct_light_helpers as dh
import rays_helpers as rh
import samples_helpers as sh
from conftest import load_golden


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def golden_scene(name):
    g = load_golden(f"rt_ref_{name}.npz")
    tris = g["tris"].view(h.RT_TRI)
    sph = g["spheres"].view(h.RT_SPHERE)
    return g, tris, (sph if len(sph) else None)


def test_header_declares_samples_entries():
    sys.path.insert(0, h.ROOT)
    b200 = importlib.import_module("computer-graphics_b200")
    header = open(os.path.join(h.ROOT, "include", "b200render.h")).read()
    assert "#define B200_RT_MAX_SAMPLES 64" in header
    for name in ("render_raytrace_samples", "draw_raytrace_samples", "rt_render_samples_device"):
        assert f"\nint {name}(" in header and name in b200.ABI_SYMBOLS


@pytest.mark.parametrize("name", ["cornell_default_160x128", "cornell_yaw_96x64", "random40_96x64"])
def test_nine_offsets_equal_render_and_committed_reference_frames(name):
    g, tris, sph = golden_scene(name)
    W, H, f = int(g["W"]), int(g["H"]), float(g["focal"])
    L = g["lights"].reshape(-1)
    got = sh.oracle_rt_samples(W, H, f, g["cam"], g["R"], L, tris, sph, sh.NINE, 4)
    want = h.oracle_rt_render(W, H, f, g["cam"], g["R"], L, tris, sph)
    for k in ("rgb", "dist"):
        assert np.array_equal(bits(got[k]), bits(want[k])), k
    assert np.array_equal(got["index"], want["index"]) and np.array_equal(got["argb"], want["argb"])
    assert got["primary"] == want["primary"] == W * H * 9 and got["shadow"] == want["shadow"]
    assert np.array_equal(bits(got["rgb"]), bits(g["rgb"])) and np.array_equal(got["argb"], g["argb"])
    assert np.array_equal(bits(got["dist"]), bits(g["dist"])) and np.array_equal(got["index"], g["index"])


@pytest.mark.parametrize("pat", ["centre", "rgss", "random4", "strat4", "random16", "random64"])
@pytest.mark.parametrize("name", ["cornell_yaw_96x64", "random40_96x64"])
def test_patterns_equal_composed_closest_direct_light_accumulation(name, pat):
    g, tris, sph = golden_scene(name)
    W, H, f = int(g["W"]), int(g["H"]), float(g["focal"])
    if pat == "random64":   # (a band keeps the composed chain small)
        H0, H1 = 24, 40
    else:
        H0, H1 = 0, H
    off = sh.pattern(pat, seed=len(pat))
    S = len(off)
    L7 = g["lights"].reshape(-1, 7)
    ds = S // 2
    got = sh.oracle_rt_samples(W, H, f, g["cam"], g["R"], L7, tris, sph, off, ds, H0, H1)
    rays = sh.sample_rays(W, H, f, g["cam"], g["R"], off).reshape(H, W, S)[H0:H1].reshape(-1)
    hits = rh.oracle_rt_closest(tris, sph, rays)
    power, n_shadow = dh.oracle_rt_direct_light(tris, sph, hits, L7)
    rgb = sh.accumulate(hits, power, tris, sph, S).reshape(H1 - H0, W, 3)
    assert np.array_equal(bits(got["rgb"][H0:H1]), bits(rgb))
    d = hits.reshape(H1 - H0, W, S)[:, :, ds]
    hit = d["distance"] < np.finfo(np.float32).max
    assert np.array_equal(bits(got["dist"][H0:H1]), bits(np.where(hit, d["distance"], np.float32(np.inf))))
    idx = np.where(d["triangle_index"] != -1, d["triangle_index"], -1 - d["sphere_index"])
    assert np.array_equal(got["index"][H0:H1], np.where(hit, idx, h.INDEX_MISS))
    assert got["primary"] == W * (H1 - H0) * S and got["shadow"] == n_shadow
    q = np.zeros((H1 - H0, W), np.uint32)
    band = np.ascontiguousarray(rgb)
    h.oracle().oracle_quantise(h.ptr(band), ctypes.c_size_t(q.size), h.ptr(q))
    assert np.array_equal(got["argb"][H0:H1], q)


def test_special_offsets_are_in_the_random_patterns():
    o = sh.pattern("random16", seed=3).reshape(-1)
    assert np.any(o == 0.5) and np.any(o == -0.5) and np.any(np.signbit(o) & (o == 0))
    assert np.any((o != 0) & (np.abs(o) < np.finfo(np.float32).tiny))
    assert np.all(np.abs(o) <= 0.5)
