"""CPU tests of the oracle's DirectLight export (oracle_rt_direct_light): the nine-sample hits of oracle_rt_closest,
shaded per light and accumulated in Draw's order, equal the committed frames of the compiled reference, bit for
bit."""
import importlib
import os
import sys

import numpy as np
import pytest

import helpers as h
import direct_light_helpers as dh
import rays_helpers as rh
from conftest import load_golden


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def test_header_declares_direct_light():
    sys.path.insert(0, h.ROOT)
    b200 = importlib.import_module("computer-graphics_b200")
    header = open(os.path.join(h.ROOT, "include", "b200render.h")).read()
    for name in ("rt_direct_light", "rt_direct_light_device"):
        assert f"\nint {name}(" in header and name in b200.ABI_SYMBOLS


@pytest.mark.parametrize("name", ["cornell_default_160x128", "cornell_yaw_96x64", "random40_96x64"])
def test_composed_draw_matches_committed_reference_frames(name):
    g = load_golden(f"rt_ref_{name}.npz")
    tris = g["tris"].view(h.RT_TRI)
    sph = g["spheres"].view(h.RT_SPHERE)
    sph = sph if len(sph) else None
    W, H = int(g["W"]), int(g["H"])
    rays = rh.camera_rays(W, H, float(g["focal"]), g["cam"], g["R"], rh.NINE_SAMPLES)
    hits = rh.oracle_rt_closest(tris, sph, rays)
    power, n_shadow = dh.oracle_rt_direct_light(tris, sph, hits, g["lights"].reshape(-1, 7))
    n_hit = int((hits["distance"] < np.finfo(np.float32).max).sum())
    assert n_shadow == n_hit * len(g["lights"].reshape(-1, 7)) and n_hit > 0
    rgb = dh.draw_accumulate(hits, power, tris, sph).reshape(H, W, 3)
    assert np.array_equal(bits(rgb), bits(g["rgb"]))


def test_entries_naming_no_primitive_give_zero(cornell_rt):
    tris, sph = cornell_rt
    hits = np.zeros(6, rh.RT_INTERSECTION)
    hits["position"] = (0.1, 0.2, 0.3, 1.0)
    hits["distance"] = 1.0
    hits["triangle_index"] = [-1, len(tris), -2, -1, -1, 3]
    hits["sphere_index"] = [-1, 0, 0, len(sph), -7, -1]
    lights = h.lights_array(h.DEFAULT_RT_LIGHTS)
    power, n_shadow = dh.oracle_rt_direct_light(tris, sph, hits, lights)
    assert n_shadow == 1
    assert np.all(bits(power[:5]) == 0)
