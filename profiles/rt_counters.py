"""Diagnostic: per-level counts of the RT filter hierarchy (library built with
-DRT_PROFILE_COUNTERS).  Usage: python profiles/rt_counters.py [workload]"""
import ctypes
import importlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402
import helpers as h  # noqa: E402
import bench  # noqa: E402

b = importlib.import_module("computer-graphics_b200")
workload = sys.argv[1] if len(sys.argv) > 1 else "rt_cornell_4k"
kind, W, H, f = bench.WORKLOADS[workload]
r = b.Renderer(0)
tris, sph = b.scene_cornell_rt_tessellated(60) if workload == "rt_tess100k_4k" else b.scene_cornell_rt()
cam = b.make_camera(bench.RT_CAM, f, h.identity_R(), W, H)
r.rt_upload_scene(tris, sph)
rgb = torch.empty((H, W, 3), dtype=torch.float32, device="cuda")
depth = torch.zeros((H, W), dtype=torch.float32, device="cuda")
index = torch.zeros((H, W), dtype=torch.int32, device="cuda")
r.rt_render_device(cam, bench.RT_LIGHTS, 0, H, rgb.data_ptr(), depth.data_ptr(), index.data_ptr())
c = (ctypes.c_uint64 * 16)()
assert b.load_library().b200_debug_counters(r.ctx, c) == 0
names = ["shadow rays", "exact evals", "primary L1 tests", "primary L1 passes", "shadow L1 tests", "shadow L1 passes",
         "shadow L2 tests", "shadow L2 non-miss", "shadow exact, own triangle", "grid list entries",
         "grid: blocks streaming the scene", "grid: light cells walked", "records streamed (camera)",
         "records streamed (lights)", "shadow exact", "-"]
npx = W * H
for n, v in zip(names, c):
    print(f"{n:36s} {v:14d}  {v / npx:8.3f} per pixel  {v / (npx / 256):10.2f} per block")

# spatial distribution (diagnostic build: depth = shadow L1 tests, index = exact evaluations of the pixel)
import numpy as np  # noqa: E402
for name, plane in (("shadow L1 tests", depth.cpu().numpy()), ("exact evals", index.cpu().numpy().astype(np.float32))):
    print(name, "percentiles 50/90/99/99.9/max:", [float(np.percentile(plane, q)) for q in (50, 90, 99, 99.9, 100)])
    blocks = plane[: H // 16 * 16, : W // 16 * 16].reshape(H // 16, 16, W // 16, 16).sum(axis=(1, 3))
    print("  per 16x16 block: mean %.0f  p99 %.0f  max %.0f ; share of the total in the top 1%% of blocks: %.2f" % (
        blocks.mean(), np.percentile(blocks, 99), blocks.max(),
        np.sort(blocks.ravel())[-blocks.size // 100:].sum() / blocks.sum()))
    coarse = plane[: H // 120 * 120, : W // 240 * 240].reshape(H // 120, 120, W // 240, 240).mean(axis=(1, 3))
    for row in coarse:
        print("   ", " ".join(f"{v:6.1f}" for v in row))

# direction-grid list lengths
cells = np.zeros(1 << 22, np.uint32)
nc, ncam = ctypes.c_int(), ctypes.c_int()
if b.load_library().b200_debug_rt_cells(r.ctx, cells.ctypes.data_as(ctypes.c_void_p), len(cells), ctypes.byref(nc), ctypes.byref(ncam)) == 0 and nc.value:
    cam_c, light_c = cells[: ncam.value], cells[ncam.value: nc.value]
    for name, c in (("camera cells", cam_c), ("light cells", light_c)):
        print(name, len(c), "entries", int(c.sum()), "nonempty", int((c > 0).sum()), "percentiles 50/90/99/max of nonempty:",
              [float(np.percentile(c[c > 0], q)) for q in (50, 90, 99, 100)] if (c > 0).any() else None)
    faces = light_c[: 6 * 4096].reshape(6, 64, 64)
    for f in range(6):
        print("face", f, "entries", int(faces[f].sum()), "max", int(faces[f].max()), "at", np.unravel_index(faces[f].argmax(), (64, 64)))
