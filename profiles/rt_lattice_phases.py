"""Diagnostic (library built with EXTRA=-DRT_PROFILE_PHASES): cycles every warp of rt_lattice_kernel spends in
each phase -- primary triangles, spheres, shadow rays, shading, the wait at the block barrier before the pixel
sums, the sums -- and the kernel's resident blocks per SM.  python profiles/rt_lattice_phases.py [workload]"""
import ctypes, importlib, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch
import helpers as h, bench
b = importlib.import_module("computer-graphics_b200")
w = sys.argv[1] if len(sys.argv) > 1 else "rt_cornell_4k"
kind, W, H, f = bench.WORKLOADS[w]
r = b.Renderer(0)
tris, sph = bench.scenes_rt(w)
cam = b.make_camera(bench.RT_CAM, f, h.identity_R(), W, H)
r.rt_upload_scene(tris, sph)
depth = torch.zeros((H, W), device="cuda"); index = torch.zeros((H, W), dtype=torch.int32, device="cuda"); rgb = torch.zeros((H, W, 3), device="cuda")
for _ in range(3):
    r.rt_render_device(cam, bench.RT_LIGHTS, 0, H, rgb.data_ptr(), depth.data_ptr(), index.data_ptr()); r.synchronize()
st = r.stats()
blocks = ctypes.c_int(0)
assert r.lib.b200_debug_rt_lattice_blocks_per_sm(r.ctx, ctypes.byref(blocks)) == 0
print(f"{w}: {torch.cuda.get_device_name(0)}; gpu_ms {st['gpu_ms']:.3f} (instrumented); "
      f"rt_lattice_kernel resident blocks per SM (cudaOccupancyMaxActiveBlocksPerMultiprocessor): {blocks.value}")

# index plane, top pixel row of each 8 x 4 warp patch: lane k < 8 holds clock64 stamp k - stamp 0 (lane 0: the SM)
Hc, Wc = H // 16 * 16, W // 16 * 16          # whole blocks only: every warp of them wrote its stamps
top = index.cpu().numpy()[:Hc:4, :Wc].reshape(Hc // 4, Wc // 8, 8).astype(np.int64)
sm = top[..., 0]
s = top.copy(); s[..., 0] = 0
d = np.diff(s, axis=-1).reshape(-1, 7)       # per warp: the seven phases
names = ["primary triangles", "spheres", "shadow rays", "shade (lane 0)", "shade (rest of the warp)",
         "wait at the final barrier", "pixel sums + counts"]
tot = s[..., 7].reshape(-1)
print(f"warps {tot.size} on {len(np.unique(sm))} SMs; cycles per warp: mean {tot.mean():.0f} p50 {np.percentile(tot, 50):.0f} "
      f"p99 {np.percentile(tot, 99):.0f} max {tot.max():.0f}; sum {tot.sum() / 1e9:.3f} G warp-cycles")
print(f"{'phase':28s} {'total Gcyc':>10s} {'share':>6s} {'p50/warp':>9s} {'p99/warp':>9s}")
for k, n in enumerate(names):
    x = d[:, k]
    print(f"{n:28s} {x.sum() / 1e9:10.3f} {100 * x.sum() / tot.sum():5.1f}% {np.percentile(x, 50):9.0f} {np.percentile(x, 99):9.0f}")
# the barrier: a block's warps leave it together; what a warp waits is the block's last arrival minus its own
arr = s[..., 5].reshape(Hc // 16, 4, Wc // 16, 2)
late = arr.max(axis=(1, 3), keepdims=True) - arr
print(f"block barrier: last arrival - own arrival per warp: mean {late.mean():.0f} p50 {np.percentile(late, 50):.0f} "
      f"p99 {np.percentile(late, 99):.0f} cycles; share of warp-cycles {100 * d[:, 5].sum() / tot.sum():.1f}%")
