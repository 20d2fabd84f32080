"""Frames with the caller's own sample offsets per pixel (rt_render_samples_device) against the nine-sample frame
entry and against the composed ray queries.

Workloads (device-resident outputs, Cornell box unless named, camera (0, 0, -3), f = H, one light):
  (a) cornell_4k_nine      3840x2160 with the reference's nine offsets: rt_render_samples_device against
                           rt_render_device (which takes the lattice kernel): the cost of generality.  Frames compared.
  (b) cornell_4k_S<n>      3840x2160 with S = 1 (centre), 4 (rotated grid), 16 (4x4 stratified), 64 (8x8 stratified);
                           rows [1072, 1088) compared with the plain-C oracle (oracle_rt_samples).
  (c) frame_720p_S<n>      1280x720 with the nine offsets and with S = 16: the fused call against
                           rt_closest_hits_device + rt_direct_light_device on the same rays, accumulated in Draw's order
                           on the host (not timed).  Frames compared.
  (d) tess100k_4k_S<n>     the 100 800-triangle box at 3840x2160 (gridded path) with S = 4 and with the nine offsets,
                           against rt_render_device.  Nine offsets: frames compared; S = 4: rows [1072, 1076) compared
                           with the composed ray queries.
Every step overwrites the L2 (256 MiB write) first; the arms alternate step by step in one process.  Time per call is
the library's own CUDA-event time (b200_get_stats gpu_ms), medians over the steps.  Prints the device and its power
limit, then one JSON line per workload.

    python profiles/rt_samples.py [--steps N]
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np
import torch

import helpers as h
import rays_helpers as rh
import samples_helpers as sh

b200 = importlib.import_module("computer-graphics_b200")


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        return None


def u32(t):
    return t.cpu().numpy().view(np.uint32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=7)
    args = ap.parse_args()
    print(json.dumps({"gpu": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w()}), flush=True)
    r = b200.Renderer(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    cam = h.f32(0, 0, -3, 1)
    L = h.DEFAULT_RT_LIGHTS
    L7 = h.lights_array(L)

    def timed(fn, step):
        flush.fill_(step & 255)
        torch.cuda.synchronize()
        fn()
        return r.stats()

    def alternate(arms, steps):
        """arms: {name: fn}; returns {name: (median ms, [min, max], last stats)}."""
        times, last = {k: [] for k in arms}, {}
        for step in range(steps + 1):   # step 0: warm-up
            for k, fn in arms.items():
                st = timed(fn, step)
                if step:
                    times[k].append(st["gpu_ms"])
                last[k] = st
        return {k: (round(float(np.median(v)), 3), [round(min(v), 3), round(max(v), 3)], last[k]) for k, v in times.items()}

    def frame_bufs(W, H):
        return torch.empty(W * H * 3, dtype=torch.float32, device="cuda"), torch.empty(W * H, dtype=torch.float32,
                                                                                    device="cuda")

    tris, sph = b200.scene_cornell_rt()
    W, H = 3840, 2160
    c4k = b200.make_camera(cam, float(H), h.identity_R(), W, H)
    r.rt_upload_scene(tris, sph)

    # (a) the reference's nine offsets against the lattice path
    s_rgb, s_dep = frame_bufs(W, H)
    f_rgb, f_dep = frame_bufs(W, H)
    res = alternate({"samples": lambda: r.rt_render_samples_device(c4k, L, sh.NINE, 4, 0, H, s_rgb.data_ptr(),
                                                                   s_dep.data_ptr()),
                     "frame": lambda: r.rt_render_device(c4k, L, 0, H, f_rgb.data_ptr(), f_dep.data_ptr())}, args.steps)
    print(json.dumps({"workload": "a_cornell_4k_nine", "samples_ms": res["samples"][0], "samples_range": res["samples"][1],
                      "frame_lattice_ms": res["frame"][0], "frame_range": res["frame"][1],
                      "ratio": round(res["samples"][0] / res["frame"][0], 2),
                      "identical": bool(np.array_equal(u32(s_rgb), u32(f_rgb)) and np.array_equal(u32(s_dep), u32(f_dep)))}),
          flush=True)

    # (b) other patterns at 4K
    for name in ("centre", "rgss", "strat4", "strat8"):
        off = sh.pattern(name)
        res = alternate({"samples": lambda: r.rt_render_samples_device(c4k, L, off, 0, 0, H, s_rgb.data_ptr(),
                                                                       s_dep.data_ptr())}, args.steps)
        o = sh.oracle_rt_samples(W, H, float(H), cam, h.identity_R(), L7, tris, sph, off, 0, 1072, 1088)
        got = s_rgb.cpu().numpy().reshape(H, W, 3)[1072:1088]
        st = res["samples"][2]
        print(json.dumps({"workload": f"b_cornell_4k_S{len(off)}", "pattern": name, "ms": res["samples"][0],
                          "range": res["samples"][1], "ms_per_sample": round(res["samples"][0] / len(off), 4),
                          "primary_rays": st["primary_rays"], "shadow_rays": st["shadow_rays"],
                          "rows_1072_1088_equal_oracle": bool(np.array_equal(got.view(np.uint32),
                                                                             o["rgb"][1072:1088].view(np.uint32)))}),
              flush=True)
    del s_rgb, s_dep, f_rgb, f_dep

    # (c) 1280x720: fused against the composed ray queries on the same rays
    W7, H7 = 1280, 720
    c7 = b200.make_camera(cam, float(H7), h.identity_R(), W7, H7)
    for name in ("nine", "strat4"):
        off = sh.NINE if name == "nine" else sh.pattern(name)
        S = len(off)
        rays = sh.sample_rays(W7, H7, float(H7), cam, h.identity_R(), off)
        n = len(rays)
        d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1).copy()).cuda()
        d_hits = torch.empty(n * 28, dtype=torch.uint8, device="cuda")
        d_pow = torch.empty(n * 3, dtype=torch.float32, device="cuda")
        d_rgb, _ = frame_bufs(W7, H7)
        comp, fused = [], []
        for step in range(args.steps + 1):
            ms = timed(lambda: r.rt_closest_hits_device(d_rays.data_ptr(), n, d_hits.data_ptr()), step)["gpu_ms"]
            ms += timed(lambda: r.rt_direct_light_device(d_hits.data_ptr(), n, L, d_pow.data_ptr()), step)["gpu_ms"]
            fm = timed(lambda: r.rt_render_samples_device(c7, L, off, 0, 0, H7, d_rgb.data_ptr()), step)["gpu_ms"]
            if step:
                comp.append(ms)
                fused.append(fm)
        hits = d_hits.cpu().numpy().view(rh.RT_INTERSECTION)
        rgb = sh.accumulate(hits, d_pow.cpu().numpy().reshape(n, 1, 3), tris, sph, S)
        mc, mf = float(np.median(comp)), float(np.median(fused))
        print(json.dumps({"workload": f"c_frame_720p_S{S}", "samples": n, "composed_ms": round(mc, 3),
                          "fused_ms": round(mf, 3), "composed_over_fused": round(mc / mf, 2),
                          "fused_range": [round(min(fused), 3), round(max(fused), 3)],
                          "identical": bool(np.array_equal(rgb.reshape(-1).view(np.uint32), u32(d_rgb)))}), flush=True)
        del d_rays, d_hits, d_pow, d_rgb

    # (d) the 100 800-triangle box at 4K: the gridded path
    ttris, tsph = b200.scene_cornell_rt_tessellated(60)
    r.rt_upload_scene(ttris, tsph)
    s_rgb, s_dep = frame_bufs(W, H)
    f_rgb, f_dep = frame_bufs(W, H)
    for name in ("rgss", "nine"):
        off = sh.NINE if name == "nine" else sh.pattern(name)
        ds = 4 if name == "nine" else 0
        res = alternate({"samples": lambda: r.rt_render_samples_device(c4k, L, off, ds, 0, H, s_rgb.data_ptr(),
                                                                       s_dep.data_ptr()),
                         "frame": lambda: r.rt_render_device(c4k, L, 0, H, f_rgb.data_ptr(), f_dep.data_ptr())},
                        max(3, args.steps // 2))
        out = {"workload": f"d_tess100k_4k_S{len(off)}", "samples_ms": res["samples"][0],
               "samples_range": res["samples"][1], "frame_ms": res["frame"][0], "frame_range": res["frame"][1],
               "ratio": round(res["samples"][0] / res["frame"][0], 2)}
        if name == "nine":
            out["identical_to_frame"] = bool(np.array_equal(u32(s_rgb), u32(f_rgb)) and np.array_equal(u32(s_dep), u32(f_dep)))
        else:
            y0, y1 = 1072, 1076
            rays = sh.sample_rays(W, H, float(H), cam, h.identity_R(), off).reshape(H, W, len(off))[y0:y1].reshape(-1)
            hits = r.rt_closest_hits(ttris, tsph, rays)
            pw = r.rt_direct_light(ttris, tsph, hits, L)
            rgb = sh.accumulate(r._hits(hits), pw, ttris, tsph, len(off))
            got = s_rgb.cpu().numpy().reshape(H, W, 3)[y0:y1].reshape(-1, 3)
            out["rows_1072_1076_equal_composed"] = bool(np.array_equal(got.view(np.uint32), rgb.view(np.uint32)))
        print(json.dumps(out), flush=True)
    r.close()


if __name__ == "__main__":
    main()
