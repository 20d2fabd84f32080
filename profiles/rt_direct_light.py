"""DirectLight for caller-supplied hits (rt_direct_light_device): the filtered kernel against
B200_OPT_RT_BRUTEFORCE = 1 and against the occlusion query alone.

Workloads (device-resident hits and results):
  (a) cornell_4k      the 8.29 M centre-sample hits of the Cornell box at 3840x2160, f = 2160, 1 light; a third arm
                      runs rt_occluded_device on the same hits' shadow rays (rays_helpers.shadow_rays): the
                      occlusion half alone;
  (b) cornell_4k_8l   the same hits, 8 lights;
  (c) tess100k_1m     the 1 M centre-sample hits (1024 x 1024, f = 1024) of the 100 800-triangle tessellated box;
  (d) frame_720p      the nine-sample frame at 1280x720 composed from rt_closest_hits_device + rt_direct_light_device
                      and accumulated in Draw's order, against rt_render_device of the same frame (pixels compared).
Every step overwrites the L2 (256 MiB write) first; the arms alternate step by step in one process.  Time per call is
the library's own CUDA-event time (b200_get_stats gpu_ms).  Prints the device and its power limit, then one JSON line
per workload.

    python profiles/rt_direct_light.py [--steps N]
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
import direct_light_helpers as dh
import rays_helpers as rh

b200 = importlib.import_module("computer-graphics_b200")
EIGHT_LIGHTS = [((0.0, -0.5, -0.7, 1.0), (14, 14, 14)), ((0.3, 0.7, -0.4, 1.0), (3, 4, 5)),
                ((0.0, 0.0, 1.5, 1.0), (20, 20, 20)), ((-0.3, 0.4, 0.2, 1.0), (2, 2, 2)),
                ((0.5, -0.9, 0.5, 1.0), (7, 1, 3)), ((-0.8, 0.8, -0.9, 1.0), (1, 9, 1)),
                ((0.0, 0.0, -2.0, 1.0), (30, 30, 30)), ((0.9, 0.0, 0.0, 0.0), (5, 5, 0.5))]


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    args = ap.parse_args()
    print(json.dumps({"gpu": torch.cuda.get_device_name(0), "power_limit_w": power_limit_w()}), flush=True)
    r = b200.Renderer(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    cam = h.f32(0, 0, -3, 1)

    def device_hits(scene, rays):
        r.rt_upload_scene(*scene)
        d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1).copy()).cuda()
        d_hits = torch.empty(len(rays) * 28, dtype=torch.uint8, device="cuda")
        r.rt_closest_hits_device(d_rays.data_ptr(), len(rays), d_hits.data_ptr())
        r.synchronize()
        return d_rays, d_hits

    def timed(fn, step):
        flush.fill_(step & 255)
        torch.cuda.synchronize()
        fn()
        return r.stats()

    def run(scene, d_hits, n, lights, steps, occ_arm=None):
        """Arms: filtered (0), brute force (1) and, with occ_arm = (d_srays, d_md, n_s), rt_occluded_device (2)."""
        r.rt_upload_scene(*scene)
        arms = [0, 1] + ([2] if occ_arm else [])
        times, outs, st_of = {a: [] for a in arms}, {}, {}
        for step in range(steps + 1):   # step 0: warm-up
            for arm in arms:
                r.set_option(b200.OPT_RT_BRUTEFORCE, 1 if arm == 1 else 0)
                if arm == 2:
                    d_s, d_md, n_s = occ_arm
                    d_out = torch.empty(n_s, dtype=torch.uint8, device="cuda")
                    st = timed(lambda: r.rt_occluded_device(d_s.data_ptr(), d_md.data_ptr(), n_s, d_out.data_ptr()), step)
                else:
                    d_out = torch.empty(n * len(lights) * 3, dtype=torch.float32, device="cuda")
                    st = timed(lambda: r.rt_direct_light_device(d_hits.data_ptr(), n, lights, d_out.data_ptr()), step)
                if step:
                    times[arm].append(st["gpu_ms"])
                st_of[arm] = st
                outs[arm] = d_out.cpu().numpy()
        r.set_option(b200.OPT_RT_BRUTEFORCE, 0)
        ms = {a: float(np.median(v)) for a, v in times.items()}
        res = {"hits": n, "lights": len(lights), "filtered_ms": round(ms[0], 3), "brute_ms": round(ms[1], 3),
               "speedup": round(ms[1] / ms[0], 2), "filtered_ms_range": [round(min(times[0]), 3), round(max(times[0]), 3)],
               "shadow_rays": st_of[0]["shadow_rays"],
               "exact_evals_per_shadow_ray": round(st_of[0]["exact_evals"] / max(1, st_of[0]["shadow_rays"]), 3),
               "identical": bool(np.array_equal(outs[0].view(np.uint32), outs[1].view(np.uint32)))}
        if occ_arm:
            res["occluded_ms"] = round(ms[2], 3)
            res["occluded_ms_range"] = [round(min(times[2]), 3), round(max(times[2]), 3)]
            res["occluded_exact_evals_per_ray"] = round(st_of[2]["exact_evals"] / max(1, occ_arm[2]), 3)
        return res, outs

    # (a), (b): Cornell 4K centre samples
    tris, sph = b200.scene_cornell_rt()
    rays = rh.camera_rays(3840, 2160, 2160.0, cam, h.identity_R())
    _, d_hits = device_hits((tris, sph), rays)
    hits = d_hits.cpu().numpy().view(rh.RT_INTERSECTION)
    srays, r_mag, which = rh.shadow_rays(hits, tris, sph, h.DEFAULT_RT_LIGHTS[0][0])
    d_s = torch.from_numpy(srays.view(np.uint8).reshape(-1).copy()).cuda()
    d_md = torch.from_numpy(np.ascontiguousarray(r_mag)).cuda()
    res, outs = run((tris, sph), d_hits, len(rays), h.DEFAULT_RT_LIGHTS, args.steps, (d_s, d_md, len(srays)))
    occ = outs[2].astype(bool)
    pw = outs[0].reshape(len(rays), 3)[which]
    res["occluded_implies_zero"] = bool(np.all(pw[occ] == 0))
    print(json.dumps({"workload": "a_cornell_4k", **res}), flush=True)
    res, _ = run((tris, sph), d_hits, len(rays), EIGHT_LIGHTS, args.steps)
    print(json.dumps({"workload": "b_cornell_4k_8_lights", **res}), flush=True)
    del d_hits, d_s, d_md

    # (c): the 100 800-triangle box
    ttris, tsph = b200.scene_cornell_rt_tessellated(60)
    trays = rh.camera_rays(1024, 1024, 1024.0, cam, h.identity_R())
    _, d_thits = device_hits((ttris, tsph), trays)
    res, _ = run((ttris, tsph), d_thits, len(trays), h.DEFAULT_RT_LIGHTS, max(2, args.steps // 2))
    print(json.dumps({"workload": "c_tess100k_1m", **res}), flush=True)
    del d_thits

    # (d): a nine-sample 1280x720 frame, composed against fused
    W, H, f = 1280, 720, 720.0
    frays = rh.camera_rays(W, H, f, cam, h.identity_R(), rh.NINE_SAMPLES)
    n = len(frays)
    r.rt_upload_scene(tris, sph)
    d_frays = torch.from_numpy(frays.view(np.uint8).reshape(-1).copy()).cuda()
    d_fhits = torch.empty(n * 28, dtype=torch.uint8, device="cuda")
    d_fpow = torch.empty(n * 3, dtype=torch.float32, device="cuda")
    d_rgb = torch.empty(W * H * 3, dtype=torch.float32, device="cuda")
    c = b200.make_camera(cam, f, h.identity_R(), W, H)
    times = {"composed": [], "fused": []}
    for step in range(args.steps + 1):
        ms = timed(lambda: r.rt_closest_hits_device(d_frays.data_ptr(), n, d_fhits.data_ptr()), step)["gpu_ms"]
        ms += timed(lambda: r.rt_direct_light_device(d_fhits.data_ptr(), n, h.DEFAULT_RT_LIGHTS, d_fpow.data_ptr()),
                    step)["gpu_ms"]
        fused = timed(lambda: r.rt_render_device(c, h.DEFAULT_RT_LIGHTS, 0, H, d_rgb.data_ptr()), step)["gpu_ms"]
        if step:
            times["composed"].append(ms)
            times["fused"].append(fused)
    fh = d_fhits.cpu().numpy().view(rh.RT_INTERSECTION)
    rgb = dh.draw_accumulate(fh, d_fpow.cpu().numpy().reshape(n, 1, 3), tris, sph)
    med = {k: float(np.median(v)) for k, v in times.items()}
    print(json.dumps({"workload": "d_frame_720p_composed", "samples": n, "composed_ms": round(med["composed"], 3),
                      "fused_ms": round(med["fused"], 3), "ratio": round(med["composed"] / med["fused"], 2),
                      "pixels_identical": bool(np.array_equal(rgb.reshape(-1).view(np.uint32),
                                                              d_rgb.cpu().numpy().view(np.uint32)))}), flush=True)
    r.close()


if __name__ == "__main__":
    main()
