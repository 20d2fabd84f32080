"""Ray queries (rt_closest_hits_device / rt_occluded_device): the filtered kernel against B200_OPT_RT_BRUTEFORCE = 1.

Workloads (device-resident rays and results):
  (a) cornell_4k      the 8.29 M centre-sample camera rays of the Cornell box at 3840x2160, f = 2160, closest hits;
  (b) cornell_4k_perm the same rays randomly permuted (how much the cull owes to coherence);
  (c) shadow_4k       the DirectLight shadow rays of (a)'s hits, occlusion query with max_distance = r_mag;
  (d) tess100k_1m     1 M camera rays (1024 x 1024, f = 1024) of the 100 800-triangle tessellated box, closest hits.
Every step overwrites the L2 (256 MiB write) first; the two arms alternate step by step in one process.  Time per
call is the library's own CUDA-event time (b200_get_stats gpu_ms).  Prints the device and its power limit, then one
JSON line per workload: rays/s of each arm, exact_evals per ray of the filtered arm, the speed-up, and whether the two
arms' outputs are bit-identical.  Also checks on (a) that distances and indices equal render_raytrace's depth and
index planes of the same frame.

    python profiles/rt_rays.py [--steps N]
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

b200 = importlib.import_module("computer-graphics_b200")
FLT_MAX = np.finfo(np.float32).max


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
    tris, sph = b200.scene_cornell_rt()
    W, H, f = 3840, 2160, 2160.0
    cam = h.f32(0, 0, -3, 1)
    rays_a = rh.camera_rays(W, H, f, cam, h.identity_R())
    perm = np.random.default_rng(0).permutation(len(rays_a))
    ttris, tsph = b200.scene_cornell_rt_tessellated(60)
    rays_d = rh.camera_rays(1024, 1024, 1024.0, cam, h.identity_R())

    def run(scene, rays, md, steps):
        r.rt_upload_scene(*scene)
        n = len(rays)
        d_rays = torch.from_numpy(rays.view(np.uint8).reshape(-1).copy()).cuda()
        d_md = torch.from_numpy(md).cuda() if md is not None else None
        outs = {}
        times = {0: [], 1: []}
        evals = {}
        for step in range(steps + 1):   # step 0: warm-up
            for brute in (0, 1):
                r.set_option(b200.OPT_RT_BRUTEFORCE, brute)
                d_out = torch.empty(n * (1 if md is not None else 28), dtype=torch.uint8, device="cuda")
                flush.fill_(step & 255)
                torch.cuda.synchronize()
                if md is not None:
                    r.rt_occluded_device(d_rays.data_ptr(), d_md.data_ptr(), n, d_out.data_ptr())
                else:
                    r.rt_closest_hits_device(d_rays.data_ptr(), n, d_out.data_ptr())
                st = r.stats()
                if step:
                    times[brute].append(st["gpu_ms"])
                evals[brute] = st["exact_evals"]
                outs[brute] = d_out.cpu().numpy()
        r.set_option(b200.OPT_RT_BRUTEFORCE, 0)
        ms = {k: float(np.median(v)) for k, v in times.items()}
        res = {"rays": n, "filtered_ms": round(ms[0], 3), "brute_ms": round(ms[1], 3),
               "filtered_rays_per_s": n / (ms[0] * 1e-3), "brute_rays_per_s": n / (ms[1] * 1e-3),
               "speedup": round(ms[1] / ms[0], 2), "exact_evals_per_ray": round(evals[0] / n, 3),
               "brute_exact_evals_per_ray": round(evals[1] / n, 3),
               "filtered_ms_range": [round(min(times[0]), 3), round(max(times[0]), 3)],
               "identical": bool(np.array_equal(outs[0], outs[1]))}
        return res, outs[0]

    res, out_a = run((tris, sph), rays_a, None, args.steps)
    hits = out_a.view(rh.RT_INTERSECTION)
    frame = r.render_raytrace(tris, sph, b200.make_camera(cam, f, h.identity_R(), W, H), h.DEFAULT_RT_LIGHTS,
                              want=("depth", "index"))
    hit = hits["distance"] < FLT_MAX
    depth = np.where(hit, hits["distance"], np.float32(np.inf)).astype(np.float32)
    idx = np.where(hit, np.where(hits["triangle_index"] != -1, hits["triangle_index"], -1 - hits["sphere_index"]),
                   h.INDEX_MISS)
    res["equals_frame_depth_index"] = bool(np.array_equal(depth.view(np.uint32), frame["depth"].reshape(-1).view(np.uint32))
                                           and np.array_equal(idx, frame["index"].reshape(-1)))
    print(json.dumps({"workload": "a_cornell_4k", **res}), flush=True)

    res, _ = run((tris, sph), np.ascontiguousarray(rays_a[perm]), None, args.steps)
    print(json.dumps({"workload": "b_cornell_4k_permuted", **res}), flush=True)

    srays, r_mag, _ = rh.shadow_rays(hits, tris, sph, h.DEFAULT_RT_LIGHTS[0][0])
    res, _ = run((tris, sph), srays, np.ascontiguousarray(r_mag), args.steps)
    print(json.dumps({"workload": "c_shadow_4k", **res}), flush=True)

    res, _ = run((ttris, tsph), rays_d, None, max(2, args.steps // 2))
    print(json.dumps({"workload": "d_tess100k_1m", **res}), flush=True)
    r.close()


if __name__ == "__main__":
    main()
