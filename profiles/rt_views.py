"""Batched views against one call per view, device-resident Cornell box.

For each resolution (320x256 at f = 256, 1280x720 at f = 720) and K in {1, 8, 64, 256} distinct poses, times
  seq    K rt_render_device calls, one per pose;
  batch  one rt_render_views_device call on the same poses,
into rgb, depth and packed-pixel device buffers of K frames.  CUDA events on the renderer's stream; three warm-up
steps per arm; the two arms alternate step by step; the L2 is overwritten (256 MiB write) before every timed step.
Prints the device and its power limit, then one JSON line per (resolution, K): median ms per view of each arm,
their ratio, and whether the two arms' outputs are bit-identical.

    python profiles/rt_views.py [--steps N]
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

b200 = importlib.import_module("computer-graphics_b200")
LIGHTS = h.DEFAULT_RT_LIGHTS


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        return None


def poses(K, W, H, f, seed):
    rng = np.random.default_rng(seed)
    cams = []
    for k in range(K):
        pos = h.f32(rng.uniform(-0.4, 0.4), rng.uniform(-0.3, 0.3), rng.uniform(-3.4, -2.4), 1)
        cams.append(b200.make_camera(pos, f * float(rng.uniform(0.8, 1.2)), h.yaw_R(float(rng.uniform(-0.35, 0.35))), W, H))
    return cams


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    dev = torch.cuda.get_device_name(0)
    print(json.dumps({"device": dev, "power_limit_w": power_limit_w()}), flush=True)
    r = b200.Renderer(0)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    r.set_stream(stream.cuda_stream)
    tris, sph = h.golden_cornell_rt()
    r.rt_upload_scene(tris, sph)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for (W, H, f) in ((320, 256, 256.0), (1280, 720, 720.0)):
        for K in (1, 8, 64, 256):
            cams = poses(K, W, H, f, seed=K)
            cam_arr = b200.make_cameras(cams)
            npix = W * H
            bufs = {arm: (torch.empty(K * npix * 3, dtype=torch.float32, device="cuda"),
                          torch.empty(K * npix, dtype=torch.float32, device="cuda"),
                          torch.empty(K * npix, dtype=torch.int32, device="cuda")) for arm in ("seq", "batch")}

            def seq():
                rgb, depth, argb = bufs["seq"]
                for k, c in enumerate(cams):
                    r.rt_render_device(c, LIGHTS, 0, H, rgb.data_ptr() + 12 * k * npix, depth.data_ptr() + 4 * k * npix,
                                       None, argb.data_ptr() + 4 * k * npix)

            def batch():
                rgb, depth, argb = bufs["batch"]
                r.rt_render_views_device(cam_arr, LIGHTS, rgb.data_ptr(), depth.data_ptr(), None, argb.data_ptr())

            arms = {"seq": seq, "batch": batch}
            for _ in range(args.warmup):
                for fn in arms.values():
                    fn()
            r.synchronize()
            ms = {a: [] for a in arms}
            for _ in range(args.steps):
                for a, fn in arms.items():
                    flush.fill_(1)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    fn()
                    e1.record(stream)
                    e1.synchronize()
                    ms[a].append(e0.elapsed_time(e1))
            r.synchronize()
            same = all(torch.equal(x.view(torch.int32), y.view(torch.int32)) for x, y in zip(bufs["seq"], bufs["batch"]))
            seq_ms, batch_ms = float(np.median(ms["seq"])) / K, float(np.median(ms["batch"])) / K
            print(json.dumps({"device": dev, "resolution": f"{W}x{H}", "focal": f, "K": K,
                              "seq_ms_per_view": round(seq_ms, 5), "batch_ms_per_view": round(batch_ms, 5),
                              "speedup": round(seq_ms / batch_ms, 3), "bit_identical": bool(same),
                              "steps": args.steps, "l2": "overwritten before every timed step"}), flush=True)
            del bufs
    r.set_stream(None)
    r.close()


if __name__ == "__main__":
    main()
