#!/usr/bin/env python
"""Benchmark of the two hot paths on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--workload rt_cornell_4k|rt_tess100k_4k|rast_cornell_4k|rast_soup_4k|...]
                    [--dump-outputs DIR]

One JSON line on stdout (rank 0).  The headline line is the raytracer on BASELINE
config 3 (Cornell box at 3840x2160, 9 spp, shadow rays, rows shared by the GPUs):
metric Mrays/s = (primary + shadow rays) / s, whole job.  With --workload left at its
default the same line carries, as nested objects with the same keys,
    "raster"       BASELINE config 4: frames/s of the 1M-triangle soup at 3840x2160
    "rt_tess100k"  BASELINE config 5: Mrays/s of the 100 800-triangle Cornell box at 3840x2160
    "rt_cornell_default" / "rast_cornell_default"   BASELINE configs 1 and 2 (320x256 / 900x720), N = 1 only

A "step" is one frame.  `value` times the device-resident path (scene already in HBM)
with CUDA events on the launching stream: every rank writes the float planes of its rows
(RGB + depth) locally and the packed 0x80RRGGBB pixels -- what Draw(screen*) leaves in
screen->buffer -- into the frame assembled on rank 0.  N > 1: one process per GPU
(torchrun); the packed rows are stored straight into rank 0's frame over NVLink by the
render kernels' epilogue (or, --gather nccl, an NCCL gather) inside the timed region;
afterwards rank 0 renders the whole frame alone and bit-compares it with the assembled one
("parity").  `e2e` times the host-pointer C-ABI call (H2D of the scene from pinned memory,
render, D2H of the packed framebuffer into pinned memory): at N = 1 draw_*_band on the
rank's context, at N > 1 ONE caller (rank 0) with a multi-GPU context (b200_init_multi),
which is what a user of the reference's Draw(screen*) would hold.

--dump-outputs DIR writes, for every workload, what the last timed step left in the buffers the
timed path renders into, so that two builds can be compared output for output (the scenes and
the sample are fixed, so the inputs are the same from run to run):
    DIR/<workload>_argb.npy   packed 0x80RRGGBB pixels of the assembled frame, as float64 (exact)
    DIR/<workload>_rgb.npy    float RGB, (n, 3) float32            (N = 1 only)
    DIR/<workload>_depth.npy  float depth, (n,) float32            (N = 1 only; a raytraced pixel whose
                              primary ray hits nothing, +inf in the depth plane, is written as -1)
n pixels, in raster order: every pixel of a frame of at most DUMP_PIXELS, otherwise a fixed
sample (numpy default_rng(0)) of DUMP_PIXELS of them; the five default workloads take < 32 MB.

`cpu_baseline` (N = 1) runs the unmodified reference (oracle/_ref) on one core over a
bounded sample of the same frame and bit-compares what it rendered with the GPU's pixels.

--impl reference times the reference's own CPU renderer (oracle/_ref, the unmodified
reference compiled as a library) on the box's host cores, one process per core, on a
bounded sample of rows of the same frame.  That arm never loads the product library.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

FLOP_PER_RT_TEST = 39.0          # SURVEY.md 8(d): always-executed stage of one ray-triangle test
RAST_BYTES_PER_PIXEL = 16.0      # RGB f32 + depth f32 written once
RAST_BYTES_PER_TRI = 84.0        # input triangle read once
PROFILE_ROUND = "r02"

WORKLOADS = {
    # name: (kind, W, H, focal)
    "rt_cornell_4k": ("rt", 3840, 2160, 2160.0),
    "rt_tess100k_4k": ("rt", 3840, 2160, 2160.0),
    "rt_cornell_default": ("rt", 320, 256, 256.0),
    "rast_cornell_4k": ("rast", 3840, 2160, 1536.0),
    "rast_soup_4k": ("rast", 3840, 2160, 1536.0),
    "rast_cornell_default": ("rast", 900, 720, 512.0),
}
DEFAULT_WORKLOADS = ["rt_cornell_4k", "rast_soup_4k", "rt_tess100k_4k"]
# BASELINE configs 1 and 2 (the reference's own resolutions): single-GPU frames, carried at N = 1 only
DEFAULT_WORKLOADS_1GPU = ["rt_cornell_default", "rast_cornell_default"]
NESTED_KEY = {"rast_soup_4k": "raster", "rt_tess100k_4k": "rt_tess100k", "rt_cornell_default": "rt_cornell_default",
              "rast_cornell_default": "rast_cornell_default"}
RT_CAM = (0.0, 0.0, -3.0, 1.0)
RT_LIGHTS = [((0.0, -0.5, -0.7, 1.0), (14.0, 14.0, 14.0))]
RAST_CAM = (0.0, 0.0, -3.001, 1.0)
RAST_LIGHT = dict(pos=(0.0, -0.5, 0.0, 1.0), power=(20.0, 20.0, 20.0), indirect=(0.2, 0.2, 0.2))
TESS_WINDOW = (1200, 1800, 1440, 1)    # x0, y0, w, h of the config-5 CPU sample: sphere outline, floor, shadow edge (~12 s on one core)
DUMP_PIXELS = 1 << 18                  # --dump-outputs: 24 B a pixel, 6 MB a workload at most


def profile_json(name):
    """profiles/<round>/<name>: figures read out of the committed ncu captures."""
    for rnd in (PROFILE_ROUND, "r01"):
        path = os.path.join(ROOT, "profiles", rnd, name)
        try:
            with open(path) as f:
                return json.load(f), f"profiles/{rnd}/{name}"
        except (OSError, ValueError):
            continue
    return {}, None


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


def workload_config(workload, world):
    """Names the workload; identical in the B200 arm and the reference arm."""
    kind, W, H, focal = WORKLOADS[workload]
    c = {"workload": workload, "width": W, "height": H, "focal": focal}
    if kind == "rt":
        c.update(spp=9, triangles=100800 if workload == "rt_tess100k_4k" else 28, spheres=1, lights=len(RT_LIGHTS))
    else:
        c.update(triangles_in=1_000_000 if workload == "rast_soup_4k" else 30)
    c["parallelism"] = f"rows of one frame shared by {world} GPU(s)"
    c["l2"] = "GPU arm: L2 flushed between timed steps (256 MiB write)"
    return c


def scenes_rt(workload):
    import helpers as h
    return h.scene_cornell_rt_tessellated(60) if workload == "rt_tess100k_4k" else h.golden_cornell_rt()


_rast_scene_cache = {}


def scenes_rast(workload):
    import helpers as h
    if workload not in _rast_scene_cache:
        if workload == "rast_soup_4k":
            _rast_scene_cache[workload] = (h.scene_soup_rast(1_000_000), np.zeros(0, h.RAST_TRI))
        else:
            _rast_scene_cache[workload] = h.golden_cornell_rast()
    return _rast_scene_cache[workload]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
# the unmodified reference on the host cores (reference arm and cpu_baseline)
# ------------------------------------------------------------------------------------------
def window_R(W, H, x0, y0, w, hh):
    """R whose translation column turns a w x hh frame into the window at (x0, y0) of the W x H
    frame: dir = R * (u - w/2, v - hh/2, f, 1) (raytracer/Source/skeleton.cpp:126-128); exact for
    integer offsets and an identity rotation."""
    import helpers as h
    R = h.identity_R()
    R[12] = float(x0 - W // 2 + w // 2)
    R[13] = float(y0 - H // 2 + hh // 2)
    return R


def _ref_rt_window_worker(args):
    """Renders the window (x0, y0, w, hh) of the W x H frame with the reference's own Draw."""
    import helpers as h
    W, H, focal, x0, y0, w, hh, tris_b, sph_b, want_pixels = args
    tris = np.frombuffer(tris_b, h.RT_TRI)
    sph = np.frombuffer(sph_b, h.RT_SPHERE)
    t0 = time.perf_counter()
    out = h.ref_rt_draw(w, hh, focal, h.f32(*RT_CAM), window_R(W, H, x0, y0, w, hh), h.lights_array(RT_LIGHTS), tris, sph)
    dt = time.perf_counter() - t0
    return (dt, out["rgb"]) if want_pixels else dt


def _oracle_rt_count_worker(args):
    import helpers as h
    W, H, focal, x0, y0, w, hh, tris, sph, _ = args
    o = h.oracle_rt_render(w, hh, focal, h.f32(*RT_CAM), window_R(W, H, x0, y0, w, hh), h.lights_array(RT_LIGHTS),
                           np.frombuffer(tris, h.RT_TRI), np.frombuffer(sph, h.RT_SPHERE), want=())
    return o["primary"] + o["shadow"]


def sample_windows(H, n_windows, rows_each):
    """Evenly spaced row windows covering the frame top to bottom."""
    n_windows = max(1, min(n_windows, H // rows_each))
    if n_windows == 1:
        return [((H - rows_each) // 2, rows_each)]      # the middle of the frame
    step = (H - rows_each) / max(1, n_windows - 1) if n_windows > 1 else 0
    return [(int(round(i * step)), rows_each) for i in range(n_windows)]


def run_reference(args, workload):
    """--impl reference.  No product code on this path: scenes come from tests/helpers.py (numpy)
    and the committed fixtures, rendering from oracle/_ref."""
    import helpers as h
    from multiprocessing import get_context
    kind, W, H, focal = WORKLOADS[workload]
    if int(os.environ.get("RANK", "0")) != 0:
        return None
    cores = args.ref_cores or os.cpu_count() or 1
    if kind != "rt":
        return run_reference_rast(args, workload, cores)
    tris, sph = scenes_rt(workload)
    warmup, steps = args.warmup, args.steps
    if workload == "rt_tess100k_4k":
        # ~16 ms per pixel per core at 100 800 triangles: a 96-pixel piece of a row per core and step
        x0, y0, _, _ = TESS_WINDOW
        wins = [(x0 + 96 * (i % 8), y0 + 40 * (i // 8), 96, 1) for i in range(cores)]
        warmup = min(warmup, 1)
    else:
        wins = [(0, y, W, hh) for (y, hh) in sample_windows(H, cores * 2, 16)]
    jobs = [(W, H, focal, x, y, w, hh, tris.tobytes(), sph.tobytes(), False) for (x, y, w, hh) in wins]
    ctx = get_context("fork")
    with ctx.Pool(cores) as pool:
        rays = sum(pool.map(_oracle_rt_count_worker, jobs, chunksize=1))   # untimed: ray count of the sample
        times = []
        for step in range(warmup + steps):
            t0 = time.perf_counter()
            pool.map(_ref_rt_window_worker, jobs, chunksize=1)
            dt = time.perf_counter() - t0
            if step >= warmup:
                times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = rays / (ms * 1e-3) / 1e6
    sample = f"{len(wins)} windows of {wins[0][2]}x{wins[0][3]} px of the {W}x{H} frame ({rays} rays) per step"
    return {"impl": "reference", "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(workload, args.gpus),
            "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": cores, "kind": "reference", "sample": sample},
            "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def run_reference_rast(args, workload, cores):
    """Rasteriser reference arm: whole reference Draw (geometry + clip + triangle loop +
    post) at the workload's resolution; single-threaded by construction, so independent
    frames are rendered concurrently and frames/s is their aggregate."""
    from multiprocessing import get_context
    kind, W, H, focal = WORKLOADS[workload]
    n_proc = max(1, min(cores, 8))      # each process owns ~365 MB of static frame buffers at 4K
    warmup, steps = min(args.warmup, 1), args.steps   # a soup frame takes seconds on a core
    ctx = get_context("fork")
    with ctx.Pool(n_proc) as pool:
        times = []
        for step in range(warmup + steps):
            t0 = time.perf_counter()
            pool.map(_ref_rast_worker, [(workload, False)] * n_proc, chunksize=1)
            dt = time.perf_counter() - t0
            if step >= warmup:
                times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = n_proc / (ms * 1e-3)
    return {"impl": "reference", "metric": "frames/s", "value": value, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(workload, args.gpus),
            "cpu_baseline": {"value": value, "unit": "frames/s", "cores": n_proc, "kind": "reference",
                             "sample": f"{n_proc} whole frames per step, one per process"},
            "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def _ref_rast_worker(args):
    import helpers as h
    workload, want_pixels = args
    kind, W, H, focal = WORKLOADS[workload]
    room, boxes = scenes_rast(workload)
    lib = h.ref_lib(h.ref_rast_name(W, H))
    argb = np.zeros((H, W), np.uint32) if want_pixels else None
    t0 = time.perf_counter()
    rc = lib.ref_rast_draw(h.c_f(focal), h.ptr(h.f32(*RAST_CAM)), h.ptr(h.identity_R()), h.ptr(h.f32(*RAST_LIGHT["pos"])),
                           h.ptr(h.f32(*RAST_LIGHT["power"])), h.ptr(h.f32(*RAST_LIGHT["indirect"])),
                           h.ptr(room), h.c_i(len(room)), h.ptr(boxes), h.c_i(len(boxes)),
                           h.ptr(argb), None, None, None, None, None, None, None, h.c_i(0), None, None)
    assert rc == 0
    dt = time.perf_counter() - t0
    return (dt, argb) if want_pixels else dt


# ------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------
def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def dump_outputs(out_dir, workload, argb, rgb=None, depth=None):
    """--dump-outputs: the pixels of DUMP_PIXELS (see the module docstring) of the device frames
    argb (H, W) int32, rgb (H, W, 3) and depth (H, W) float32 as DIR/<workload>_<name>.npy."""
    import torch
    n = argb.numel()
    idx = np.arange(n) if n <= DUMP_PIXELS else np.sort(np.random.default_rng(0).choice(n, DUMP_PIXELS, replace=False))
    sel = torch.from_numpy(idx).to(argb.device)
    out = {"argb": argb.reshape(-1)[sel].cpu().numpy().view(np.uint32).astype(np.float64)}
    if rgb is not None:
        out["rgb"] = rgb.reshape(-1, 3)[sel].cpu().numpy()
        d = depth.reshape(-1)[sel].cpu().numpy()
        d[d == np.inf] = -1.0      # misses: hit distances are positive, so -1 is unambiguous
        out["depth"] = d
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{workload}_{name}.npy"), a)


def cpu_baseline_rt(b200, r, workload, W, H, focal, tris, sph):
    """The unmodified reference (oracle/_ref), one core, on a bounded sample of the same frame.
    The GPU renders the same windows through the C ABI: its counters give the sample's ray
    count, and its float colours are bit-compared with the reference's (parity on the headline
    configuration, every run)."""
    import helpers as h
    if not h.have_ref("libref_rt.so"):
        return {"value": None, "unit": "Mrays/s", "cores": 1, "kind": "reference", "sample": "oracle/_ref missing"}
    if workload == "rt_tess100k_4k":
        wins = [TESS_WINDOW]                     # ~7.5 s on one core at 100 800 triangles
    else:
        wins = [(0, y, W, hh) for (y, hh) in sample_windows(H, 30, 16)]
    rays, secs, px, bad = 0, 0.0, 0, 0
    for (x0, y0, w, hh) in wins:
        cam = b200.make_camera(RT_CAM, focal, window_R(W, H, x0, y0, w, hh), w, hh)
        got = r.render_raytrace(tris, sph, cam, RT_LIGHTS, want=("rgb",))
        st = r.stats()
        rays += st["primary_rays"] + st["shadow_rays"]
        dt, ref_rgb = _ref_rt_window_worker((W, H, focal, x0, y0, w, hh, tris.tobytes(), sph.tobytes(), True))
        secs += dt
        px += w * hh
        bad += int(np.count_nonzero((bits(got["rgb"]) != bits(ref_rgb)).any(axis=-1)))
    return {"value": rays / secs / 1e6, "unit": "Mrays/s", "cores": 1, "kind": "reference",
            "sample": f"{len(wins)} windows of {wins[0][2]}x{wins[0][3]} px of the {W}x{H} frame, {rays} rays, {secs:.1f} s",
            "parity_pixels_checked": px, "parity_rows_checked": sum(w[3] for w in wins), "mismatches": bad,
            "parity": "float RGB of the sampled windows, GPU (render_raytrace) vs reference Draw, bit for bit"}


def cpu_baseline_rast(b200, r, workload, room, boxes, cam, L):
    import helpers as h
    kind, W, H, focal = WORKLOADS[workload]
    if not h.have_ref(h.ref_rast_name(W, H)):
        return {"value": None, "unit": "frames/s", "cores": 1, "kind": "reference", "sample": "oracle/_ref missing"}
    n = 2 if workload == "rast_soup_4k" else 6
    _, ref_argb = _ref_rast_worker((workload, True))
    secs = [_ref_rast_worker((workload, False)) for _ in range(n)]
    got = r.draw_raster(room, boxes, cam, L)
    bad = int(np.count_nonzero(got != ref_argb))
    return {"value": 1.0 / float(np.median(secs)), "unit": "frames/s", "cores": 1, "kind": "reference",
            "sample": f"{n} whole frames (median), reference Draw incl. geometry and post pass",
            "parity_pixels_checked": W * H, "parity_rows_checked": H, "mismatches": bad,
            "parity": "screen->buffer of the whole frame, GPU (draw_raster) vs reference Draw, bit for bit"}


def run_b200(args, workloads):
    """Measures the given workloads in one process (one per GPU under torchrun); returns
    the list of result dicts on rank 0."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    out = [run_b200_one(args, w) for w in workloads]
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out


def run_b200_one(args, workload):
    import torch
    import torch.distributed as dist
    import helpers as h
    b200 = importlib.import_module("computer-graphics_b200")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    kind, W, H, focal = WORKLOADS[workload]
    peaks, peaks_src = measured_peaks()
    r = b200.Renderer(local)
    # one non-default stream carries the kernels, the NCCL gathers and the timing events
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    r.set_stream(stream.cuda_stream)
    if "B200_RAST_TILE_LOG2" in os.environ:      # tuning knob, default chosen by the library
        r.set_option(b200.OPT_RAST_TILE_LOG2, int(os.environ["B200_RAST_TILE_LOG2"]))
    row0, row1 = rank * H // world, (rank + 1) * H // world
    rows = row1 - row0
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- where each rank's share of the frame goes ------------------------------------
    # N == 1: plain device buffers.  N > 1: the frame lives on rank 0 and
    #   "p2p_store"  (default) every rank is handed a peer mapping of rank 0's frame
    #                (torch symmetric memory over NVLink) and its kernels store their rows
    #                straight into it -- the exchange happens in the epilogue of the render
    #                kernels, followed by one device-side barrier;
    #   "nccl"       each rank renders into a local band, then an NCCL gather to rank 0.
    # The device entry points address outputs as full frames (pixel (x, y) at y*W + x).
    gather, gather_note, symm_handles = "none", None, []
    # Every rank writes the float planes of its own rows (RGB + depth, 16 B per pixel: the
    # algorithmic output of SURVEY 8(d)) into LOCAL memory, and the packed 0x80RRGGBB pixels --
    # what Draw(screen*) leaves in screen->buffer -- into the frame that is assembled on rank 0.
    interleaved_rt = world > 1 and kind == "rt" and args.gather == "p2p"
    if interleaved_rt:          # blocks spread over the whole frame: full-size local planes
        loc_rgb = torch.empty((H, W, 3), dtype=torch.float32, device="cuda")
        loc_depth = torch.empty((H, W), dtype=torch.float32, device="cuda")
        p_rgb, p_depth = loc_rgb.data_ptr(), loc_depth.data_ptr()
    else:
        loc_rgb = torch.empty((rows, W, 3), dtype=torch.float32, device="cuda")
        loc_depth = torch.empty((rows, W), dtype=torch.float32, device="cuda")
        p_rgb = loc_rgb.data_ptr() - row0 * W * 12       # frame origin above the band
        p_depth = loc_depth.data_ptr() - row0 * W * 4
    band_argb = full_argb = frame_argb = None
    if world > 1 and args.gather == "p2p":
        try:
            import torch.distributed._symmetric_memory as symm
            frame_argb = symm.empty((H, W), dtype=torch.int32, device="cuda")
            h_argb = symm.rendezvous(frame_argb, dist.group.WORLD)
            p_argb = int(h_argb.buffer_ptrs[0])
            symm_handles = [h_argb, frame_argb]
            gather = "p2p_store"
        except Exception as e:                      # both branches are GPU paths; say which one ran
            gather_note = f"symmetric memory unavailable ({type(e).__name__}: {e}); NCCL gather used"
    if gather != "p2p_store":
        interleaved_rt = False
        band_argb = torch.empty((rows, W), dtype=torch.int32, device="cuda")
        p_argb = band_argb.data_ptr() - row0 * W * 4
        if world > 1:
            gather = "nccl_gather"
            if rank == 0:
                full_argb = torch.empty((H, W), dtype=torch.int32, device="cuda")

    def exchange():
        if gather == "p2p_store":
            symm_handles[0].barrier(channel=0)      # every rank's rows have landed in rank 0's frame
        elif gather == "nccl_gather":
            dist.gather(band_argb, list(full_argb.view(world, rows, W).unbind(0)) if rank == 0 else None, dst=0)

    def assembled():
        """rank 0: the packed frame the exchange left behind."""
        return frame_argb if gather == "p2p_store" else (full_argb if gather == "nccl_gather" else band_argb)

    result = {}
    pinned = torch.empty(rows * W, dtype=torch.int32).pin_memory()
    interleaved = False
    if kind == "rt":
        tris, sph = scenes_rt(workload)
        cam = b200.make_camera(RT_CAM, focal, h.identity_R(), W, H)
        r.rt_upload_scene(tris, sph)

        # N > 1 with the peer-mapped frame: the ranks share the frame by interleaved 16-row blocks
        # (better balanced than contiguous bands); each stores its blocks straight into rank 0's frame
        interleaved = interleaved_rt and gather == "p2p_store"
        if interleaved:
            r.set_option(b200.OPT_RT_INTERLEAVE_N, world)
            r.set_option(b200.OPT_RT_INTERLEAVE_R, rank)

        def step():
            if interleaved:
                r.rt_render_device(cam, RT_LIGHTS, 0, H, p_rgb, p_depth, None, p_argb)
            else:
                r.rt_render_device(cam, RT_LIGHTS, row0, row1, p_rgb, p_depth, None, p_argb)
            exchange()

        def render_alone(d_argb):
            r.set_option(b200.OPT_RT_INTERLEAVE_N, 1)
            r.rt_render_device(cam, RT_LIGHTS, 0, H, None, None, None, d_argb)
            r.synchronize()

        tris_pin = torch.from_numpy(tris.view(np.uint8).copy()).pin_memory()
        sph_pin = torch.from_numpy(sph.view(np.uint8).copy()).pin_memory()
        tris_h = tris_pin.numpy().view(b200.RT_TRI)
        sph_h = sph_pin.numpy().view(b200.RT_SPHERE)

        def step_e2e():
            r.draw_raytrace_band(tris_h, sph_h, cam, RT_LIGHTS, row0, row1, pinned.data_ptr())

        h2d = tris.nbytes + sph.nbytes
        d2h = rows * W * 4
    else:
        room, boxes = scenes_rast(workload)
        cam = b200.make_camera(RAST_CAM, focal, h.identity_R(), W, H)
        L = b200.make_rast_light(RAST_LIGHT["pos"], RAST_LIGHT["power"], RAST_LIGHT["indirect"])
        r.rast_upload_scene(room, boxes)
        # frames sized from the last verified frame instead of mid-frame read-backs; the
        # verification (b200_synchronize) is part of the step, so a frame that had to be
        # rendered twice would be timed twice
        r.set_option(b200.OPT_RAST_PIPELINED, 0 if args.rast_sync else 1)
        r.set_option(b200.OPT_RAST_BAND_CULL, 1)     # N > 1: every rank's geometry stage keeps its band's triangles only
        respec0 = r.stats()["respeculated"]

        respec_seen = [respec0]

        def step():
            r.rast_draw_device(cam, L, row0, row1, p_rgb, p_depth, None, p_argb)
            exchange()                           # enqueued behind the frame: no host round trip in between
            r.synchronize()                      # verifies the pipelined frame (renders it again if it outgrew its sizes)
            now = r.stats()["respeculated"]
            if world > 1 and now != respec_seen[0]:
                respec_seen[0] = now
                exchange()                       # ... in which case the rows were stored again

        def render_alone(d_argb):
            r.rast_draw_device(cam, L, 0, H, None, None, None, d_argb)
            r.synchronize()

        room_pin = torch.from_numpy(room.view(np.uint8).copy()).pin_memory()
        boxes_pin = torch.from_numpy(boxes.view(np.uint8).copy() if len(boxes) else np.zeros(84, np.uint8)).pin_memory()
        room_h = room_pin.numpy().view(b200.RAST_TRI)
        boxes_h = boxes_pin.numpy().view(b200.RAST_TRI)[: len(boxes)]

        def step_e2e():
            r.draw_raster_band(room_h, boxes_h, cam, L, row0, row1, pinned.data_ptr())

        h2d = room.nbytes + boxes.nbytes
        d2h = rows * W * 4

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        total_ms, launches, last_stats = 0.0, 0, None
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        wall0 = time.perf_counter()
        for _ in range(steps):
            flush.fill_(1)                       # L2 flush between timed iterations (not timed)
            if world > 1:
                dist.barrier()                   # the ranks enter the step together (not timed): no host skew in the exchange
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            total_ms += e0.elapsed_time(e1)
            last_stats = r.stats()
            launches += last_stats["kernel_launches"]
        barrier()
        wall = time.perf_counter() - wall0
        clocks = sampler.stop() if rank == 0 else None
        t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps, launches, last_stats, clocks, wall

    ms, launches, st, clocks, wall = timed(step, args.steps, max(args.warmup, 3))
    if args.dump_outputs:
        if rank == 0:       # N > 1: the float planes stay on the rank that rendered them
            dump_outputs(args.dump_outputs, workload, assembled(), *((loc_rgb, loc_depth) if world == 1 else ()))
        barrier()
    # whole-job units per step (sum over ranks of what each rank processed)
    if kind == "rt":
        units = torch.tensor([st["primary_rays"] + st["shadow_rays"], st["prim_tests"], st["exact_evals"]],
                             dtype=torch.float64, device="cuda")
    else:
        units = torch.tensor([1.0 / world, float(st["fragments"]), 0.0], dtype=torch.float64, device="cuda")
    kernel_ms = torch.tensor([st["gpu_ms"]], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(units, op=dist.ReduceOp.SUM)
        dist.all_reduce(kernel_ms, op=dist.ReduceOp.MAX)

    # ---- N > 1: the assembled frame against rank 0 rendering the whole frame alone ----------
    parity = None
    own_argb = None
    if world > 1:
        step()                                   # one more exchange whose result is inspected
        barrier()
        if rank == 0:
            a_argb = assembled()
            own_argb = torch.empty((H, W), dtype=torch.int32, device="cuda")
            render_alone(own_argb.data_ptr())
            torch.cuda.synchronize()
            bad = int((a_argb != own_argb).sum().item())
            parity = {"assembled_frame_vs_single_gpu": "bit-exact" if bad == 0 else "MISMATCH",
                      "pixels_checked": W * H, "argb_mismatches": bad,
                      "mode": ("interleaved 16-row blocks, " if interleaved else "row bands, ") + gather}
        barrier()
        if interleaved:
            r.set_option(b200.OPT_RT_INTERLEAVE_N, world)
            r.set_option(b200.OPT_RT_INTERLEAVE_R, rank)

    # ---- end to end: the call a user of the reference makes, host buffers in and out ---------
    # N = 1: draw_*_band on this context.  N > 1: ONE caller -- rank 0 -- with a multi-GPU context
    # (b200_init_multi: the library shares the frame among the N devices and returns when the
    # assembled frame is in the caller's pinned buffer); the other ranks wait on the host.
    e2e_note = None
    if world == 1:
        ms_e2e, _, _, _, _ = timed(step_e2e, args.steps, 3)
    else:
        host_group = dist.new_group(backend="gloo")
        ms_e2e = float("inf")                    # only rank 0 measures (and prints) it
        dist.barrier(group=host_group)
        if rank == 0:
            m = b200.Renderer(n_gpus=world)
            whole = torch.empty(H * W, dtype=torch.int32).pin_memory()

            def whole_frame():
                if kind == "rt":
                    m.draw_raytrace_band(tris_h, sph_h, cam, RT_LIGHTS, 0, H, whole.data_ptr())
                else:
                    m.draw_raster_band(room_h, boxes_h, cam, L, 0, H, whole.data_ptr())

            for _ in range(max(12, args.warmup)):  # warm-up: buffers, pipelined sizes, adaptive bands (they move every other frame), planned RT frames
                whole_frame()
            k = args.steps
            t0 = time.perf_counter()
            for _ in range(k):
                whole_frame()
            ms_e2e = (time.perf_counter() - t0) * 1e3 / k
            bad = int((whole.view(H, W).cuda() != own_argb).sum().item())
            parity["library_multi_frame_vs_single_gpu"] = "bit-exact" if bad == 0 else "MISMATCH"
            parity["library_multi_mismatches"] = bad
            m.close()
            e2e_note = (f"one caller (rank 0), b200_init_multi({world}): host wall clock of {k} blocking whole-frame calls; "
                        "the other ranks idle on a host barrier")
        dist.barrier(group=host_group)
        del own_argb


    config = workload_config(workload, world)
    detail = {"gather": gather, "gather_note": gather_note,
              "split": (f"interleaved 16-row blocks x{world}" if interleaved else f"row bands x{world}")}
    if kind == "rt":
        rays, tests = float(units[0]), float(units[1])
        value, unit, metric = rays / (ms * 1e-3) / 1e6, "Mrays/s", "Mrays/s"
        e2e_value = rays / (ms_e2e * 1e-3) / 1e6
        fp32_peak = r.measure_fp32_peak()
        # executed FP32 work: thread-level FADD + FMUL + 2 x FFMA of all kernels of one whole frame, from
        # the committed ncu counters of this workload (the count does not depend on the run)
        flops, flops_src = profile_json("rt_flops.json")
        fl = flops.get(workload)
        executed = float(fl["flop_per_frame"]) if fl else None
        achieved = executed / world / (float(kernel_ms) * 1e-3) / 1e12 if executed else None     # per GPU
        delivered = tests * FLOP_PER_RT_TEST / (float(kernel_ms) * 1e-3) / 1e12 / world
        roofline = {"bound": "fp32", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s",
                    "frac": achieved / fp32_peak if achieved else None, "traffic": None,
                    "kernel": "all kernels of the frame (rt_prep_planes_kernel, grid kernels, rt_filtered_kernel)",
                    "kernel_ms": float(kernel_ms),
                    "peak_source": "FFMA microbenchmark run in this process (b200_measure_fp32_peak)",
                    "executed_flop_per_frame": executed,
                    "executed_flop_source": (f"{flops_src}: smsp__sass_thread_inst_executed_op_fadd/fmul/ffma_pred_on.sum "
                                             "(ffma x 2) summed over the frame's launches") if fl else
                                            "no committed counter capture for this workload: achieved/frac not stated",
                    "work_delivered": {"tflops": delivered, "vs_peak": delivered / fp32_peak,
                                       "definition": f"{FLOP_PER_RT_TEST:.0f} flop per ray-primitive test x {tests:.0f} tests / time: "
                                                     "the reference's work delivered per second, NOT pipe utilisation "
                                                     "(the filters decide most pairs without executing them)",
                                       "exact_evals": float(units[2])}}
        detail["rays_per_frame"] = rays
    else:
        frames = 1.0
        value, unit, metric = frames / (ms * 1e-3), "frames/s", "frames/s"
        e2e_value = frames / (ms_e2e * 1e-3)
        n_in = len(room) + len(boxes)
        bytes_alg = W * H * RAST_BYTES_PER_PIXEL + n_in * RAST_BYTES_PER_TRI
        achieved = bytes_alg / world / (float(kernel_ms) * 1e-3) / 1e9
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": achieved / peaks["hbm_gbs"], "traffic": None, "kernel": "whole raster frame (all kernels)",
                    "kernel_ms": float(kernel_ms), "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peaks_src})",
                    "algorithmic_work": f"{bytes_alg / 1e6:.1f} MB per frame (16 B/pixel + 84 B/triangle)"}
        detail.update(fragments_per_frame=float(units[1]), pipelined=not args.rast_sync,
                      frames_rendered_twice=int(r.stats()["respeculated"] - respec0))

    traffic, traffic_src = profile_json("traffic.json")
    t = traffic.get(workload)
    if t:
        roofline["traffic"] = t.get("traffic_bytes")
        roofline["traffic_kernel"] = t.get("kernel")
        roofline["traffic_source"] = traffic_src
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r.set_stream(None)
        if kind == "rt":
            cpu = cpu_baseline_rt(b200, r, workload, W, H, focal, tris, sph)
        else:
            cpu = cpu_baseline_rast(b200, r, workload, room, boxes, cam, L)

    if rank == 0:
        result = {"metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps,
                  "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
                  "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config, "detail": detail,
                  "clocks": clocks,
                  "e2e": {"value": e2e_value, "unit": unit,
                          "h2d_bytes_per_step": int(h2d) * (world if kind == "rt" else 1),   # RT: scene to every device; RAST: one slice each
                          "d2h_bytes_per_step": H * W * 4, "ms_per_step": ms_e2e,
                          "call": "draw_raytrace_band" if kind == "rt" else "draw_raster_band", "note": e2e_note},
                  "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "parity": parity}
    r.set_stream(None)
    r.close()
    return result


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="default", choices=["default"] + sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--rast-sync", action="store_true",
                    help="rasteriser: read list/table sizes back mid-frame instead of pipelined frames")
    ap.add_argument("--gather", default="p2p", choices=["p2p", "nccl"],
                    help="N > 1: peer stores into rank 0's frame (default) or an NCCL gather")
    ap.add_argument("--ref-cores", type=int, default=0,
                    help="--impl reference: worker processes (default: every host core; the count is reported)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step rendered as DIR/<workload>_<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs: the reference arm renders samples of rows, not whole frames")
    # default: the headline raytracer line (BASELINE config 3) carrying the rasteriser figure
    # (config 4) and the large raytracer scene (config 5) as nested objects
    workloads = DEFAULT_WORKLOADS if args.workload == "default" else [args.workload]
    if args.workload == "default" and args.gpus == 1 and int(os.environ.get("WORLD_SIZE", "1")) == 1:
        workloads = workloads + DEFAULT_WORKLOADS_1GPU
    if args.impl == "reference":
        lines = [run_reference(args, w) for w in workloads]
    else:
        lines = run_b200(args, workloads)
    if int(os.environ.get("RANK", "0")) != 0:
        return
    line = lines[0]
    keep = ("metric", "value", "unit", "ms_per_step", "config", "detail", "e2e", "gpu_launches", "roofline",
            "cpu_baseline", "parity", "steps", "warmup")
    for w, nested in zip(workloads[1:], lines[1:]):
        if nested:
            line[NESTED_KEY.get(w, w)] = {k: nested[k] for k in keep if k in nested}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
