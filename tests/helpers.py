"""ctypes/numpy plumbing shared by the tests and bench.py.

Three libraries are wrapped here:

* ``oracle/liboracle.so``      -- the plain-C restatement of the reference (checker)
* ``oracle/_ref/libref_*.so``  -- the unmodified reference compiled as a library
                                  (checker; built in the dev container, travels
                                  to the GPU box as a prebuilt file)
* the product C ABI (``include/b200render.h``) lives in the package, see
  ``computer-graphics_b200/__init__.py``.

Nothing here is product code.
"""
import ctypes
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_DIR = os.path.join(ORACLE_DIR, "_ref")

INDEX_MISS = -2147483648

RT_TRI = np.dtype([("v0", "<f4", 4), ("v1", "<f4", 4), ("v2", "<f4", 4),
                   ("normal", "<f4", 4), ("color", "<f4", 3)])
RT_SPHERE = np.dtype([("radius", "<f4"), ("radius2", "<f4"), ("centre", "<f4", 3),
                      ("color", "<f4", 3), ("normal", "<f4", 3)])
RAST_TRI = np.dtype([("v0", "<f4", 4), ("v1", "<f4", 4), ("v2", "<f4", 4),
                     ("normal", "<f4", 4), ("color", "<f4", 3),
                     ("texture", "<i4"), ("index", "<i4")])
assert RT_TRI.itemsize == 76 and RT_SPHERE.itemsize == 44 and RAST_TRI.itemsize == 84

c_f = ctypes.c_float
c_i = ctypes.c_int
VP = ctypes.c_void_p


def ptr(a):
    """void* of a numpy array (None -> NULL)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(VP)


def f32(*vals):
    return np.array(vals, dtype=np.float32)


def identity_R():
    return np.eye(4, dtype=np.float32).reshape(-1).copy()


def yaw_R(yaw):
    """The reference's yaw update (raytracer skeleton.cpp:236-238), column-major."""
    R = np.eye(4, dtype=np.float32)
    c, s = np.float32(np.cos(yaw)), np.float32(np.sin(yaw))
    # R[c][r] in glm = column c, row r ; flat index 4*c + r
    R[0, 0] = c; R[0, 2] = -s
    R[2, 0] = s; R[2, 2] = c
    return R.reshape(-1).copy()


# ----------------------------------------------------------------------------
# oracle (plain C restatement)
# ----------------------------------------------------------------------------
_oracle = None


def build_oracle():
    subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "liboracle.so"])


def oracle():
    global _oracle
    if _oracle is None:
        path = os.path.join(ORACLE_DIR, "liboracle.so")
        srcs = [os.path.join(ORACLE_DIR, f) for f in os.listdir(ORACLE_DIR) if f.endswith(".c")]
        if not os.path.exists(path) or any(os.path.getmtime(s) > os.path.getmtime(path) for s in srcs):
            build_oracle()
        _oracle = ctypes.CDLL(path)
    return _oracle


def lights_array(lights):
    """[(pos4, colour3), ...] -> flat float32[7*n]."""
    out = np.zeros((len(lights), 7), np.float32)
    for i, (p, c) in enumerate(lights):
        out[i, :4] = p
        out[i, 4:] = c
    return out.reshape(-1)


DEFAULT_RT_LIGHTS = [((0, -0.5, -0.7, 1.0), (14, 14, 14))]


def oracle_rt_render(W, H, focal, cam, R, lights7, tris, spheres, row0=0, row1=None,
                     want=("rgb", "dist", "index", "argb")):
    lib = oracle()
    row1 = H if row1 is None else row1
    rgb = np.zeros((H, W, 3), np.float32) if "rgb" in want else None
    dist = np.zeros((H, W), np.float32) if "dist" in want else None
    index = np.zeros((H, W), np.int32) if "index" in want else None
    argb = np.zeros((H, W), np.uint32) if "argb" in want else None
    counts = np.zeros(2, np.uint64)
    n_l = len(lights7) // 7
    rc = lib.oracle_rt_render(c_i(W), c_i(H), c_f(focal), ptr(np.asarray(cam, np.float32)),
                              ptr(np.asarray(R, np.float32)), ptr(np.asarray(lights7, np.float32)),
                              c_i(n_l), ptr(tris), c_i(len(tris)), ptr(spheres),
                              c_i(0 if spheres is None else len(spheres)), c_i(row0), c_i(row1),
                              ptr(rgb), ptr(dist), ptr(index), ptr(argb), ptr(counts))
    assert rc == 0
    return dict(rgb=rgb, dist=dist, index=index, argb=argb, primary=int(counts[0]), shadow=int(counts[1]))


# ----------------------------------------------------------------------------
# compiled reference (oracle/_ref)
# ----------------------------------------------------------------------------
def have_ref(name):
    return os.path.exists(os.path.join(REF_DIR, name))


_ref_cache = {}


def ref_lib(name):
    if name not in _ref_cache:
        _ref_cache[name] = ctypes.CDLL(os.path.join(REF_DIR, name))
    return _ref_cache[name]


def ref_rt_testmodel():
    lib = ref_lib("libref_rt.so")
    tris = np.zeros(64, RT_TRI)
    sph = np.zeros(8, RT_SPHERE)
    nt, ns = c_i(0), c_i(0)
    assert lib.ref_rt_load_testmodel(ptr(tris), 64, ptr(sph), 8, ctypes.byref(nt), ctypes.byref(ns)) == 0
    return tris[:nt.value].copy(), sph[:ns.value].copy()


def ref_rt_draw(W, H, focal, cam, R, lights7, tris=None, spheres=None):
    lib = ref_lib("libref_rt.so")
    argb = np.zeros((H, W), np.uint32)
    rgb = np.zeros((H, W, 3), np.float32)
    rc = lib.ref_rt_draw(c_i(W), c_i(H), c_f(focal), ptr(np.asarray(cam, np.float32)),
                         ptr(np.asarray(R, np.float32)), ptr(np.asarray(lights7, np.float32)),
                         c_i(len(lights7) // 7), ptr(tris), c_i(0 if tris is None else len(tris)),
                         ptr(spheres), c_i(0 if spheres is None else len(spheres)), ptr(argb), ptr(rgb))
    assert rc == 0
    return dict(argb=argb, rgb=rgb)


def ref_rt_trace(W, H, focal, cam, R, tris=None, spheres=None):
    lib = ref_lib("libref_rt.so")
    dist = np.zeros((H, W), np.float32)
    index = np.zeros((H, W), np.int32)
    rc = lib.ref_rt_trace(c_i(W), c_i(H), c_f(focal), ptr(np.asarray(cam, np.float32)),
                          ptr(np.asarray(R, np.float32)), ptr(tris), c_i(0 if tris is None else len(tris)),
                          ptr(spheres), c_i(0 if spheres is None else len(spheres)), ptr(dist), ptr(index))
    assert rc == 0
    return dict(dist=dist, index=index)


# ----------------------------------------------------------------------------
# scene helpers (numpy; independent of both the reference and the product)
# ----------------------------------------------------------------------------
def compute_normals(tris):
    """Triangle::ComputeNormal (raytracer TestModelH.h:96-105) in float32 steps."""
    v0 = tris["v0"][:, :3]; v1 = tris["v1"][:, :3]; v2 = tris["v2"][:, :3]
    e1 = (v1 - v0).astype(np.float32)
    e2 = (v2 - v0).astype(np.float32)
    # glm::cross(e2, e1)
    cx = (e2[:, 1] * e1[:, 2]).astype(np.float32) - (e1[:, 1] * e2[:, 2]).astype(np.float32)
    cy = (e2[:, 2] * e1[:, 0]).astype(np.float32) - (e1[:, 2] * e2[:, 0]).astype(np.float32)
    cz = (e2[:, 0] * e1[:, 1]).astype(np.float32) - (e1[:, 0] * e2[:, 1]).astype(np.float32)
    d = ((cx * cx).astype(np.float32) + (cy * cy).astype(np.float32)).astype(np.float32)
    d = (d + (cz * cz).astype(np.float32)).astype(np.float32)
    inv = (np.float32(1.0) / np.sqrt(d, dtype=np.float32)).astype(np.float32)
    tris["normal"][:, 0] = cx * inv
    tris["normal"][:, 1] = cy * inv
    tris["normal"][:, 2] = cz * inv
    tris["normal"][:, 3] = 1.0
    return tris


def random_rt_scene(n_tris, seed, extent=1.0, size=0.6, n_spheres=1):
    rng = np.random.default_rng(seed)
    tris = np.zeros(n_tris, RT_TRI)
    c = rng.uniform(-extent, extent, (n_tris, 3)).astype(np.float32)
    tris["v0"][:, :3] = c
    tris["v1"][:, :3] = c + rng.uniform(-size, size, (n_tris, 3)).astype(np.float32)
    tris["v2"][:, :3] = c + rng.uniform(-size, size, (n_tris, 3)).astype(np.float32)
    tris["v0"][:, 3] = tris["v1"][:, 3] = tris["v2"][:, 3] = 1.0
    tris["color"] = rng.uniform(0.15, 0.75, (n_tris, 3)).astype(np.float32)
    compute_normals(tris)
    sph = np.zeros(n_spheres, RT_SPHERE)
    for i in range(n_spheres):
        r = np.float32(rng.uniform(0.1, 0.4))
        sph[i]["radius"] = r
        sph[i]["radius2"] = r * r
        sph[i]["centre"] = rng.uniform(-0.7, 0.7, 3).astype(np.float32)
        sph[i]["color"] = rng.uniform(0.15, 0.75, 3).astype(np.float32)
    return tris, sph


# ----------------------------------------------------------------------------
# rasteriser: oracle + compiled reference wrappers
# ----------------------------------------------------------------------------
DEFAULT_RAST_LIGHT = dict(pos=(0.0, -0.5, 0.0, 1.0), power=(20.0, 20.0, 20.0), indirect=(0.2, 0.2, 0.2))
DEFAULT_RAST_CAM = (0.0, 0.0, -3.001, 1.0)


def ref_rast_name(W, H):
    return f"libref_rast_{W}x{H}.so"


def ref_rast_testmodel(W=64, H=48):
    lib = ref_lib(ref_rast_name(W, H))
    room, boxes = np.zeros(16, RAST_TRI), np.zeros(32, RAST_TRI)
    a, b = c_i(0), c_i(0)
    assert lib.ref_rast_load_testmodel(ptr(room), 16, ptr(boxes), 32, ctypes.byref(a), ctypes.byref(b)) == 0
    return room[:a.value].copy(), boxes[:b.value].copy()


def ref_rast_draw(W, H, focal, cam, R, light, room, boxes, clipped_cap=1 << 16):
    """Whole reference Draw on a world-space scene."""
    lib = ref_lib(ref_rast_name(W, H))
    out = dict(argb=np.zeros((H, W), np.uint32), rgb=np.zeros((H, W, 3), np.float32),
               depth=np.zeros((H, W), np.float32), screen_post=np.zeros((H, W, 3), np.float32),
               low=np.zeros((H, W, 3), np.float32), high=np.zeros((H, W, 3), np.float32),
               shadow=np.zeros((H, W), np.int32))
    clipped = np.zeros(clipped_cap, RAST_TRI)
    n = c_i(0)
    lc = np.zeros(4, np.float32)
    rc = lib.ref_rast_draw(c_f(focal), ptr(np.asarray(cam, np.float32)), ptr(np.asarray(R, np.float32)),
                           ptr(f32(*light["pos"])), ptr(f32(*light["power"])), ptr(f32(*light["indirect"])),
                           ptr(room), c_i(len(room)), ptr(boxes), c_i(len(boxes)),
                           ptr(out["argb"]), ptr(out["rgb"]), ptr(out["depth"]), ptr(out["screen_post"]),
                           ptr(out["low"]), ptr(out["high"]), ptr(out["shadow"]),
                           ptr(clipped), c_i(clipped_cap), ctypes.byref(n), ptr(lc))
    assert rc == 0, rc
    out["clipped"] = clipped[:n.value].copy()
    out["light_cam"] = lc
    return out


def ref_rast_draw_clipped(W, H, focal, light_cam, light, clipped, want_index=True):
    lib = ref_lib(ref_rast_name(W, H))
    out = dict(argb=np.zeros((H, W), np.uint32), rgb=np.zeros((H, W, 3), np.float32),
               depth=np.zeros((H, W), np.float32), screen=np.zeros((H, W, 3), np.float32),
               low=np.zeros((H, W, 3), np.float32), high=np.zeros((H, W, 3), np.float32),
               shadow=np.zeros((H, W), np.int32),
               index=np.zeros((H, W), np.int32) if want_index else None)
    rc = lib.ref_rast_draw_clipped(c_f(focal), ptr(np.asarray(light_cam, np.float32)), ptr(f32(*light["power"])),
                                   ptr(f32(*light["indirect"])), ptr(clipped), c_i(len(clipped)),
                                   ptr(out["argb"]), ptr(out["rgb"]), ptr(out["depth"]), ptr(out["screen"]),
                                   ptr(out["low"]), ptr(out["high"]), ptr(out["shadow"]), ptr(out["index"]))
    assert rc == 0
    return out


def oracle_rast_draw_clipped(W, H, focal, light_cam, light, clipped):
    lib = oracle()
    out = dict(argb=np.zeros((H, W), np.uint32), rgb=np.zeros((H, W, 3), np.float32),
               depth=np.zeros((H, W), np.float32), screen_post=np.zeros((H, W, 3), np.float32),
               low=np.zeros((H, W, 3), np.float32), high=np.zeros((H, W, 3), np.float32),
               shadow=np.zeros((H, W), np.int32), index=np.zeros((H, W), np.int32),
               screen=np.zeros((H, W, 3), np.float32))
    frags = np.zeros(1, np.uint64)
    rc = lib.oracle_rast_draw_clipped(c_i(W), c_i(H), c_f(focal), ptr(np.asarray(light_cam, np.float32)),
                                      ptr(f32(*light["power"])), ptr(f32(*light["indirect"])),
                                      ptr(clipped), c_i(len(clipped)), ptr(out["depth"]), ptr(out["screen_post"]),
                                      ptr(out["low"]), ptr(out["high"]), ptr(out["shadow"]), ptr(out["index"]),
                                      ptr(out["screen"]), ptr(out["rgb"]), ptr(out["argb"]), ptr(frags))
    assert rc == 0
    out["fragments"] = int(frags[0])
    return out


# ---- textures (rasteriser/Source/skeleton.cpp:63-75, 133-169): synthetic images, see oracle/refbuild/stubs/cv_stub.hpp ----
TEX_IMAGES = ("marble", "grill", "grill_opacity", "grill_normal", "woven", "woven_occlusion", "woven_opacity", "woven_normal")


def synthetic_textures(seed=7, noise_amp=0.01):
    """Random decoded images of the sizes findU / findV are called with (2000 for the marble, 1024 for the
    rest): three channels, except the two opacity maps, which are what cv::threshold leaves (one channel,
    0 / 255, in blocks so that holes have edges).  marble_noise is normalMap_marble (vec4 per entry)."""
    rng = np.random.default_rng(seed)
    t = {}
    for name in TEX_IMAGES:
        n = 2000 if name == "marble" else 1024
        if name.endswith("opacity"):
            blocks = rng.uniform(0, 1, (n // 16, n // 16)) < 0.7
            t[name] = np.ascontiguousarray(np.kron(blocks, np.ones((16, 16), bool)).astype(np.uint8) * np.uint8(255)).reshape(n, n, 1)
        else:
            t[name] = rng.integers(0, 256, (n, n, 3), dtype=np.uint8)
    noise = rng.uniform(-noise_amp, noise_amp, (2000 * 2000, 4)).astype(np.float32)
    noise[:, 3] = 0.0
    t["marble_noise"] = noise
    return t


REF_TEX_STEP = 4


def coarse_texture(im):
    """Every REF_TEX_STEP-th texel of every REF_TEX_STEP-th row, each repeated over its REF_TEX_STEP^2 block:
    what the committed fixture keeps of the metal-grill and woven-wood images (at full resolution they would
    take 4 MB), at the size the reference samples them with."""
    s = REF_TEX_STEP
    return np.ascontiguousarray(im[::s, ::s].repeat(s, axis=0).repeat(s, axis=1))


def reference_textures(seed=7, textures_dir=None):
    """The texture state the reference's main() builds (rasteriser/Source/skeleton.cpp:133-169) from the image
    files of ITS repository: metal grill and woven wood, decoded with OpenCV (cv2: the decoder cv::imread uses)
    and post-processed like :148-155 (BGR2GRAY, threshold 100 -> 0 / 255 on the two opacity maps).  The opacity
    maps are exact; the colour, normal and occlusion images go through coarse_texture.
    Textures/Marble2000x2000.jpg (:135) is not in the repository: marble and normalMap_marble stay synthetic.
    textures_dir: decode the reference's rasteriser/Textures/*.jpg from there (None when the files or cv2 are
    missing); otherwise the committed pixels, tests/golden/rast_reference_textures.npz (tests/golden/make_golden.py
    textures), which hold the images before the repetition of coarse_texture."""
    t = synthetic_textures(seed)
    if textures_dir is None:
        z = np.load(os.path.join(ROOT, "tests", "golden", "rast_reference_textures.npz"))
        for k in z.files:
            s = 1 if k.endswith("opacity") else REF_TEX_STEP
            t[k] = np.ascontiguousarray(z[k].repeat(s, axis=0).repeat(s, axis=1))
        return t
    d = textures_dir
    try:
        import cv2
    except ImportError:
        return None
    names = {"grill": "Metal_Grill_002_basecolor.jpg", "grill_opacity": "Metal_Grill_002_opacity.jpg",
             "grill_normal": "Metal_Grill_002_normal.jpg", "woven": "woven1024x1024.jpg",
             "woven_occlusion": "Wood_wicker_003_ambientOcclusion.jpg", "woven_opacity": "Wood_wicker_003_opacity.jpg",
             "woven_normal": "Wood_wicker_003_normal.jpg"}
    for key, f in names.items():
        im = cv2.imread(os.path.join(d, f), cv2.IMREAD_UNCHANGED)
        if im is None:
            return None
        if key.endswith("opacity"):
            gray = cv2.cvtColor(im, cv2.COLOR_BGR2GRAY)
            t[key] = np.ascontiguousarray(cv2.threshold(gray, 100, 255, cv2.THRESH_BINARY)[1].reshape(gray.shape[0], gray.shape[1], 1))
        else:
            t[key] = coarse_texture(im)
    return t


def ref_rast_set_textures(W, H, tex, cam, R, yaw):
    lib = ref_lib(ref_rast_name(W, H))
    for i, name in enumerate(TEX_IMAGES):
        im = tex[name]
        assert lib.ref_rast_set_image(c_i(i), ptr(im), c_i(im.shape[0]), c_i(im.shape[1]), c_i(im.shape[2])) == 0
    lib.ref_rast_set_marble_noise(ptr(tex["marble_noise"]), ctypes.c_longlong(len(tex["marble_noise"])))
    lib.ref_rast_set_view(ptr(np.asarray(cam, np.float32)), ptr(np.asarray(R, np.float32)), c_f(yaw))


_oracle_tex_keep = None


def oracle_rast_set_textures(tex, cam=None, R=None, yaw=0.0):
    """tex = None switches the oracle back to the untextured reading of every triangle."""
    global _oracle_tex_keep
    lib = oracle()
    _oracle_tex_keep = tex          # the oracle keeps pointers into these arrays
    lib.oracle_rast_enable_textures(c_i(0 if tex is None else 1))
    if tex is None:
        return
    for i, name in enumerate(TEX_IMAGES):
        im = tex[name]
        lib.oracle_rast_set_image(c_i(i), ptr(im), c_i(im.shape[0]), c_i(im.shape[1]), c_i(im.shape[1] * im.shape[2]))
    lib.oracle_rast_set_marble_noise(ptr(tex["marble_noise"]), ctypes.c_longlong(len(tex["marble_noise"])))
    lib.oracle_rast_set_view(ptr(np.asarray(cam, np.float32)), ptr(np.asarray(R, np.float32)), c_i(1 if yaw != 0 else 0))


_libc = None


def srand(seed):
    """Seeds the C library's rand() of this process -- shared by the compiled reference, the oracle and the
    product library (colour modes 1 / 2, rasteriser/Source/skeleton.cpp:647-662)."""
    global _libc
    if _libc is None:
        _libc = ctypes.CDLL(None)
    _libc.srand(ctypes.c_uint(seed))


def rand():
    srand.__doc__  # (same libc handle)
    return _libc.rand()


def ref_rast_testmodel_tex(setting, setting_boxes, W=64, H=48):
    lib = ref_lib(ref_rast_name(W, H))
    room, boxes = np.zeros(16, RAST_TRI), np.zeros(32, RAST_TRI)
    a, b = c_i(0), c_i(0)
    assert lib.ref_rast_load_testmodel_tex(c_i(setting), c_i(setting_boxes), ptr(room), 16, ptr(boxes), 32,
                                           ctypes.byref(a), ctypes.byref(b)) == 0
    return room[:a.value].copy(), boxes[:b.value].copy()


def rows_call(fn, focal, verts, cap=1 << 14, dims=None):
    y0, n = c_i(0), c_i(0)
    rows = np.zeros((cap, 8), np.float32)
    v = np.ascontiguousarray(verts, np.float32).reshape(-1)
    if dims is None:
        rc = fn(c_f(focal), ptr(v), ctypes.byref(y0), ctypes.byref(n), ptr(rows), c_i(cap))
    else:
        rc = fn(c_i(dims[0]), c_i(dims[1]), c_f(focal), ptr(v), ctypes.byref(y0), ctypes.byref(n), ptr(rows), c_i(cap))
    assert rc == 0
    return y0.value, rows[:n.value].copy()


def oracle_rast_geometry(W, H, focal, cam, R, light, room, boxes, cap=None):
    """Geometry stage (Draw :205-241) restated in C: clipped list + camera-space light."""
    lib = oracle()
    cap = cap or max(64, 40 * (len(room) + 7 * len(boxes)))
    out = np.zeros(cap, RAST_TRI)
    lc = np.zeros(4, np.float32)
    n = lib.oracle_rast_geometry(c_i(W), c_i(H), c_f(focal), ptr(np.asarray(cam, np.float32)),
                                 ptr(np.asarray(R, np.float32)), ptr(f32(*light["pos"])), ptr(room),
                                 c_i(len(room)), ptr(boxes), c_i(len(boxes)), ptr(out), c_i(cap), ptr(lc))
    assert n >= 0
    return out[:n].copy(), lc


def clipped_equal(a, b):
    """Byte equality of two clipped lists, ignoring `index` of shadow-volume
    triangles (uninitialised in the reference, rasteriser skeleton.cpp:1705-1710)."""
    if len(a) != len(b):
        return False
    for k in ("v0", "v1", "v2", "normal", "color"):
        if not np.array_equal(np.ascontiguousarray(a[k]).view(np.uint32), np.ascontiguousarray(b[k]).view(np.uint32)):
            return False
    real = a["color"][:, 0] >= 0
    return np.array_equal(a["texture"], b["texture"]) and np.array_equal(a["index"][real], b["index"][real])


def oracle_rast_draw(W, H, focal, cam, R, light, room, boxes):
    """Whole Draw restated: geometry stage, then triangle loop + post pass."""
    clipped, lc = oracle_rast_geometry(W, H, focal, cam, R, light, room, boxes)
    out = oracle_rast_draw_clipped(W, H, focal, lc, light, clipped)
    out["clipped"], out["light_cam"] = clipped, lc
    return out


def smoke_rast(b200, r):
    """Used by __graft_entry__.smoke(): one small whole-Draw frame vs the oracle."""
    room, boxes = b200.scene_cornell_rast()
    W, H, f = 160, 120, 85.0
    cam = b200.make_camera(DEFAULT_RAST_CAM, f, identity_R(), W, H)
    L = b200.make_rast_light(DEFAULT_RAST_LIGHT["pos"], DEFAULT_RAST_LIGHT["power"], DEFAULT_RAST_LIGHT["indirect"])
    got = r.render_raster(room, boxes, cam, L)
    want = oracle_rast_draw(W, H, f, DEFAULT_RAST_CAM, identity_R(), DEFAULT_RAST_LIGHT, room, boxes)
    assert np.array_equal(got["index"], want["index"]), "RAST owner mismatch"
    assert np.array_equal(got["depth"].view(np.uint32), want["depth"].view(np.uint32)), "RAST depth mismatch"
    assert np.array_equal(got["rgb"].view(np.uint32), want["rgb"].view(np.uint32)), "RAST colour mismatch"
    st = r.stats()
    print(f"smoke RAST ok: {W}x{H}, {len(want['clipped'])} clipped triangles, {st['fragments']} fragments, "
          f"{st['gpu_ms']:.3f} ms, {st['kernel_launches']} launches")


def random_clipped_list(n, seed, W, H, focal, shadow_frac=0.3, size=0.5):
    """Camera-space triangles in front of the camera that project near the screen
    (what the reference's clip stage would hand to the triangle loop)."""
    rng = np.random.default_rng(seed)
    t = np.zeros(n, RAST_TRI)
    z = rng.uniform(0.5, 4.0, n).astype(np.float32)
    cx = (rng.uniform(-0.5, 0.5, n) * W / focal * z).astype(np.float32)
    cy = (rng.uniform(-0.5, 0.5, n) * H / focal * z).astype(np.float32)
    for name in ("v0", "v1", "v2"):
        t[name][:, 0] = cx + rng.uniform(-size, size, n).astype(np.float32)
        t[name][:, 1] = cy + rng.uniform(-size, size, n).astype(np.float32)
        t[name][:, 2] = np.maximum(z + rng.uniform(-size, size, n).astype(np.float32), np.float32(0.05))
        t[name][:, 3] = t[name][:, 2] / np.float32(focal)
    t["color"] = rng.uniform(0.15, 0.75, (n, 3)).astype(np.float32)
    sh = rng.uniform(0, 1, n) < shadow_frac
    t["color"][sh] = -1.0
    compute_normals(t)
    return t


# ----------------------------------------------------------------------------
# BASELINE's synthetic scenes restated in numpy (so that bench.py's reference arm and
# the CPU tests never load the product library); byte-equal to the product's builders
# (computer-graphics_b200/host/scenes.cpp), which tests/test_abi_and_host.py checks.
# ----------------------------------------------------------------------------
def golden_cornell_rt():
    g = np.load(os.path.join(ROOT, "tests", "golden", "rt_cornell.npz"))
    return g["tris"].view(RT_TRI).copy(), g["spheres"].view(RT_SPHERE).copy()


def golden_cornell_rast():
    g = np.load(os.path.join(ROOT, "tests", "golden", "rast_ref_cornell_64x48.npz"))
    return g["room"].view(RAST_TRI).copy(), g["boxes"].view(RAST_TRI).copy()


def scene_cornell_rt_tessellated(n):
    """BASELINE config 5: every Cornell triangle split into n*n similar triangles that keep the
    parent's colour and normal (n = 60: 100 800), plus the sphere."""
    base, sph = golden_cornell_rt()
    f = np.float32
    i_idx, j_idx = [], []
    for i in range(n):
        for j in range(2 * (n - i) - 1):
            i_idx.append(i); j_idx.append(j)
    i_idx, j_idx = np.array(i_idx), np.array(j_idx)
    jj, odd = j_idx // 2, (j_idx & 1) == 1
    # (s, u) of the three vertices of child (i, j)
    s = np.stack([np.where(odd, jj + 1, jj), jj + 1, jj], axis=1)
    u = np.stack([i_idx, np.where(odd, i_idx + 1, i_idx), i_idx + 1], axis=1)
    fs = (s.astype(f) / f(n)).astype(f)          # (float)s / (float)n
    fu = (u.astype(f) / f(n)).astype(f)
    per = len(i_idx)
    out = np.zeros(len(base) * per, RT_TRI)
    p0 = base["v0"][:, None, None, :3]; p1 = base["v1"][:, None, None, :3]; p2 = base["v2"][:, None, None, :3]
    d1 = (p1 - p0).astype(f); d2 = (p2 - p0).astype(f)
    pts = ((p0 + (fs[None, :, :, None] * d1).astype(f)).astype(f) + (fu[None, :, :, None] * d2).astype(f)).astype(f)
    pts = pts.reshape(len(base) * per, 3, 3)
    for k, name in enumerate(("v0", "v1", "v2")):
        out[name][:, :3] = pts[:, k]
        out[name][:, 3] = 1.0
    out["color"] = np.repeat(base["color"], per, axis=0)
    out["normal"] = np.repeat(base["normal"], per, axis=0)
    return out, sph


def scene_soup_rast(n, seed=0x5EED, edge=0.01):
    """BASELINE config 4: std::mt19937(seed) raw outputs, 24 bits each -> [0, 1)."""
    f = np.float32
    raw = np.random.RandomState(seed)._bit_generator.random_raw(12 * n).astype(np.uint32)   # init_genrand seeding
    u = ((raw >> np.uint32(8)).astype(f) * f(1.0 / 16777216.0)).astype(f).reshape(n, 12)

    def uni(lo, hi, x):
        return (f(lo) + ((f(hi) - f(lo)) * x).astype(f)).astype(f)
    t = np.zeros(n, RAST_TRI)
    t["v0"][:, :3] = uni(-1, 1, u[:, 0:3])
    t["v1"][:, :3] = (t["v0"][:, :3] + uni(-edge, edge, u[:, 3:6])).astype(f)
    t["v2"][:, :3] = (t["v0"][:, :3] + uni(-edge, edge, u[:, 6:9])).astype(f)
    t["v0"][:, 3] = t["v1"][:, 3] = t["v2"][:, 3] = 1.0
    t["color"] = uni(0.15, 0.75, u[:, 9:12])
    compute_normals(t)
    return t


# ---- the reference PROGRAMS (oracle/refbuild/prog_harness.cpp) ---------------------------
SDLK = {"UP": 0x40000052, "DOWN": 0x40000051, "LEFT": 0x40000050, "RIGHT": 0x4000004F,
        **{c: ord(c) for c in "wsadqenmiozxfg12 "}}


def prog_run(name, frames, model=None):
    """Runs the reference program `name` (libprog_*.so under oracle/_ref): its own main() with a
    script of key presses, `frames` = one list of key names per frame drawn.  The library is
    loaded from a private copy so that every run starts from the program's initial globals.
    Returns the screenshot main() saves after its loop, (H, W) uint32."""
    import shutil
    import tempfile
    src = os.path.join(REF_DIR, name)
    with tempfile.TemporaryDirectory() as tmp:
        # keep the $ORIGIN-relative rpath of the drop-in flavour working: same depth below ROOT
        d = os.path.join(ROOT, "oracle", "_ref")
        path = os.path.join(d, f".run_{os.getpid()}_{abs(hash((name, str(frames), tmp))) & 0xffffff:x}_{name}")
        shutil.copyfile(src, path)
        try:
            lib = ctypes.CDLL(path)
            if model is not None:   # (setting, settingBoxes) of TestModelH.h:9-10; the images are cv_stub.hpp's
                lib.prog_set_model(c_i(model[0]), c_i(model[1]))
            keys = np.array([SDLK[k] for fr in frames for k in fr] + [0], np.int32)
            lens = np.array([len(fr) for fr in frames], np.int32)
            shot = np.zeros(3840 * 2160, np.uint32)
            W, H = c_i(0), c_i(0)
            rc = lib.prog_run(ptr(keys), ptr(lens), c_i(len(frames)), ptr(shot), ctypes.byref(W), ctypes.byref(H))
            assert rc == 0
            return shot[: W.value * H.value].reshape(H.value, W.value).copy()
        finally:
            os.unlink(path)
