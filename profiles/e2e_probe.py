import importlib, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch
import helpers as h, bench
b = importlib.import_module("computer-graphics_b200")
w="rt_tess100k_4k"; kind,W,H,f=bench.WORKLOADS[w]
r=b.Renderer(0)
tris,sph=bench.scenes_rt(w)
tp=torch.from_numpy(tris.view(np.uint8).copy()).pin_memory(); sp=torch.from_numpy(sph.view(np.uint8).copy()).pin_memory()
th,sh=tp.numpy().view(b.RT_TRI),sp.numpy().view(b.RT_SPHERE)
cam=b.make_camera(bench.RT_CAM,f,h.identity_R(),W,H)
out=torch.empty(H*W,dtype=torch.int32).pin_memory()
argb=torch.empty(H*W,dtype=torch.int32,device="cuda")
def T(fn,n=5):
    fn(); fn()
    torch.cuda.synchronize(); t0=time.perf_counter()
    for _ in range(n): fn()
    torch.cuda.synchronize(); return (time.perf_counter()-t0)*1e3/n
print("upload_scene", T(lambda: (r.rt_upload_scene(th,sh), r.synchronize())))
print("render_device argb", T(lambda: (r.rt_render_device(cam,bench.RT_LIGHTS,0,H,None,None,None,argb.data_ptr()), r.synchronize())))
print("d2h 33MB", T(lambda: out.copy_(argb)))
print("draw_raytrace_band", T(lambda: r.draw_raytrace_band(th,sh,cam,bench.RT_LIGHTS,0,H,out.data_ptr())))
