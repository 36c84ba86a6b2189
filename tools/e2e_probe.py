import importlib, os, sys, time
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
g19 = importlib.import_module("2019global_b200"); abi = g19.abi
W,H,SPP,D=1920,1080,64,5
sc, cam, light = g19.Octree.builtin(abi.SCENE_CORNELL, n=0, w=W, h=H)
rt = g19.RayTracer(cam, light, device=0); rt.setScene(sc); rt.start()
host = torch.empty(H*W*3, dtype=torch.uint8).pin_memory(); host_np = host.numpy().reshape(H,W,3)
d_rgb = torch.zeros(H*W*3, dtype=torch.uint8, device="cuda")
stream = torch.cuda.current_stream().cuda_stream
def t(f, n=20):
    f(); torch.cuda.synchronize(); t0=time.perf_counter()
    for _ in range(n): f()
    torch.cuda.synchronize(); return (time.perf_counter()-t0)/n*1e3
print("g19_render host rgb      : %.3f ms" % t(lambda: rt.run(W,H,mode=abi.MODE_PATH,want=("rgb",),out={"rgb":host_np},spp=SPP,max_depth=D,seed=0)))
p = rt.params(W,H,mode=abi.MODE_PATH,spp=SPP,max_depth=D,seed=0)
def dev_sync():
    rt.run_device(p, d_rgb=d_rgb.data_ptr(), stream=stream); torch.cuda.synchronize()
print("run_device + sync        : %.3f ms" % t(dev_sync))
def dev_copy():
    rt.run_device(p, d_rgb=d_rgb.data_ptr(), stream=stream); host.copy_(d_rgb, non_blocking=True); torch.cuda.synchronize()
print("run_device + D2H + sync  : %.3f ms" % t(dev_copy))
def dev_async():
    rt.run_device(p, d_rgb=d_rgb.data_ptr(), stream=stream)
print("run_device async         : %.3f ms" % t(dev_async))
t0=time.perf_counter(); rt.run_device(p, d_rgb=d_rgb.data_ptr(), stream=stream); t1=time.perf_counter(); torch.cuda.synchronize()
print("host enqueue time of one frame: %.3f ms" % ((t1-t0)*1e3))
import numpy as np
print("g19_render no outputs    : %.3f ms" % t(lambda: rt.run(W,H,mode=abi.MODE_PATH,want=(),spp=SPP,max_depth=D,seed=0)))
pageable = np.zeros((H,W,3), np.uint8)
print("g19_render pageable rgb  : %.3f ms" % t(lambda: rt.run(W,H,mode=abi.MODE_PATH,want=("rgb",),out={"rgb":pageable},spp=SPP,max_depth=D,seed=0)))
print("g19_render pinned rgb    : %.3f ms" % t(lambda: rt.run(W,H,mode=abi.MODE_PATH,want=("rgb",),out={"rgb":host_np},spp=SPP,max_depth=D,seed=0)))
import ctypes as C
L = rt._L
pp = rt.params(W,H,mode=abi.MODE_PATH,spp=SPP,max_depth=D,seed=0)
lightv = abi.d3(rt.light)
def raw():
    L.g19_render(rt.h, C.byref(rt.camera), lightv, C.byref(pp), C.c_void_p(host.data_ptr()), None, None)
print("g19_render raw ctypes    : %.3f ms" % t(raw))
