"""Primary rays traced as a device ray LIST (MODE 0) vs generated in the kernel (MODE 1), in row-major and in tile order."""
import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "bih-gpu-raytracer_b200"))
import bihrt
from bihrt import scenes
st = torch.cuda.Stream(); r = bihrt.Renderer(0, stream=st.cuda_stream)
key = sys.argv[1] if len(sys.argv) > 1 else "1m"
tri = scenes.displaced_sphere(scenes.SPHERE_NSEG[key]); cam = scenes.pinhole_camera(aspect=1920 / 1080)
r.load_models(torch.from_numpy(tri).cuda()).build(); r.sync()
W, H = 1920, 1080
rays = scenes.camera_rays(cam, W, H)                      # row-major pixel order
# tile order (8x4 tiles inside 32x32 tiles), like the render kernel walks pixels
idx = np.arange(W * H).reshape(H, W)
def tiled(a, th, tw):
    h2, w2 = a.shape[0] // th * th, a.shape[1] // tw * tw
    b = a[:h2, :w2].reshape(h2 // th, th, w2 // tw, tw).transpose(0, 2, 1, 3).reshape(-1, th * tw)
    return b
order = tiled(idx[:1056, :], 4, 8).reshape(-1)       # 1056 = 33*32 rows; fine for a benchmark
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
def bench(fn, n):
    ts = []
    for _ in range(6):
        with torch.cuda.stream(st):
            flush.zero_(); e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st); fn(); e1.record(st)
        torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
    return n / min(ts) / 1e3
print("render (MODE 1)          %.0f Mr/s" % bench(lambda: r.render(cam, W, H, spp=1), W * H))
for name, rr in (("row-major list", rays), ("8x4-tiled list", rays[order])):
    d = torch.from_numpy(np.ascontiguousarray(rr)).cuda(); n = len(rr)
    ot = torch.empty(n, device="cuda"); oi = torch.empty(n, dtype=torch.int32, device="cuda")
    print("%-24s %.0f Mr/s" % (name, bench(lambda: r.trace(d, t=ot, slot=oi, prim=oi), n)))
