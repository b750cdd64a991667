"""Where does the fixed ~0.4 ms of a small launch go?  Times single rays / small ray lists (development aid)."""
import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "bih-gpu-raytracer_b200"))
import bihrt
from bihrt import scenes
st = torch.cuda.Stream()
r = bihrt.Renderer(0, stream=st.cuda_stream)
tri = scenes.displaced_sphere(scenes.SPHERE_NSEG["1m"])
r.load_models(torch.from_numpy(tri).cuda()).build(); r.sync()
w, h = 480, 270
cam = scenes.pinhole_camera(aspect=w / h)
rays = scenes.camera_rays(cam, w, h)
def timed(fn, reps=7):
    ts = []
    for _ in range(reps):
        with torch.cuda.stream(st):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st); fn(); e1.record(st)
        torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
    return min(ts)
def run(name, rr):
    d = torch.from_numpy(np.ascontiguousarray(rr)).cuda()
    n = len(rr)
    ot = torch.empty(n, dtype=torch.float32, device="cuda"); os_ = torch.empty(n, dtype=torch.int32, device="cuda")
    _, _, _, cnt = r.trace(rr, counted=True)
    t = timed(lambda: r.trace(d, t=ot, slot=os_, prim=os_))
    print("%-44s rays %7d  %.3f ms   nodes/ray %.1f tris/ray %.1f" % (name, n, t, cnt["nodes"] / n, cnt["tris"] / n), flush=True)
k = 208 * w + 182
run("worst ray x32", np.repeat(rays[k:k + 1], 32, axis=0))
run("worst ray x1", rays[k:k + 1])
run("a centre ray x32", np.repeat(rays[(h // 2) * w + w // 2:(h // 2) * w + w // 2 + 1], 32, axis=0))
run("a miss ray x32", np.repeat(rays[0:1], 32, axis=0))
run("row 208 (480 rays)", rays[208 * w:209 * w])
run("whole 480x270 frame as a list", rays)
print("render 480x270: %.3f ms" % timed(lambda: r.render(cam, w, h, spp=1)))
