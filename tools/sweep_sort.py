"""Ray lists of the atrium (shadow / diffuse bounce), traced in list order and through the sort permutation (development aid)."""
import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "bih-gpu-raytracer_b200"))
import bihrt
from bihrt import scenes
st = torch.cuda.Stream()
r = bihrt.Renderer(0, stream=st.cuda_stream)
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
def timed(fn, reps=7):
    ts = []
    for _ in range(reps):
        with torch.cuda.stream(st):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st); fn(); e1.record(st)
        torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
    return float(np.median(ts))
for scene in ("atrium", "1m"):
    tri = scenes.atrium() if scene == "atrium" else scenes.displaced_sphere(scenes.SPHERE_NSEG[scene])
    cam = scenes.atrium_camera(1920 / 1080) if scene == "atrium" else scenes.pinhole_camera(aspect=1920 / 1080)
    with torch.cuda.stream(st):
        r.load_models(torch.from_numpy(tri).cuda()).build()
        tp = timed(lambda: r.render(cam, 1920, 1080, spp=1))
        print("%s primary 1080p x 1: %.3f ms %.0f Mrays/s" % (scene, tp, 1920 * 1080 / tp / 1e3), flush=True)
        for kind in ("shadow", "diffuse"):
            db, _ = r.secondary_rays(cam, 1920, 1080, spp=1, kind=kind, light=(0.0, 0.8, 0.0))
            n = len(db)
            ot = torch.empty(n, dtype=torch.float32, device="cuda"); os_ = torch.empty(n, dtype=torch.int32, device="cuda")
            _t, _s, _p, cnt = r.trace(db, counted=True)
            print("  %-8s nodes/ray %.1f tris/ray %.1f hit %.2f" % (kind, cnt["nodes"] / n, cnt["tris"] / n, float((_s >= 0).float().mean())), flush=True)
            for srt in (0, 1):
                r.set_option("trace_sort_rays", srt)
                r.trace(db, t=ot, slot=os_, prim=os_); r.sync()
                ms = timed(lambda: r.trace(db, t=ot, slot=os_, prim=os_))
                print("  %-8s sort=%d: %.3f ms %.0f Mrays/s (%d rays)" % (kind, srt, ms, n / ms / 1e3, n), flush=True)
            r.set_option("trace_sort_rays", 0)
