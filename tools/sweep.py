"""Sweep trace-kernel options in one process (development aid)."""
import argparse, itertools, os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "bih-gpu-raytracer_b200"))
import bihrt
from bihrt import scenes
ap = argparse.ArgumentParser()
ap.add_argument("--scene", default="1m"); ap.add_argument("--w", type=int, default=1920); ap.add_argument("--h", type=int, default=1080)
ap.add_argument("--spp", default="1,16"); ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--sets", default="", help="semicolon-separated option sets k=v,k=v")
a = ap.parse_args()
st = torch.cuda.Stream()
r = bihrt.Renderer(0, stream=st.cuda_stream)
tri = scenes.atrium() if a.scene == "atrium" else scenes.displaced_sphere(scenes.SPHERE_NSEG[a.scene])
cam = scenes.atrium_camera(a.w / a.h) if a.scene == "atrium" else scenes.pinhole_camera(aspect=a.w / a.h)
r.load_models(torch.from_numpy(tri).cuda()).build(); r.sync()
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
DEFAULTS = {"trace_blocks_per_sm": 0, "trace_sm_queues": -1, "trace_lane_groups": -1}
for oset in a.sets.split(";"):
    opts = dict(DEFAULTS)
    for kv in filter(None, oset.split(",")):
        k, v = kv.split("="); opts[k] = int(v)
    for k, v in opts.items():
        r.set_option(k, v)
    res = []
    for spp in [int(x) for x in a.spp.split(",")]:
        ts = []
        for _ in range(a.reps):
            with torch.cuda.stream(st):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st); r.render(cam, a.w, a.h, spp=spp, jitter=spp > 1); e1.record(st)
            torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
        res.append("spp%d %.0f Mr/s" % (spp, a.w * a.h * spp / min(ts) / 1e3))
    cnt = r.render_counted(cam, a.w // 2, a.h // 2, spp=1)
    print("%-70s %s  nodes/ray %.1f" % (oset or "(default)", "  ".join(res), cnt["nodes"] / cnt["rays"]), flush=True)
