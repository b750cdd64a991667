"""Sweep trace options on secondary-ray lists (shadow / diffuse bounce from the atrium's primary hits)."""
import argparse, os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "bih-gpu-raytracer_b200"))
import bihrt
from bihrt import scenes
ap = argparse.ArgumentParser(); ap.add_argument("--sets", default=""); ap.add_argument("--scene", default="atrium"); a = ap.parse_args()
st = torch.cuda.Stream(); r = bihrt.Renderer(0, stream=st.cuda_stream)
if a.scene == "atrium": tri, cam = scenes.atrium(), scenes.atrium_camera(1920 / 1080)
else: tri, cam = scenes.displaced_sphere(scenes.SPHERE_NSEG[a.scene]), scenes.pinhole_camera(aspect=1920 / 1080)
r.load_models(torch.from_numpy(tri).cuda()).build(); r.sync()
W, H = 1920, 1080
t_, s_, p_ = r.render_hits(cam, W, H, spp=1)
u = (np.arange(W, dtype=np.float32) + 0.5) / W; v = (np.arange(H, dtype=np.float32) + 0.5) / H
dirs = (cam[3:6][None, None, :] + u[None, :, None] * cam[6:9][None, None, :] + v[:, None, None] * cam[9:12][None, None, :] - cam[:3]).reshape(-1, 3)
hit = s_ >= 0
P = cam[:3][None, :] + t_[hit, None] * dirs[hit]
vv = tri[p_[hit]].reshape(-1, 3, 3); nrm = np.cross(vv[:, 1] - vv[:, 0], vv[:, 2] - vv[:, 0]); nrm /= np.maximum(np.linalg.norm(nrm, axis=1, keepdims=True), 1e-20)
P = (P + 1e-3 * nrm).astype(np.float32)
rng = np.random.default_rng(1984); dd = rng.normal(size=P.shape); dd /= np.linalg.norm(dd, axis=1, keepdims=True); dd = np.where((dd * nrm).sum(1, keepdims=True) < 0, -dd, dd)
light = np.array([0.0, 0.8, 0.0], np.float32)
batches = {"shadow": np.concatenate([P, light - P], 1), "bounce": np.concatenate([P, dd], 1)}
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
DEF = {"trace_sm_queues": -1}
for oset in a.sets.split(";"):
    o = dict(DEF)
    for kv in filter(None, oset.split(",")):
        k, v2 = kv.split("="); o[k] = int(v2)
    for k, v2 in o.items(): r.set_option(k, v2)
    res = []
    for nm, b in batches.items():
        db = torch.from_numpy(np.ascontiguousarray(b, np.float32)).cuda(); ot = torch.empty(len(b), device="cuda"); oi = torch.empty(len(b), dtype=torch.int32, device="cuda")
        ts = []
        for _ in range(5):
            with torch.cuda.stream(st):
                flush.zero_(); e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st); r.trace(db, t=ot, slot=oi, prim=oi); e1.record(st)
            torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
        _, _, _, c = r.trace(db, t=ot, slot=oi, prim=oi, counted=True)
        res.append("%s %.0f Mr/s (n/r %.0f t/r %.0f)" % (nm, len(b) / min(ts) / 1e3, c["nodes"] / len(b), c["tris"] / len(b)))
    print("%-60s %s" % (oset or "(default)", "  ".join(res)), flush=True)
