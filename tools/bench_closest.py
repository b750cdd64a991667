"""Cost of closest-point queries (bihrt_closest_point) on one GPU.

Every arm runs on device-resident torch buffers, on the context's stream set to torch's current stream, timed with CUDA events
over --reps calls after --warmup calls (the L2 is NOT flushed between calls: the 1 M-triangle BIH is ~100 MB and mostly stays
resident in the 126 MB L2, the atrium's entirely).  The arms of a workload alternate run by run (--runs runs each); the script
reports the median and the spread per arm in Mqueries/s, the GPU's name, power limit and max SM clock (one nvidia-smi query),
and, per workload, the node fetches and distance evaluations per query that the CPU restatement of the walk
(tests/closest_oracle.c, the kernel's order and pruning) counts on --count-points of the same points.  No counted GPU
variant exists: the counts come from the restatement.

Workloads (all outputs requested):
  sphere_1m_uniform      1 M-triangle sphere, 2 M points uniform in 1.2x the scene box, unbounded radius:
                         arms "random" (generation order) | "morton" (sorted on the host by the points' 30-bit Morton code;
                         the records are un-permuted and checked equal to the random arm's)
  sphere_1m_near         the same sphere, the pixel-centre primary hits of the 1920x1080 pinhole camera moved +-1e-3 along the
                         normal (alternating), unbounded radius
  sphere_1m_near_r001    the same points with rmax = 0.01
  atrium_near            the atrium, the same construction from the atrium camera, unbounded radius

    python tools/bench_closest.py --runs 5 --out profiles/bench_closest.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "bih-gpu-raytracer_b200")
sys.path[:0] = [ROOT, PKG, os.path.join(ROOT, "tests")]

ALL = ("d2", "u", "v", "slot", "prim", "q", "ng")
W, H = 1920, 1080


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True)
    except OSError as ex:
        return "unknown (%s)" % ex
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi: %d)" % q.returncode


def summary(xs):
    xs = sorted(xs)
    med = xs[len(xs) // 2] if len(xs) % 2 else 0.5 * (xs[len(xs) // 2 - 1] + xs[len(xs) // 2])
    return {"runs": xs, "median": med, "min": xs[0], "max": xs[-1], "spread_frac": (xs[-1] - xs[0]) / med}


def time_ms(fn, reps, warmup):
    import torch
    for _ in range(warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def morton_order(p):
    """Permutation sorting the points by the 30-bit Morton code of their cell in their own bounding box."""
    lo, hi = p.min(0), p.max(0)
    q = np.clip(((p - lo) / np.maximum(hi - lo, 1e-30) * 1024).astype(np.int64), 0, 1023)
    code = np.zeros(len(p), np.int64)
    for b in range(10):
        for k in range(3):
            code |= ((q[:, k] >> b) & 1) << (3 * b + 2 - k)
    return np.argsort(code, kind="stable")


def near_surface(r, cam):
    """Pixel-centre primary hits of `cam` (bihrt_intersect on the device) moved +-1e-3 along the unit normal, alternating."""
    import torch
    import bihrt
    from bihrt import scenes
    rays = torch.from_numpy(scenes.camera_rays(cam, W, H)).cuda()
    h = r.intersect(bihrt.interval_rays(rays), outputs=("t", "slot", "ng"))
    hit = h["slot"] >= 0
    p = rays[hit, 0:3] + h["t"][hit, None] * rays[hit, 3:6]
    n = h["ng"][hit] / h["ng"][hit].norm(dim=1, keepdim=True)
    sgn = torch.ones(p.shape[0], device=p.device)
    sgn[1::2] = -1.0
    return (p + 1e-3 * sgn[:, None] * n).contiguous()


def workloads(r):
    """Yields (name, {arm: device queries}, un-permutation per arm or None) one at a time (each loads its scene into r)."""
    import torch
    import bihrt
    from bihrt import scenes
    sphere = scenes.displaced_sphere(scenes.SPHERE_NSEG["1m"])
    r.load_models(sphere).build()
    v = sphere.reshape(-1, 3)
    lo, hi = v.min(0), v.max(0)
    c, ext = (lo + hi) * 0.5, hi - lo
    pts = np.random.default_rng(17).uniform(c - 0.6 * ext, c + 0.6 * ext, (2 << 20, 3)).astype(np.float32)
    perm = morton_order(pts)
    yield "sphere_1m_uniform", {"random": torch.from_numpy(bihrt.point_queries(pts)).cuda(),
                                "morton": torch.from_numpy(bihrt.point_queries(pts[perm])).cuda()}, {"morton": perm}
    near = near_surface(r, scenes.pinhole_camera(aspect=W / H))
    yield "sphere_1m_near", {"near": bihrt.point_queries(near)}, {}
    yield "sphere_1m_near_r001", {"near_r001": bihrt.point_queries(near, 0.01)}, {}
    r.load_models(scenes.atrium()).build()
    yield "atrium_near", {"near": bihrt.point_queries(near_surface(r, scenes.atrium_camera(W / H)))}, {}


def restated_counts(r, q, npts):
    """Node fetches, distance evaluations per query and the deepest stack of the CPU restatement's walk on the exported blob,
    over the first npts queries of q (rows in a random order)."""
    import torch
    from closest_oracle import blob_tree, build_lib, run_closest
    nbytes = r.bih_blob_bytes()
    blob = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    r.bih_export(blob, nbytes)
    r.sync()
    t = blob_tree(blob.cpu().numpy().view(np.uint32))
    lib = build_lib(tempfile.mkdtemp(prefix="bench_closest_"))
    qh = q.cpu().numpy()
    sel = qh[np.random.default_rng(0).permutation(len(qh))[:npts]]
    c = run_closest(lib, t, sel)["counters"]
    return {"points": int(len(sel)), "nodes_per_query": c["nodes"] / len(sel), "dist_evals_per_query": c["tris"] / len(sel),
            "max_stack": c["max_stack"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20, help="timed calls per run and arm")
    ap.add_argument("--warmup", type=int, default=3, help="untimed calls before each timed window")
    ap.add_argument("--count-points", type=int, default=100000, help="queries per workload the CPU restatement counts (0: none)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import bihrt
    if not torch.cuda.is_available():
        sys.exit("bench_closest: no CUDA device (there is no CPU fallback)")
    r = bihrt.Renderer(0)
    r.set_stream(torch.cuda.current_stream().cuda_stream)       # events and library calls on one stream
    res = {"gpu": gpu_info(), "l2_flushed": False, "reps": a.reps, "warmup": a.warmup, "workloads": {}}
    for name, arms, unperm in workloads(r):
        ms = {k: [] for k in arms}
        order = list(arms)
        for i in range(a.runs):
            for arm in (order if i % 2 == 0 else order[::-1]):      # alternate which arm goes first
                ms[arm].append(time_ms(lambda x=arms[arm]: r.closest_point(x, outputs=ALL), a.reps, a.warmup))
        results = {arm: {k: v.cpu().numpy() for k, v in r.closest_point(arms[arm], outputs=ALL).items()} for arm in order}
        same = True
        for arm, perm in unperm.items():          # un-permute the sorted arm: the same records as the list-order arm
            ref = results[order[0]]
            same &= all(np.array_equal(results[arm][k].view(np.uint32) if results[arm][k].dtype == np.float32 else results[arm][k],
                                       (ref[k].view(np.uint32) if ref[k].dtype == np.float32 else ref[k])[perm]) for k in ALL)
        n = next(iter(arms.values())).shape[0]
        s = {arm: {"ms": summary(ms[arm]), "mqueries_s_median": n / (summary(ms[arm])["median"] * 1e-3) / 1e6,
                   "hit_frac": float((results[arm]["slot"] >= 0).mean())} for arm in order}
        w = {"queries": int(n), "arms": s, "same_records": bool(same)}
        if a.count_points:
            w["restated_counts"] = restated_counts(r, arms[order[0]], a.count_points)
        res["workloads"][name] = w
        print(name, json.dumps({k: (round(v["ms"]["median"], 4), round(v["ms"]["spread_frac"], 4), round(v["mqueries_s_median"], 1),
                                    round(v["hit_frac"], 4)) for k, v in s.items()}),
              "same_records", same, w.get("restated_counts"), flush=True)
    r.close()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
