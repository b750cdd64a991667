"""Cost of multi-hit ray queries (bihrt_intersect_k) against bihrt_intersect and against the peeling loop they replace, on one
GPU.

Timing rules are tools/bench_intersect.py's (its helpers are reused): device-resident torch buffers, the context's stream set
to torch's current stream, CUDA events over --reps calls after --warmup calls (the L2 is NOT flushed between calls), the arms
of a workload alternating run by run (--runs runs each), medians and spreads, the GPU's name, power limit and max SM clock
read in the same call.

Workloads (parity trees, the default build):
  sphere_1m_primary_two_sided  1 M-triangle sphere, 1920x1080 pixel-centre primary rays as a list, two-sided (entry and exit)
  atrium_camera_two_sided      the atrium camera's 1920x1080 primary rays, two-sided (many layers)
  atrium_diffuse               the atrium's diffuse bounce list at 1920x1080 (bihrt_secondary_rays), one-sided
Arms: bihrt_intersect (all outputs; the baseline) | intersect_k at k = 1 / 4 / 16 / 64 (all outputs and count) | k = 0 with
the total (a pure crossing count) | peeling loops of 4 and 16 bihrt_intersect calls, tmin set to the last t on the device
between calls (a miss ends the ray: tmin = NaN).

Agreement: the k = 1 row against bihrt_intersect (t bit for bit, slot up to exact-t ties), and the peeled t of every ray
against the distinct t of its rows at k = 64 where its total is <= 64.  Node fetches and triangle tests per ray of every arm
come from the CPU restatement (tests/intersect_k_oracle.c, tests/walk_oracle.c) on the exported blob of the tree the GPU
built and --cpu-rays rays of each list.

    python tools/bench_intersect_k.py --runs 5 --out profiles/bench_intersect_k.json
"""
import argparse
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [ROOT, os.path.join(os.path.dirname(ROOT), "tests")]

from bench_intersect import ALL, PKG, atrium_lists, gpu_info, sphere_primary_list, summary, time_ms  # noqa: E402

sys.path.insert(0, PKG)
KS = (1, 4, 16, 64)
PEELS = (4, 16)


def peel(r, x8, calls, two_sided):
    """calls bihrt_intersect calls, each from the last one's t; returns the (N, calls) t of every call (FLT_MAX: missed)"""
    import torch
    x = x8.clone()
    ts = []
    for _ in range(calls):
        h = r.intersect(x, two_sided=two_sided, outputs=ALL)
        ts.append(h["t"])
        x[:, 3] = torch.where(h["slot"] >= 0, h["t"], torch.full_like(h["t"], float("nan")))
    return torch.stack(ts, 1)


def workloads(r):
    """Yields (name, device rays8, two_sided, triangles) one workload at a time (each loads its scene into r)."""
    import torch
    import bihrt
    from bihrt import scenes
    w, h = 1920, 1080
    sphere = scenes.displaced_sphere(scenes.SPHERE_NSEG["1m"])
    r.load_models(sphere).build()
    yield "sphere_1m_primary_two_sided", bihrt.interval_rays(sphere_primary_list(w, h)), True, sphere
    atrium = scenes.atrium()
    r.load_models(atrium).build()
    cam = torch.from_numpy(scenes.camera_rays(scenes.atrium_camera(w / h), w, h)).cuda()
    yield "atrium_camera_two_sided", bihrt.interval_rays(cam), True, atrium
    _, diffuse = atrium_lists(r, w, h)
    yield "atrium_diffuse", bihrt.interval_rays(diffuse), False, atrium


def arms_of(r, x8, two_sided):
    arms = {"intersect": lambda: r.intersect(x8, two_sided=two_sided, outputs=ALL)}
    for k in KS:
        arms["k%d" % k] = lambda k=k: r.intersect_k(x8, k, two_sided=two_sided, outputs=ALL + ("count",))
    arms["k0_total"] = lambda: r.intersect_k(x8, 0, two_sided=two_sided, outputs=("count", "total"))
    for c in PEELS:
        arms["peel%d" % c] = lambda c=c: peel(r, x8, c, two_sided)
    return arms


def agreement(res):
    import numpy as np
    import torch
    a, b = res["k1"], res["intersect"]
    tie = a["slot"][:, 0] != b["slot"]
    out = {"k1_t_equal": bool(torch.equal(a["t"][:, 0], b["t"])), "k1_slot_ties": int(tie.sum().item()),
           "k1_ties_smaller_slot": bool((a["slot"][tie, 0] < b["slot"][tie]).all().item())}
    full = {o: v.cpu().numpy() for o, v in res["k64"].items()}
    total = res["k0_total"]["total"].cpu().numpy()
    ok = total <= 64
    ok[np.arange(len(ok)) % max(1, len(ok) // 50000) != 0] = False      # a strided subset of 50 k rays or fewer
    flt_max = np.float32(np.finfo(np.float32).max)
    for c in PEELS:
        peeled = res["peel%d" % c].cpu().numpy()
        bad = 0
        for i in np.nonzero(ok)[0]:
            d = sorted(set(full["t"][i, :full["count"][i]].tolist()))[:c]
            want = d + [float(flt_max)] * (c - len(d))
            bad += want != peeled[i].tolist()
        out["peel%d_rays_checked" % c] = int(ok.sum())
        out["peel%d_mismatches" % c] = int(bad)
    out["rays_total_over_64"] = int((total > 64).sum())
    return out


def cpu_counts(r, tri, x8, two_sided, nrays, lib):
    """Node fetches and triangle tests per ray of every arm, from the CPU restatement on the tree r holds (its exported blob)
    and a strided subset of nrays rays of the list."""
    from types import SimpleNamespace
    import numpy as np
    import torch
    from closest_oracle import blob_tree
    from intersect_k_oracle import run_intersect_k
    from walk_oracle import FLT_MAX, Tree
    nbytes = r.bih_blob_bytes()
    blob = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    r.bih_export(blob, nbytes)
    r.sync()
    bt = blob_tree(blob.cpu().numpy().view(np.uint32))
    tree = SimpleNamespace(lib=lib, tri9=np.ascontiguousarray(tri, np.float32).reshape(-1, 9), hdr=bt.hdr, nodes=bt.nodes,
                           tris=bt.tris)
    step = max(1, len(x8) // nrays)
    r8 = x8[::step][:nrays].cpu().numpy()
    n = len(r8)

    def walk(rays):              # walk_oracle's closest-hit walk (Tree.walk) on the blob
        return Tree._run(tree, False, rays, "closest", 0.0, np.inf, two_sided, FLT_MAX)

    def per(c):
        return {"nodes": c["nodes"] / n, "tris": c["tris"] / n}
    out = {"rays": n, "intersect": per(walk(r8)["counters"])}
    for k in KS:
        out["k%d" % k] = per(run_intersect_k(lib, tree, r8, k, two_sided=two_sided)["counters"])
    out["k0_total"] = per(run_intersect_k(lib, tree, r8, 0, total=True, two_sided=two_sided)["counters"])
    for c in PEELS:
        x, acc = r8.copy(), {"nodes": 0, "tris": 0}
        for _ in range(c):
            h = walk(x)
            acc = {k: acc[k] + h["counters"][k] for k in acc}
            x[:, 3] = np.where(h["slot"] >= 0, h["t"], np.float32(np.nan))
        out["peel%d" % c] = per(acc)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20, help="timed calls per run and arm")
    ap.add_argument("--warmup", type=int, default=3, help="untimed calls before each timed window")
    ap.add_argument("--cpu-rays", type=int, default=4000, help="rays of each list counted on the CPU restatement")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import bihrt
    from intersect_k_oracle import build_lib
    if not torch.cuda.is_available():
        sys.exit("bench_intersect_k: no CUDA device (there is no CPU fallback)")
    lib = build_lib(tempfile.mkdtemp(prefix="bench_intersect_k_"))
    r = bihrt.Renderer(0)
    r.set_stream(torch.cuda.current_stream().cuda_stream)       # events and library calls on one stream
    res = {"gpu": gpu_info(), "l2_flushed": False, "reps": a.reps, "warmup": a.warmup, "workloads": {}}
    for name, x8, two_sided, tri in workloads(r):
        n = x8.shape[0]
        arms = arms_of(r, x8, two_sided)
        ms = {k: [] for k in arms}
        order = list(arms)
        for i in range(a.runs):
            for arm in (order if i % 2 == 0 else order[::-1]):      # alternate which arm goes first
                ms[arm].append(time_ms(arms[arm], a.reps, a.warmup))
        results = {arm: arms[arm]() for arm in order}
        torch.cuda.synchronize()
        s = {arm: {"ms": summary(ms[arm]), "mrays_s_median": n / (summary(ms[arm])["median"] * 1e-3) / 1e6} for arm in order}
        base = s["intersect"]["ms"]["median"]
        for arm in order:
            s[arm]["time_vs_intersect"] = s[arm]["ms"]["median"] / base - 1.0
        total = results["k0_total"]["total"].float()
        res["workloads"][name] = {"rays": int(n), "two_sided": two_sided, "arms": s, "agreement": agreement(results),
                                  "total_mean": total.mean().item(), "total_max": int(total.max().item()),
                                  "per_ray_cpu": cpu_counts(r, tri, x8, two_sided, a.cpu_rays, lib)}
        print(name, json.dumps({k: (round(v["ms"]["median"], 4), round(v["ms"]["spread_frac"], 4),
                                    round(v["time_vs_intersect"], 4), round(v["mrays_s_median"], 1)) for k, v in s.items()}),
              json.dumps(res["workloads"][name]["agreement"]), flush=True)
    r.close()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
