"""Cost of winding-number queries (bihrt_winding_number) on one GPU.

Every arm runs on device-resident torch buffers, on the context's stream set to torch's current stream, timed with CUDA events
over --reps calls after --warmup calls (the L2 is NOT flushed between calls: the 1 M-triangle sphere's BIH and far-field table
are ~350 MB together, so most of a walk's fetches come from HBM; the atrium's fit in the 126 MB L2).  The arms of a workload
(beta 2 and beta 4) alternate run by run (--runs runs each); the script reports the median and the spread per arm in
Mqueries/s, the GPU's name, power limit and max SM clock (one nvidia-smi query), and, per workload and beta, the internal nodes,
far-field terms and exact triangle terms per query that the CPU restatement (tests/winding_oracle.c, the kernel's walk) counts
on --count-points of the same points.  No counted GPU variant exists: the counts come from the restatement.

The far-field table is built by the first call after a build: "table_build_ms" is that call's time minus a steady call's, on
32 points, per tree kind, over --runs builds.

Workloads:
  sphere_1m_near      1 M-triangle sphere, the pixel-centre primary hits of the 1920x1080 pinhole camera moved +-1e-3 along
                      the normal (alternating)
  sphere_1m_uniform   the same sphere, 2 M points uniform in 1.2x the scene box
  atrium_near         the atrium, the same construction as sphere_1m_near from the atrium camera

    python tools/bench_winding.py --runs 5 --out profiles/bench_winding.json
"""
import argparse
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "bih-gpu-raytracer_b200")
sys.path[:0] = [ROOT, PKG, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]

from bench_closest import gpu_info, near_surface, summary, time_ms  # noqa: E402

BETAS = (2.0, 4.0)


def workloads(r):
    """Yields (name, device queries) one at a time (each loads its scene into r)."""
    import torch
    import bihrt
    from bihrt import scenes
    sphere = scenes.displaced_sphere(scenes.SPHERE_NSEG["1m"])
    r.load_models(sphere).build()
    yield "sphere_1m_near", bihrt.point_queries(near_surface(r, scenes.pinhole_camera(aspect=16 / 9)))
    v = sphere.reshape(-1, 3)
    lo, hi = v.min(0), v.max(0)
    c, ext = (lo + hi) * 0.5, hi - lo
    pts = np.random.default_rng(17).uniform(c - 0.6 * ext, c + 0.6 * ext, (2 << 20, 3)).astype(np.float32)
    yield "sphere_1m_uniform", torch.from_numpy(bihrt.point_queries(pts)).cuda()
    r.load_models(scenes.atrium()).build()
    yield "atrium_near", bihrt.point_queries(near_surface(r, scenes.atrium_camera(16 / 9)))


def restated_counts(r, q, npts, lib):
    """Per beta: internal nodes, far-field terms and exact triangle terms per query of the CPU restatement's walk on the
    exported blob, over npts of the queries (rows in a random order)."""
    import torch
    from closest_oracle import blob_tree
    from winding_oracle import Winding
    nbytes = r.bih_blob_bytes()
    blob = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    r.bih_export(blob, nbytes)
    r.sync()
    t = blob_tree(blob.cpu().numpy().view(np.uint32))
    qh = q.cpu().numpy()
    sel = qh[np.random.default_rng(0).permutation(len(qh))[:npts]]
    w = Winding(lib)
    out = {}
    for beta in BETAS:
        _, c = w(t, sel, beta)
        out["beta_%g" % beta] = {k + "_per_query": v / len(sel) for k, v in c.items()}
    out["points"] = int(len(sel))
    return out


def table_build_ms(r, runs):
    """Per tree kind: time of the first winding_number call after a build minus a steady call's, on 32 points (1 M sphere)."""
    import torch
    import bihrt
    from bihrt import scenes
    sphere = scenes.displaced_sphere(scenes.SPHERE_NSEG["1m"])
    q = torch.from_numpy(bihrt.point_queries(np.zeros((32, 3), np.float32))).cuda()
    res = {}
    for kind, bits in (("parity", 30), ("quality_cap4", 63)):
        r.set_option("morton_bits", bits)
        r.load_models(sphere).build()
        first, steady = [], []
        for _ in range(runs):
            r.build()
            r.sync()
            first.append(time_ms(lambda: r.winding_number(q), 1, 0))
            steady.append(time_ms(lambda: r.winding_number(q), 10, 2))
        res[kind] = {"first_call_ms": summary(first), "steady_call_ms": summary(steady),
                     "table_build_ms_median": summary(first)["median"] - summary(steady)["median"]}
        print("table", kind, json.dumps(res[kind]["table_build_ms_median"]), flush=True)
    r.set_option("morton_bits", 30)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--reps", type=int, default=10, help="timed calls per run and arm")
    ap.add_argument("--warmup", type=int, default=2, help="untimed calls before each timed window")
    ap.add_argument("--count-points", type=int, default=20000, help="queries per workload the CPU restatement counts (0: none)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import bihrt
    if not torch.cuda.is_available():
        sys.exit("bench_winding: no CUDA device (there is no CPU fallback)")
    from winding_oracle import build_lib
    lib = build_lib(tempfile.mkdtemp(prefix="bench_winding_")) if a.count_points else None
    r = bihrt.Renderer(0)
    r.set_stream(torch.cuda.current_stream().cuda_stream)       # events and library calls on one stream
    res = {"gpu": gpu_info(), "l2_flushed": False, "reps": a.reps, "warmup": a.warmup, "workloads": {}}
    res["table_build"] = table_build_ms(r, a.runs)
    for name, q in workloads(r):
        ms = {b: [] for b in BETAS}
        for i in range(a.runs):
            for beta in (BETAS if i % 2 == 0 else BETAS[::-1]):        # alternate which arm goes first
                ms[beta].append(time_ms(lambda b=beta: r.winding_number(q, b), a.reps, a.warmup))
        n = q.shape[0]
        arms = {}
        for beta in BETAS:
            w = r.winding_number(q, beta).cpu().numpy()
            s = summary(ms[beta])
            arms["beta_%g" % beta] = {"ms": s, "mqueries_s_median": n / (s["median"] * 1e-3) / 1e6,
                                      "inside_frac": float((w > 0.5).mean()), "nan": int(np.isnan(w).sum())}
        wl = {"queries": int(n), "arms": arms}
        if a.count_points:
            wl["restated_counts"] = restated_counts(r, q, a.count_points, lib)
        res["workloads"][name] = wl
        print(name, json.dumps({k: (round(v["ms"]["median"], 4), round(v["ms"]["spread_frac"], 4), round(v["mqueries_s_median"], 1))
                                for k, v in arms.items()}), wl.get("restated_counts"), flush=True)
    r.close()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
