"""Cost of k-nearest-triangle queries (bihrt_closest_k) on one GPU, against bihrt_closest_point.

The timing rules are tools/bench_closest.py's (whose helpers this script uses): device-resident torch buffers, the context's
stream set to torch's current stream, CUDA events over --reps calls after --warmup calls, the L2 not flushed between calls, the
arms of a workload alternating run by run (--runs runs each), medians and spreads in Mqueries/s, and the GPU's name, power
limit and max SM clock from one nvidia-smi query in the same call.  Every arm asks for all the record's outputs (and count);
the k = 1 rows are checked equal to bihrt_closest_point's records.  Node fetches and distance evaluations per query come from
the CPU restatement of the walk (tests/closest_k_oracle.c) on --count-points of the same points.

Workloads (bench_closest.py's points):
  sphere_1m_near         1 M-triangle sphere, 1920x1080 primary hits moved +-1e-3 along the normal, unbounded radius
  sphere_1m_near_r001    the same points with rmax = 0.01; also the total at k = 0 (a pure count) and at k = 16
  sphere_1m_uniform      the same sphere, 2 M points uniform in 1.2x the scene box, unbounded radius
  atrium_near            the atrium, primary hits of the atrium camera moved +-1e-3, unbounded radius
Arms: closest_point (bihrt_closest_point), k1, k4, k16, k64 (bihrt_closest_k without the total).

    python tools/bench_closest_k.py --runs 5 --out profiles/bench_closest_k.json
"""
import argparse
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [ROOT, os.path.join(ROOT, "bih-gpu-raytracer_b200"), os.path.join(ROOT, "tests"), HERE]

from bench_closest import ALL, H, W, gpu_info, near_surface, summary, time_ms  # noqa: E402

KS = (1, 4, 16, 64)


def workloads(r):
    """Yields (name, device queries, extra arms {name: (k, total)}) one at a time (each loads its scene into r)."""
    import torch
    import bihrt
    from bihrt import scenes
    sphere = scenes.displaced_sphere(scenes.SPHERE_NSEG["1m"])
    r.load_models(sphere).build()
    near = near_surface(r, scenes.pinhole_camera(aspect=W / H))
    yield "sphere_1m_near", bihrt.point_queries(near), {}
    yield "sphere_1m_near_r001", bihrt.point_queries(near, 0.01), {"k0_total": (0, True), "k16_total": (16, True)}
    v = sphere.reshape(-1, 3)
    lo, hi = v.min(0), v.max(0)
    c, ext = (lo + hi) * 0.5, hi - lo
    pts = np.random.default_rng(17).uniform(c - 0.6 * ext, c + 0.6 * ext, (2 << 20, 3)).astype(np.float32)
    yield "sphere_1m_uniform", torch.from_numpy(bihrt.point_queries(pts)).cuda(), {}
    r.load_models(scenes.atrium()).build()
    yield "atrium_near", bihrt.point_queries(near_surface(r, scenes.atrium_camera(W / H))), {}


def restated_counts(r, q, arms, npts):
    """Node fetches and distance evaluations per query of the CPU restatement's walk on the exported blob, per arm, over npts
    of the queries (rows in a random order)."""
    import torch
    from closest_k_oracle import build_lib, run_closest_k
    from closest_oracle import blob_tree
    nbytes = r.bih_blob_bytes()
    blob = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    r.bih_export(blob, nbytes)
    r.sync()
    t = blob_tree(blob.cpu().numpy().view(np.uint32))
    lib = build_lib(tempfile.mkdtemp(prefix="bench_closest_k_"))
    qh = q.cpu().numpy()
    sel = qh[np.random.default_rng(0).permutation(len(qh))[:npts]]
    out = {}
    for arm, (k, total) in arms.items():
        c = run_closest_k(lib, t, sel, k, total=total)["counters"]
        out[arm] = {"nodes_per_query": c["nodes"] / len(sel), "dist_evals_per_query": c["tris"] / len(sel)}
    return {"points": int(len(sel)), "arms": out}


def bits(x):
    x = np.ascontiguousarray(x)
    return x.view(np.uint32) if x.dtype == np.float32 else x


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
        sys.exit("bench_closest_k: no CUDA device (there is no CPU fallback)")
    r = bihrt.Renderer(0)
    r.set_stream(torch.cuda.current_stream().cuda_stream)       # events and library calls on one stream
    res = {"gpu": gpu_info(), "l2_flushed": False, "reps": a.reps, "warmup": a.warmup, "workloads": {}}
    rows = ALL + ("count",)
    for name, q, extra in workloads(r):
        arms = {"closest_point": None}
        arms.update({"k%d" % k: (k, False) for k in KS})
        arms.update(extra)

        def call(arm):
            if arms[arm] is None:
                return r.closest_point(q, outputs=ALL)
            k, total = arms[arm]
            return r.closest_k(q, k, outputs=rows + (("total",) if total else ()))

        ms = {arm: [] for arm in arms}
        order = list(arms)
        for i in range(a.runs):
            for arm in (order if i % 2 == 0 else order[::-1]):      # alternate which arm goes first
                ms[arm].append(time_ms(lambda x=arm: call(x), a.reps, a.warmup))
        cp = {k: v.cpu().numpy() for k, v in call("closest_point").items()}
        k1 = {k: v.cpu().numpy() for k, v in call("k1").items()}
        same = all(np.array_equal(bits(k1[o][:, 0]), bits(cp[o])) for o in ALL)
        n = q.shape[0]
        s = {arm: {"ms": summary(ms[arm]), "mqueries_s_median": n / (summary(ms[arm])["median"] * 1e-3) / 1e6} for arm in order}
        w = {"queries": int(n), "arms": s, "k1_rows_equal_closest_point": bool(same),
             "hit_frac": float((cp["slot"] >= 0).mean())}
        if "k16_total" in arms:
            tot = call("k16_total")["total"].cpu().numpy()
            w["total_over_16_frac"] = float((tot > 16).mean())
            w["total_mean"] = float(tot.mean())
        if a.count_points:
            w["restated_counts"] = restated_counts(r, q, {arm: kt for arm, kt in arms.items() if kt is not None}, a.count_points)
        res["workloads"][name] = w
        print(name, json.dumps({arm: (round(v["ms"]["median"], 4), round(v["ms"]["spread_frac"], 4), round(v["mqueries_s_median"], 1))
                                for arm, v in s.items()}), "k1 == closest_point", same, flush=True)
    r.close()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
