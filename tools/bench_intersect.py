"""Cost of ray queries with intervals and hit records (bihrt_intersect) against the calls they generalise, on one GPU.

Every arm runs on device-resident torch buffers, on the context's stream set to torch's current stream, timed with CUDA
events over --reps calls after --warmup calls (the L2 is NOT flushed between calls: the BIH and the ray lists stay
resident in the 126 MB L2 where they fit).  The arms of a workload alternate run by run (--runs runs each); the script
reports the median and the spread per arm, the GPU's name and power limit, and whether the arms' results agree.

Workloads:
  sphere_1m_primary  1 M-triangle sphere, 1920x1080 pixel-centre primary rays as a list:
                     bihrt_trace  |  bihrt_intersect(0, inf) with t/slot/prim  |  bihrt_intersect(0, inf) with all outputs
  atrium_shadow      shadow list of the atrium at 1920x1080 (bihrt_secondary_rays):
                     bihrt_trace_any(tmax = 1)  |  bihrt_intersect ANY with per-ray (0, 1), slot only
  atrium_diffuse     diffuse bounce list of the atrium at 1920x1080:
                     bihrt_trace  |  bihrt_intersect(0, inf) with all outputs
Two-sided queries (BIHRT_INTERSECT_TWO_SIDED) against the one-sided query on the same list; their results differ by
design, so these report each arm's hit fraction and check that every one-sided hit is a two-sided hit with t <= its t:
  sphere_1m_primary_two_sided  the sphere_1m_primary list, all outputs: one-sided | two-sided
  atrium_diffuse_two_sided     the atrium_diffuse list, all outputs: one-sided | two-sided
  atrium_shadow_two_sided      the atrium_shadow list, ANY with per-ray (0, 1), slot only: one-sided | two-sided
  sphere_1m_inside_two_sided   1 M-triangle sphere, 1920x1080 camera inside it, all outputs: two-sided only (a one-sided
                               query sees nothing from there)

    python tools/bench_intersect.py --runs 5 --out bench_intersect.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "bih-gpu-raytracer_b200")
sys.path[:0] = [ROOT, PKG]

ALL = ("t", "u", "v", "slot", "prim", "ng")


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


def sphere_primary_list(w, h):
    """Pixel-centre primary rays of the 1 M-triangle sphere's camera, as a device list."""
    import torch
    from bihrt import scenes
    return torch.from_numpy(scenes.camera_rays(scenes.pinhole_camera(aspect=w / h), w, h)).cuda()


def atrium_lists(r, w, h):
    """Shadow and diffuse bounce lists (bihrt_secondary_rays) of the atrium camera; the atrium must be built in r."""
    from bihrt import scenes
    cam = scenes.atrium_camera(w / h)
    shadow, _ = r.secondary_rays(cam, w, h, spp=1, kind="shadow", light=(0.1, 0.8, -0.2))
    diffuse, _ = r.secondary_rays(cam, w, h, spp=1, kind="diffuse")
    return shadow.contiguous(), diffuse.contiguous()


def workloads(r):
    """Yields (name, device rays, {arm: call}) one workload at a time (each loads its scene into r)."""
    import torch
    import bihrt
    from bihrt import scenes
    w, h = 1920, 1080

    sphere = scenes.displaced_sphere(scenes.SPHERE_NSEG["1m"])
    r.load_models(sphere).build()
    prim6 = sphere_primary_list(w, h)
    yield "sphere_1m_primary", prim6, {
        "trace": lambda x=prim6: r.trace(x),
        "intersect_t_slot_prim": lambda x=bihrt.interval_rays(prim6): r.intersect(x, outputs=("t", "slot", "prim")),
        "intersect_all": lambda x=bihrt.interval_rays(prim6): r.intersect(x, outputs=ALL),
    }

    r.load_models(scenes.atrium()).build()
    shadow, diffuse = atrium_lists(r, w, h)
    yield "atrium_shadow", shadow, {
        "trace_any_tmax1": lambda x=shadow: r.trace_any(x, tmax=1.0),
        "intersect_any_0_1_slot": lambda x=bihrt.interval_rays(shadow, 0.0, 1.0): r.intersect(x, any_hit=True, outputs=("slot",)),
    }
    yield "atrium_diffuse", diffuse, {
        "trace": lambda x=diffuse: r.trace(x),
        "intersect_all": lambda x=bihrt.interval_rays(diffuse): r.intersect(x, outputs=ALL),
    }
    yield "atrium_diffuse_two_sided", diffuse, {
        "intersect_all": lambda x=bihrt.interval_rays(diffuse): r.intersect(x, outputs=ALL),
        "intersect_all_two_sided": lambda x=bihrt.interval_rays(diffuse): r.intersect(x, two_sided=True, outputs=ALL),
    }
    yield "atrium_shadow_two_sided", shadow, {
        "intersect_any_0_1_slot": lambda x=bihrt.interval_rays(shadow, 0.0, 1.0): r.intersect(x, any_hit=True, outputs=("slot",)),
        "intersect_any_0_1_slot_two_sided": lambda x=bihrt.interval_rays(shadow, 0.0, 1.0):
            r.intersect(x, any_hit=True, two_sided=True, outputs=("slot",)),
    }

    r.load_models(sphere).build()
    yield "sphere_1m_primary_two_sided", prim6, {
        "intersect_all": lambda x=bihrt.interval_rays(prim6): r.intersect(x, outputs=ALL),
        "intersect_all_two_sided": lambda x=bihrt.interval_rays(prim6): r.intersect(x, two_sided=True, outputs=ALL),
    }
    inside = torch.from_numpy(scenes.camera_rays(scenes.pinhole_camera(origin=(0.03, -0.02, 0.05), half=0.9, aspect=w / h), w, h)).cuda()
    yield "sphere_1m_inside_two_sided", inside, {
        "intersect_all_two_sided": lambda x=bihrt.interval_rays(inside): r.intersect(x, two_sided=True, outputs=ALL),
    }


def hit_frac(v):
    s = v["slot"] if isinstance(v, dict) else v[1] if isinstance(v, tuple) else v
    return (s >= 0).float().mean().item()


def agree(name, res):
    """The arms report the same hits: closest-hit arms the same (t, slot, prim), occlusion arms the same hit / miss.
    Two-sided workloads: every hit of the one-sided arm is a hit of the two-sided arm, with t <= (closest hit)."""
    import torch
    vals = list(res.values())
    if name.endswith("_two_sided"):
        if len(vals) == 1:
            return True
        one, two = vals
        h1 = one["slot"] >= 0
        ok = bool((two["slot"][h1] >= 0).all())
        return ok and ("t" not in one or bool((two["t"][h1] <= one["t"][h1]).all()))
    if name == "atrium_shadow":
        a, b = vals
        return bool(torch.equal(a >= 0, b["slot"] >= 0))
    ref = vals[0]
    for v in vals[1:]:
        if not (torch.equal(ref[0], v["t"]) and torch.equal(ref[1], v["slot"]) and torch.equal(ref[2], v["prim"])):
            return False
    return True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--reps", type=int, default=200, help="timed calls per run and arm")
    ap.add_argument("--warmup", type=int, default=5, help="untimed calls before each timed window")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import bihrt
    if not torch.cuda.is_available():
        sys.exit("bench_intersect: no CUDA device (there is no CPU fallback)")
    r = bihrt.Renderer(0)
    r.set_stream(torch.cuda.current_stream().cuda_stream)       # events and library calls on one stream
    res = {"gpu": gpu_info(), "l2_flushed": False, "reps": a.reps, "warmup": a.warmup, "workloads": {}}
    for name, rays, arms in workloads(r):
        n = rays.shape[0]
        ms = {k: [] for k in arms}
        order = list(arms)
        for i in range(a.runs):
            for arm in (order if i % 2 == 0 else order[::-1]):      # alternate which arm goes first
                ms[arm].append(time_ms(arms[arm], a.reps, a.warmup))
        results = {arm: arms[arm]() for arm in order}
        torch.cuda.synchronize()
        s = {arm: {"ms": summary(ms[arm]), "mrays_s_median": n / (summary(ms[arm])["median"] * 1e-3) / 1e6,
                   "hit_frac": hit_frac(results[arm])} for arm in order}
        base = s[order[0]]["ms"]["median"]
        for arm in order:
            s[arm]["time_vs_" + order[0]] = s[arm]["ms"]["median"] / base - 1.0
        res["workloads"][name] = {"rays": int(n), "arms": s, "same_hits": agree(name, results)}
        print(name, json.dumps({k: (round(v["ms"]["median"], 4), round(v["ms"]["spread_frac"], 4), round(v["time_vs_" + order[0]], 4),
                                    round(v["mrays_s_median"], 1), round(v["hit_frac"], 4))
                                for k, v in s.items()}), "same_hits", res["workloads"][name]["same_hits"], flush=True)
    r.close()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
