"""A/B of two builds of libbihrt.so on one GPU: the library a change starts from against the one it produces.

    python tools/ab_libs.py OLD.so NEW.so --runs 5 --out ab_libs.json

The two libraries alternate run by run (BIHRT_LIB picks the library of each child process; which arm goes first
alternates too).  Every run of an arm measures:
  * bench.py --no-extras (the flagship: 1 M triangles, 3840x2160 x 16 spp): value, frame_crc32, oracle tile check, and the
    roofline's per-ray counts and SIMD efficiencies (instrumented kernel);
  * renders at 1920x1080 (L2 not flushed): the 1 M-triangle sphere and the atrium at 1 spp (1 spp warps span 8x4 pixels),
    the bench's 60-frame orbit around the sphere at 1 spp, the atrium at 4 spp jittered (the smallest pixel groups that
    walk in their ray octant), and the atrium at 4 spp jittered on a quality-mode tree (morton_bits = 63);
  * per-sample hit records at 1920x1080 (bihrt_render_hits, outputs copied to the host): the 1 M-triangle sphere at
    1 spp and the atrium at 4 spp jittered;
  * ray lists, device-resident and timed with CUDA events (tools/bench_intersect.py builds them): the atrium's diffuse
    bounce list through bihrt_trace, its shadow list through bihrt_trace_any, and the sphere's 1920x1080 primary list
    through bihrt_intersect with all outputs, one- and two-sided.
Each workload also reports a CRC32 of its outputs (frames, or every output array of a list), which must be the same in
both arms.  Prints one JSON document (per-run values, median and spread per arm, the GPU's name, power limit and max SM
clock); --out also writes it.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
import zlib

from bench_intersect import ALL, atrium_lists, gpu_info, sphere_primary_list, summary, time_ms

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "bih-gpu-raytracer_b200")
W, H = 1920, 1080


def last_json(text):
    for line in reversed(text.splitlines()):
        if line.startswith("{"):
            return json.loads(line)
    raise RuntimeError("no JSON line in:\n" + text[-2000:])


def orbit_cameras(scenes, w, h, frames=60):
    """bench.py's moving_camera views: 6 degrees per frame around the mesh."""
    import numpy as np
    return [scenes.look_at_camera((3.0 * np.sin(2 * np.pi * k / frames) + 0.1, 0.2, -3.0 * np.cos(2 * np.pi * k / frames)),
                                  (0.0, 0.0, 0.0), 0.45, w / h) for k in range(frames)]


def render_timing(r, cams, spp, reps):
    """ms per W x H render (cycling through cams) and a CRC of one frame per camera."""
    import numpy as np
    for k in range(max(20, len(cams))):                      # warm-up; also gives the cost-ordered tile schedule its history
        r.render(cams[k % len(cams)], W, H, spp=spp, jitter=spp > 1)
    r.sync()
    n = max(len(cams), (reps // spp // len(cams)) * len(cams))
    t0 = time.perf_counter()
    for k in range(n):
        r.render(cams[k % len(cams)], W, H, spp=spp, jitter=spp > 1)
    r.sync()
    ms = (time.perf_counter() - t0) * 1e3 / n
    crc = 0
    for c in cams:
        crc = zlib.crc32(np.ascontiguousarray(r.render(c, W, H, spp=spp, jitter=spp > 1).framebuffer()).tobytes(), crc)
    return {"ms": ms, "mrays_s": W * H * spp / (ms * 1e-3) / 1e6, "crc32": "%08x" % crc}


def hits_timing(r, cam, spp, reps):
    """ms per W x H render_hits call (per-sample t, slot, prim copied to the host; jittered at spp > 1) and a CRC of them."""
    import numpy as np
    for _ in range(20):                                      # warm-up, and the tile schedule's history
        r.render_hits(cam, W, H, spp=spp, jitter=spp > 1)
    n = max(1, reps // spp)
    t0 = time.perf_counter()
    for _ in range(n):
        out = r.render_hits(cam, W, H, spp=spp, jitter=spp > 1)
    ms = (time.perf_counter() - t0) * 1e3 / n
    crc = 0
    for x in out:
        crc = zlib.crc32(np.ascontiguousarray(x).tobytes(), crc)
    return {"ms": ms, "mrays_s": W * H * spp / (ms * 1e-3) / 1e6, "crc32": "%08x" % crc}


def list_timing(fn, nrays, reps):
    """ms per call of a ray-list query (CUDA events) and a CRC of all its outputs."""
    import torch
    ms = time_ms(fn, reps, 5)
    out = fn()
    arrays = out.values() if isinstance(out, dict) else out if isinstance(out, tuple) else (out,)
    crc = 0
    for x in arrays:
        crc = zlib.crc32(x.cpu().numpy().tobytes(), crc)
    torch.cuda.synchronize()
    return {"ms": ms, "mrays_s": nrays / (ms * 1e-3) / 1e6, "crc32": "%08x" % crc}


def timing(reps):
    """Child process (BIHRT_LIB picks the library): every workload but the bench, one JSON line."""
    sys.path[:0] = [ROOT, PKG]
    import torch
    import bihrt
    from bihrt import scenes
    r = bihrt.Renderer(0)
    r.set_stream(torch.cuda.current_stream().cuda_stream)       # CUDA events and library calls on one stream
    out = {"lib": bihrt.load_library()._name}
    sphere = scenes.displaced_sphere(scenes.SPHERE_NSEG["1m"])
    atrium = scenes.atrium()
    atrium_cam = [scenes.atrium_camera(W / H)]

    r.load_models(sphere).build()
    out["sphere_1m_1080p_1spp"] = render_timing(r, [scenes.pinhole_camera(aspect=W / H)], 1, reps)
    out["orbit_1m_1080p_1spp"] = render_timing(r, orbit_cameras(scenes, W, H), 1, reps)
    out["sphere_1m_1080p_1spp_render_hits"] = hits_timing(r, scenes.pinhole_camera(aspect=W / H), 1, reps)
    prim = bihrt.interval_rays(sphere_primary_list(W, H))
    n = prim.shape[0]
    out["sphere_1m_primary_intersect_all"] = list_timing(lambda: r.intersect(prim, outputs=ALL), n, reps)
    out["sphere_1m_primary_intersect_all_two_sided"] = list_timing(lambda: r.intersect(prim, two_sided=True, outputs=ALL), n, reps)

    r.load_models(atrium).build()
    out["atrium_1080p_1spp"] = render_timing(r, atrium_cam, 1, reps)
    out["atrium_1080p_4spp"] = render_timing(r, atrium_cam, 4, reps)
    out["atrium_1080p_4spp_render_hits"] = hits_timing(r, atrium_cam[0], 4, reps)
    shadow, diffuse = atrium_lists(r, W, H)
    out["atrium_diffuse_trace"] = list_timing(lambda: r.trace(diffuse), diffuse.shape[0], reps)
    out["atrium_shadow_trace_any"] = list_timing(lambda: r.trace_any(shadow, tmax=1.0), shadow.shape[0], reps)

    r.set_option("morton_bits", 63)
    r.load_models(atrium).build()
    out["atrium_quality_1080p_4spp"] = render_timing(r, atrium_cam, 4, reps)
    r.close()
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old", nargs="?", help="library the change starts from")
    ap.add_argument("new", nargs="?", help="library the change produces")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=300, help="calls per timing (renders: a quarter of them at 4 spp)")
    ap.add_argument("--out", default=None)
    ap.add_argument("--timing", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.timing:
        return timing(a.reps)
    if not (a.old and a.new):
        ap.error("two libraries are needed: OLD.so NEW.so")
    arms = {"old": os.path.abspath(a.old), "new": os.path.abspath(a.new)}
    for lib in arms.values():
        if not os.path.exists(lib):
            sys.exit("%s does not exist" % lib)
    tmp = tempfile.mkdtemp(prefix="ab_libs_")
    res = {"gpu": gpu_info(), "arms": arms, "bench": {k: [] for k in arms}, "timing": {k: [] for k in arms}}
    order = list(arms)
    for i in range(a.runs):
        for arm in (order if i % 2 == 0 else order[::-1]):       # alternate which arm goes first
            env = dict(os.environ, BIHRT_LIB=arms[arm])
            p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(a.steps),
                                "--warmup", str(a.warmup), "--no-extras"], env=env, cwd=tmp, capture_output=True, text=True)
            if p.returncode:
                sys.exit("bench.py failed (%s):\n%s" % (arm, p.stderr[-3000:]))
            j = last_json(p.stdout)
            roof = j.get("roofline") or {}
            res["bench"][arm].append({"value": j["value"], "frame_crc32": j.get("frame_crc32"),
                                      "oracle_tile_check_equal": (j.get("oracle_tile_check") or {}).get("equal"),
                                      "roofline": {k: roof.get(k) for k in ("nodes_per_ray", "tris_per_ray", "lanes_active",
                                                                                  "simd_efficiency_node_phase", "simd_efficiency_leaf_phase")}})
            print(arm, "bench", j["value"], j.get("frame_crc32"), flush=True)
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--timing", "--reps", str(a.reps)], env=env,
                               cwd=tmp, capture_output=True, text=True)
            if p.returncode:
                sys.exit("timing failed (%s):\n%s" % (arm, p.stderr[-3000:]))
            res["timing"][arm].append(last_json(p.stdout))
            print(arm, "timing", json.dumps(res["timing"][arm][-1]), flush=True)
    s = {}
    for arm in arms:
        b = res["bench"][arm]
        s[arm] = {"bench": {"mrays_s": summary([x["value"] for x in b]), "crc32": sorted({str(x["frame_crc32"]) for x in b}),
                            "oracle_tile_check_equal": all(x["oracle_tile_check_equal"] for x in b),
                            "roofline": sorted({json.dumps(x["roofline"], sort_keys=True) for x in b})}}
        for key in res["timing"][arm][0]:
            if key != "lib":
                t = res["timing"][arm]
                s[arm][key] = {"mrays_s": summary([x[key]["mrays_s"] for x in t]), "crc32": sorted({x[key]["crc32"] for x in t})}
    new, old = s["new"], s["old"]
    res["summary"] = s
    res["change"] = {k: new[k]["mrays_s"]["median"] / old[k]["mrays_s"]["median"] - 1.0 for k in new}
    # a workload is slower when its median loses more than both arms' spreads together, or 0.5 %, whichever is larger
    res["slower"] = [k for k in new if -res["change"][k] > max(0.005, new[k]["mrays_s"]["spread_frac"] + old[k]["mrays_s"]["spread_frac"])]
    res["same_outputs"] = all(new[k]["crc32"] == old[k]["crc32"] and len(new[k]["crc32"]) == 1 for k in new) and \
        new["bench"]["roofline"] == old["bench"]["roofline"]
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
