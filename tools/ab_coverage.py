"""A/B of the coverage exit of the framebuffer kernel (csrc/trace.cu, TRACE_COVERAGE_EXIT) on one GPU.

Builds the library with -DTRACE_COVERAGE_EXIT=0 (every sample searches for its closest hit, the behaviour before the exit)
into a temporary directory, then alternates the two libraries (BIHRT_LIB) run by run:
  * bench.py --no-extras (the flagship: 1 M triangles, 3840x2160 x 16 spp): value, frame_crc32, oracle tile check;
  * Renderer.render of the 1 M-triangle sphere and of the atrium at 1920x1080 x 1 spp (L2 not flushed), so that a loss
    away from the flagship shape shows too.
Prints one JSON document (per-run values, median and spread per arm, the GPU's name and power limit); --out also writes it.

    python tools/ab_coverage.py --runs 5 --out ab_coverage.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "bih-gpu-raytracer_b200")


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True)
    except OSError as ex:
        return "unknown (%s)" % ex
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi: %d)" % q.returncode


def last_json(text):
    for line in reversed(text.splitlines()):
        if line.startswith("{"):
            return json.loads(line)
    raise RuntimeError("no JSON line in:\n" + text[-2000:])


def timing(reps):
    """Child process (BIHRT_LIB picks the library): ms per Renderer.render at 1920x1080 x 1 spp, and the frame's CRC."""
    sys.path[:0] = [ROOT, PKG]
    import numpy as np
    import bihrt
    from bihrt import scenes
    r = bihrt.Renderer(0)
    out = {"lib": bihrt.load_library()._name}
    for key, tri, cam in (("sphere_1m_1080p_1spp", scenes.displaced_sphere(scenes.SPHERE_NSEG["1m"]), scenes.pinhole_camera(aspect=1920 / 1080)),
                          ("atrium_1080p_1spp", scenes.atrium(), scenes.atrium_camera(1920 / 1080))):
        r.load_models(tri).build()
        for _ in range(20):                                  # warm-up; also gives the cost-ordered tile schedule its history
            r.render(cam, 1920, 1080, spp=1)
        r.sync()
        t0 = time.perf_counter()
        for _ in range(reps):
            r.render(cam, 1920, 1080, spp=1)
        r.sync()
        ms = (time.perf_counter() - t0) * 1e3 / reps
        fb = np.ascontiguousarray(r.framebuffer())
        out[key] = {"ms": ms, "mrays_s": 1920 * 1080 / (ms * 1e-3) / 1e6, "frame_crc32": "%08x" % zlib.crc32(fb.tobytes())}
    r.close()
    print(json.dumps(out))


def summary(xs):
    xs = sorted(xs)
    med = xs[len(xs) // 2] if len(xs) % 2 else 0.5 * (xs[len(xs) // 2 - 1] + xs[len(xs) // 2])
    return {"runs": xs, "median": med, "min": xs[0], "max": xs[-1], "spread_frac": (xs[-1] - xs[0]) / med}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=300, help="renders per 1080p timing")
    ap.add_argument("--out", default=None)
    ap.add_argument("--timing", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.timing:
        return timing(a.reps)
    shipped = os.path.join(PKG, "libbihrt.so")
    if not os.path.exists(shipped):
        sys.exit("%s not built (make -C %s)" % (shipped, PKG))
    tmp = tempfile.mkdtemp(prefix="ab_coverage_")
    variant = os.path.join(tmp, "libbihrt_cov0.so")
    subprocess.check_call(["make", "-s", "-C", PKG, "variant", "EXTRA=-DTRACE_COVERAGE_EXIT=0", "LIB=" + variant])
    arms = {"coverage_exit": shipped, "closest_hit": variant}
    res = {"gpu": gpu_info(), "arms": arms, "bench": {k: [] for k in arms}, "render_1080p": {k: [] for k in arms}}
    order = list(arms)
    for i in range(a.runs):
        for arm in (order if i % 2 == 0 else order[::-1]):       # alternate which arm goes first
            env = dict(os.environ, BIHRT_LIB=arms[arm])
            p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(a.steps),
                                "--warmup", str(a.warmup), "--no-extras"], env=env, cwd=tmp, capture_output=True, text=True)
            if p.returncode:
                sys.exit("bench.py failed (%s):\n%s" % (arm, p.stderr[-3000:]))
            j = last_json(p.stdout)
            res["bench"][arm].append({"value": j["value"], "frame_crc32": j.get("frame_crc32"),
                                      "oracle_tile_check_equal": (j.get("oracle_tile_check") or {}).get("equal")})
            print(arm, "bench", j["value"], j.get("frame_crc32"), flush=True)
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--timing", "--reps", str(a.reps)], env=env,
                               cwd=tmp, capture_output=True, text=True)
            if p.returncode:
                sys.exit("timing failed (%s):\n%s" % (arm, p.stderr[-3000:]))
            res["render_1080p"][arm].append(last_json(p.stdout))
            print(arm, "1080p", res["render_1080p"][arm][-1], flush=True)
    s = {}
    for arm in arms:
        s[arm] = {"bench_value_mrays_s": summary([x["value"] for x in res["bench"][arm]]),
                  "frame_crc32": sorted({x["frame_crc32"] for x in res["bench"][arm]}),
                  "oracle_tile_check_equal": all(x["oracle_tile_check_equal"] for x in res["bench"][arm])}
        for key in ("sphere_1m_1080p_1spp", "atrium_1080p_1spp"):
            s[arm][key + "_mrays_s"] = summary([x[key]["mrays_s"] for x in res["render_1080p"][arm]])
            s[arm][key + "_frame_crc32"] = sorted({x[key]["frame_crc32"] for x in res["render_1080p"][arm]})
    new, old = s["coverage_exit"], s["closest_hit"]
    res["summary"] = s
    res["gain"] = {k: new[k]["median"] / old[k]["median"] - 1.0 for k in new if k.endswith("_mrays_s")}
    res["same_frames"] = all(new[k] == old[k] for k in new if k.endswith("crc32"))
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
