"""A/B of the octant copies of the framebuffer kernel's node phase (csrc/trace.cu, TRACE_OCTANT_WALK) on one GPU.

Builds the library with -DTRACE_OCTANT_WALK=0 (the generic node phase only, the behaviour before the copies) into a
temporary directory, then alternates the two libraries (BIHRT_LIB) run by run:
  * bench.py --no-extras (the flagship: 1 M triangles, 3840x2160 x 16 spp): value, frame_crc32, oracle tile check;
  * Renderer.render of the 1 M-triangle sphere and of the atrium at 1920x1080 x 1 spp (L2 not flushed): 1 spp warps span
    8x4 pixels, and inside the atrium mixed-sign warps are common;
  * the bench's 60-frame orbit around the 1 M-triangle sphere at 1920x1080 x 1 spp, whose views hold other octants;
  * the atrium at 1920x1080 x 4 spp jittered: warps of 8 pixels x 4 samples, the smallest pixel groups that take the
    octant copies.
Prints one JSON document (per-run values, median and spread per arm, the GPU's name, power limit and max SM clock);
--out also writes it.

    python tools/ab_octant.py --runs 5 --out ab_octant.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
import zlib

from ab_coverage import gpu_info, last_json, summary

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "bih-gpu-raytracer_b200")
KEYS = ("sphere_1m_1080p_1spp", "atrium_1080p_1spp", "orbit_1m_1080p_1spp", "atrium_1080p_4spp")


def orbit_cameras(scenes, w, h, frames=60):
    """bench.py's moving_camera views: 6 degrees per frame around the mesh."""
    import numpy as np
    return [scenes.look_at_camera((3.0 * np.sin(2 * np.pi * k / frames) + 0.1, 0.2, -3.0 * np.cos(2 * np.pi * k / frames)),
                                  (0.0, 0.0, 0.0), 0.45, w / h) for k in range(frames)]


def timing(reps):
    """Child process (BIHRT_LIB picks the library): ms per 1920x1080 render of each workload, and a CRC of its frames."""
    sys.path[:0] = [ROOT, PKG]
    import numpy as np
    import bihrt
    from bihrt import scenes
    r = bihrt.Renderer(0)
    out = {"lib": bihrt.load_library()._name}
    W, H = 1920, 1080
    sphere = scenes.displaced_sphere(scenes.SPHERE_NSEG["1m"])
    atrium = scenes.atrium()
    for key, tri, cams, spp in ((KEYS[0], sphere, [scenes.pinhole_camera(aspect=W / H)], 1),
                                (KEYS[1], atrium, [scenes.atrium_camera(W / H)], 1),
                                (KEYS[2], sphere, orbit_cameras(scenes, W, H), 1),
                                (KEYS[3], atrium, [scenes.atrium_camera(W / H)], 4)):
        r.load_models(tri).build()
        for k in range(max(20, len(cams))):                  # warm-up; also gives the cost-ordered tile schedule its history
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
        out[key] = {"ms": ms, "mrays_s": W * H * spp / (ms * 1e-3) / 1e6, "frame_crc32": "%08x" % crc}
    r.close()
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=300, help="renders per 1080p x 1 spp timing (a quarter of them at 4 spp)")
    ap.add_argument("--out", default=None)
    ap.add_argument("--timing", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.timing:
        return timing(a.reps)
    shipped = os.path.join(PKG, "libbihrt.so")
    if not os.path.exists(shipped):
        sys.exit("%s not built (make -C %s)" % (shipped, PKG))
    tmp = tempfile.mkdtemp(prefix="ab_octant_")
    variant = os.path.join(tmp, "libbihrt_oct0.so")
    subprocess.check_call(["make", "-s", "-C", PKG, "variant", "EXTRA=-DTRACE_OCTANT_WALK=0", "LIB=" + variant])
    arms = {"octant_walk": shipped, "generic_walk": variant}
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
        for key in KEYS:
            s[arm][key + "_mrays_s"] = summary([x[key]["mrays_s"] for x in res["render_1080p"][arm]])
            s[arm][key + "_frame_crc32"] = sorted({x[key]["frame_crc32"] for x in res["render_1080p"][arm]})
    new, old = s["octant_walk"], s["generic_walk"]
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
