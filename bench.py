#!/usr/bin/env python
"""bench.py -- Mrays/s (and BIH build ms/Mtri) of the BIH hot path on N B200s of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
  python bench.py --impl reference [--gpus N] ...                # the reference algorithm on host cores
  python bench.py ... --dump-outputs DIR                         # also save the last timed frame as DIR/framebuffer.npy

Workload (config.workload): the 1 002 528-triangle displaced sphere of BASELINE config 5 (the scene
the north star's 70 % target is quoted on) seen by the config-2 camera, traced with config 4's ray
load: 3840x2160 pixels x 16 jittered primary rays = 132 710 400 rays per step.  A step = one frame's
trace with the BIH resident in HBM.  At N > 1 the frame's rays are partitioned over the ranks (strong
scaling: total work fixed) by unit interleave (every rank walks every tile and owns every N-th run of
32-ray units, i.e. a few neighbouring pixels with all their samples); the BIH built on rank 0 is
replicated by one NCCL broadcast before the timed region; the gather is fused into the trace kernel:
every rank stores the final colour of its pixels straight into rank 0's framebuffer (CUDA IPC mapping,
NVLink) and a one-element all-reduce closes the frame (BIHRT_BENCH_SHARD=interleave|samples|tiles select
the NCCL-reduce variants instead).

`value`  = rays of the whole frame / max-over-ranks device time (CUDA events on the launching stream).
`e2e`    = the same metric for the reference's full per-frame sequence through the C ABI with HOST
           buffers: vertices H2D from pinned memory (the reference rebuilds every frame,
           R/src/Renderer.cpp:415-503) -> bihrt_build -> [broadcast] -> bihrt_render -> [reduce] ->
           framebuffer D2H to pinned memory.
One JSON line on stdout (rank 0); everything else goes to stderr.
"""
import argparse
import json
import os
import subprocess
import sys
import hashlib
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "bih-gpu-raytracer_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "Mrays/s"
L2_FLUSH_BYTES = 256 << 20          # > 126 MB L2
NODE_BYTES = 64                     # one node record: the BIH pair of clip planes + child references (16 B) and the two children boxes (48 B)
DUMP_BYTES = 64 << 20               # --dump-outputs: at most this much in all


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# Exactly ONE line may reach stdout.  Libraries (NCCL prints its version banner there) write to fd 1
# directly, so fd 1 is pointed at stderr for the whole run and the JSON line goes to a saved copy.
_REAL_STDOUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(obj):
    _REAL_STDOUT.write(json.dumps(obj) + "\n")
    _REAL_STDOUT.flush()


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def host_cores():
    """Host threads this process may use.  NOT omp_get_max_threads(): torch.distributed.run exports
    OMP_NUM_THREADS=1 to its children, which would time the CPU arm on one core and call it all of them."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def crc32(a):
    return "%08x" % (zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF)


def kernel_source_sha():
    """Hash of the trace kernel's CODE (comments and blank lines stripped): ncu-derived counters in profiles/ are only quoted
    for the kernel they were captured on (profiles/trace_counters.json records the hash at capture time)."""
    import re
    h = hashlib.sha256()
    for f in ("csrc/trace.cu", "csrc/bihrt_internal.cuh"):
        src = open(os.path.join(ROOT, "bih-gpu-raytracer_b200", f)).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        src = "\n".join(l.split("//")[0].rstrip() for l in src.splitlines())
        src = "\n".join(l for l in src.splitlines() if l.strip())
        h.update(src.encode())
    return h.hexdigest()[:16]


def ncu_counters(workload_key):
    """ncu counters of the trace kernel on a named workload, from the committed capture -- or None when the kernel
    source has changed since (stale numbers are not quoted)."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "trace_counters.json")))
        e = d["captures"][workload_key]
        if d.get("kernel_source_sha") != kernel_source_sha():
            return {"stale": "profiles/trace_counters.json was captured on another version of the kernel (%s != %s)" % (
                d.get("kernel_source_sha"), kernel_source_sha())}
        return e
    except Exception as ex:       # noqa
        return {"stale": "no capture: %r" % (ex,)}


def dump_outputs(path, **arrays):
    """--dump-outputs: the arrays the timed path returned in its last step, one <path>/<name>.npy each, so that two
    builds of the project can be compared output for output.  Values are stored as float32 (the framebuffer's packed
    r | g<<8 | b<<16 pixels are below 2**24 and therefore exact).  The files take at most DUMP_BYTES in all: each array
    gets an equal share, and one larger than its share is replaced by a fixed, seeded sample of its elements,
    <name>_sample.npy, with their flat indices in <name>_sample_index.npy."""
    os.makedirs(path, exist_ok=True)
    share = DUMP_BYTES // len(arrays) - 2 * 4096          # (room for the .npy headers)
    for name, a in arrays.items():
        a = np.asarray(a)
        assert np.all(np.asarray(a, np.float32) == a), name + " is not exact in float32"
        a = a.astype(np.float32)
        if a.nbytes <= share:
            np.save(os.path.join(path, name + ".npy"), a)
            continue
        idx = np.sort(np.random.default_rng(1984).choice(a.size, share // 12, replace=False))
        np.save(os.path.join(path, name + "_sample.npy"), a.ravel()[idx])
        np.save(os.path.join(path, name + "_sample_index.npy"), idx.astype(np.float64))
    log("outputs of the last timed step written to %s: %s" % (path, ", ".join(sorted(os.listdir(path)))))


def oracle_tile_check(fb, tri_or_bih, cam, W, H, spp, tiles=12, seed=1984):
    """A third party's check of the frame the bench just timed: the literal reference traversal (oracle, CPU) of every
    jittered sample of a few 32x32-pixel tiles spread over the frame (centre, silhouette, background), packed like
    cudaRender does, against the same windows of the GPU framebuffer."""
    from oracle import oracle as O
    ob = tri_or_bih if isinstance(tri_or_bih, O.Bih) else O.Bih(tri_or_bih)
    tx, ty = (W + 31) // 32, (H + 31) // 32
    picks, k = [], 0
    while len(picks) < tiles:
        # a low-discrepancy walk over the tile grid, biased to the middle band where the mesh is
        fx = (0.5 + 0.61803398875 * k) % 1.0
        fy = 0.5 + ((0.5 + 0.75487766625 * k) % 1.0 - 0.5) * 0.7
        t = (min(tx - 1, int(fx * tx)), min(ty - 1, int(fy * ty)))
        if t not in picks:
            picks.append(t)
        k += 1
    ok, pix, hit_pix = True, 0, 0
    gpu_crc, orc_crc = 0, 0
    for (i, j) in picks:
        x0, y0 = i * 32, j * 32
        ww, wh = min(32, W - x0), min(32, H - y0)
        rays = O.camera_rays_window(cam, W, H, x0, y0, ww, wh, spp=spp, jitter=True, seed=seed)
        _, slot, _ = ob.trace(rays, "ref", threads=host_cores())
        want = O.pack_framebuffer(slot, ww, wh, spp).reshape(wh, ww)
        got = np.ascontiguousarray(fb[y0:y0 + wh, x0:x0 + ww]).astype(np.uint32)
        ok = ok and bool(np.array_equal(want, got))
        pix += ww * wh
        hit_pix += int((slot.reshape(-1, spp) >= 0).any(axis=1).sum())
        gpu_crc = zlib.crc32(got.tobytes(), gpu_crc)
        orc_crc = zlib.crc32(want.tobytes(), orc_crc)
    return {"equal": ok, "tiles": len(picks), "pixels": pix, "rays": pix * spp, "pixels_with_a_hit": hit_pix,
            "crc32_gpu_tiles": "%08x" % gpu_crc, "crc32_oracle_tiles": "%08x" % orc_crc,
            "what": "literal TraverseTree (oracle/bih_oracle.c, CPU) on every jittered sample of %d 32x32-pixel tiles of the timed frame, "
                    "packed like cudaRender, vs the same windows of the GPU framebuffer" % len(picks)}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.lines, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for l in self.proc.stdout:
            self.lines.append((time.time(), l.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ts, l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 6 or not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def workload(args):
    from bihrt import scenes
    nseg = scenes.SPHERE_NSEG[args.scene]
    cam = scenes.pinhole_camera(aspect=args.width / args.height)
    name = ("%s-triangle displaced sphere (nseg=%d, BASELINE config 5 scene), config-2 pinhole camera, %dx%d x %d spp "
            "jittered primary rays (config 4 ray load)" % (args.scene, nseg, args.width, args.height, args.spp))
    return nseg, cam, name


# ---------------------------------------------------------------------------------------------
# reference arm: the reference's algorithm (oracle port) on the box's host cores
# ---------------------------------------------------------------------------------------------
def cpu_sample(args, div):
    """Bounded sample of the workload's rays: the same camera at 1/div resolution, pixel centres."""
    return max(args.width // div, 1), max(args.height // div, 1)


def run_reference(args, rank):
    if rank != 0:
        return
    from bihrt import scenes
    from oracle import oracle as O
    nseg, cam, name = workload(args)
    tri = scenes.displaced_sphere(nseg)
    t0 = time.perf_counter()
    ob = O.Bih(tri)
    build_s = time.perf_counter() - t0
    w, h = cpu_sample(args, 8)
    rays = O.camera_rays(cam, w, h)
    cores = host_cores()                      # explicit: OMP_NUM_THREADS=1 under torch.distributed.run must not shrink the arm
    for _ in range(args.warmup):
        ob.trace(rays, "ref", threads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ob.trace(rays, "ref", threads=cores)
    dt = time.perf_counter() - t0
    val = len(rays) * args.steps / dt / 1e6
    # one-thread figure on a smaller sample of the same rays (every 16th)
    r1 = np.ascontiguousarray(rays[::16])
    t0 = time.perf_counter()
    ob.trace(r1, "ref", threads=1)
    val_1t = len(r1) / (time.perf_counter() - t0) / 1e6
    sample = ("%dx%d pixel-centre rays of the same camera per step (1/64 of one sample per pixel of the frame), literal "
              "TraverseTree semantics, OpenMP over %d threads; BIH build single-threaded %.1f ms/Mtri" % (
                  w, h, cores, build_s * 1e3 / (len(tri) / 1e6)))
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": name, "note": "CPU restatement of the reference's GPU algorithm (the reference has no CPU path; "
                      "oracle/bih_oracle.c); bounded sample per step"},
           "cpu_baseline": {"value": val, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample,
                            "one_thread_mrays_s": val_1t, "omp_num_threads_env": os.environ.get("OMP_NUM_THREADS"),
                            "build_ms_per_mtri": build_s * 1e3 / (len(tri) / 1e6)},
           "e2e": {"value": val, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    emit(out)


# ---------------------------------------------------------------------------------------------
# this repo's arm
# ---------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch
    import bihrt
    from bihrt import multi, scenes

    dist = None
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.Stream(device=dev)
    r = bihrt.Renderer(device=local_rank, stream=stream.cuda_stream)
    nseg, cam, name = workload(args)
    W, H, spp = args.width, args.height, args.spp
    rays_total = W * H * spp

    # every rank owns a pinned copy of the vertices: the e2e frame uploads them over the rank's own PCIe link
    tri = scenes.displaced_sphere(nseg)
    n_tri = 2 * nseg * nseg
    pinned_tri = torch.from_numpy(tri).pin_memory()
    if rank == 0:
        r.load_models(pinned_tri)
        r.build()
        r.sync()
    with torch.cuda.stream(stream):
        if world > 1:
            multi.replicate_bih_inplace(r, dist, n_tri, src=0)
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    fb_t = None

    # N > 1: unit interleave (every rank walks every tile and owns every N-th 32-ray unit of it: balanced, and a
    # pixel keeps all its samples in consecutive lanes); samples / tiles per rank are the fall-backs
    mode = os.environ.get("BIHRT_BENCH_SHARD", "p2p") if world > 1 else "single"
    if mode in ("p2p", "interleave") and (32 * (spp & -spp if spp & -spp < 32 else 32)) % world != 0:
        mode = "samples"
    # p2p = unit interleave with the gather fused into the trace kernel: every rank stores its finished pixels
    # straight into rank 0's framebuffer (CUDA IPC mapping, NVLink); a one-element all-reduce closes the frame.
    # The shared framebuffer holds TWO frames (w x 2h): the pipelined e2e loop renders frame k into half k % 2 while
    # half (k-1) % 2 is still being copied to the host.
    peer_ptr, peer_opened, token = None, False, None
    if mode == "p2p":
        try:
            with torch.cuda.stream(stream):
                peer_ptr, peer_opened = multi.open_peer_framebuffer(r, dist, W, 2 * H, dst=0, device=dev)
                token = torch.zeros(1, dtype=torch.int32, device=dev)
        except Exception as ex:       # noqa  (no peer mapping on this box: NCCL reduce instead)
            log("rank %d: peer framebuffer unavailable (%r); using interleave + reduce" % (rank, ex))
            peer_ptr = None
        ok = torch.tensor([1 if peer_ptr else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            mode = "interleave"
    own_two_frames = None
    if world == 1:
        own_two_frames = torch.empty((2, H, W), dtype=torch.int32, device=dev)     # the e2e pipeline's two frame halves
        peer_ptr = own_two_frames.data_ptr()
    if mode == "samples" and spp < world:
        mode = "tiles"
    by_sample = mode in ("samples", "interleave")        # per-pixel hit counts, resolved after the reduce
    s0, s1 = multi.sample_range(spp, rank, world)
    half_bytes = W * H * 4

    def render_my_share(half=None):
        if world == 1 and half is None:
            r.render(cam, W, H, spp=spp, seed=1984, jitter=True)          # the reference-facing call: frame into the context's framebuffer
        elif world == 1:
            r.render_interleaved_to(cam, W, H, spp, 0, 1, target_ptr=peer_ptr + half * half_bytes, seed=1984, jitter=True)
        elif mode == "p2p":
            half = half or 0
            r.render_interleaved_to(cam, W, H, spp, rank, world, target_ptr=peer_ptr + half * half_bytes, seed=1984, jitter=True)
        elif mode == "interleave":
            r.render_interleaved(cam, W, H, spp, rank, world, seed=1984, jitter=True)
        elif mode == "samples":
            r.render_samples(cam, W, H, spp, s0, s1, seed=1984, jitter=True)
        else:
            r.render(cam, W, H, spp=spp, seed=1984, jitter=True, shard=(rank, world))

    def close_frame():
        nonlocal fb_t
        if mode == "p2p":
            multi.frame_barrier(dist, token)
        elif world > 1:
            if fb_t is None:
                fb_t = multi.framebuffer_tensor(r)
            multi.gather_framebuffer(fb_t, dist, dst=0)
            if by_sample and rank == 0:
                r.framebuffer_resolve(spp)

    def step():
        render_my_share()
        close_frame()

    def timed_loop(fn, k):
        """K steps, L2 flushed (untimed) before each, CUDA events on the launching stream; returns
        this rank's total ms."""
        tot = 0.0
        with torch.cuda.stream(stream):
            for _ in range(k):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                fn()
                e1.record(stream)
                e1.synchronize()
                tot += e0.elapsed_time(e1)
        return tot

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def frame_from_device(half=0):
        """rank 0: the gathered frame as a host (H, W) uint32 array."""
        if mode == "p2p":
            fb2 = torch.as_tensor(multi._CudaView(peer_ptr, (2, H, W), "<i4"), device=dev)
            torch.cuda.synchronize(dev)
            return fb2[half].cpu().numpy().view(np.uint32)
        return r.framebuffer().copy()

    with torch.cuda.stream(stream):
        for _ in range(max(args.warmup, 3)):
            step()
    barrier()
    launches0 = r.get_stat("kernel_launches")
    sampler = ClockSampler(local_rank) if rank == 0 else None
    t_wall0 = time.time()
    ms = timed_loop(step, args.steps)
    barrier()
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    launches = r.get_stat("kernel_launches") - launches0
    ms = max_over_ranks(ms)
    ms_per_step = ms / args.steps
    value = rays_total / (ms_per_step * 1e-3) / 1e6

    # ---- the frame the timed loop produced: CRC32 of rank 0's framebuffer (equal at every N: a reader of the N = 1 and
    # N = 8 lines can compare them) and an oracle check of a sample of its tiles -------------------------------------
    frame_crc, tile_check = None, None
    if rank == 0:
        frame = frame_from_device(0)
        frame_crc = crc32(frame)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, framebuffer=frame)
        try:
            tile_check = oracle_tile_check(frame, tri, cam, W, H, spp)
        except Exception as ex:       # noqa
            tile_check = {"error": repr(ex)[:200]}
    barrier()

    # ---- N > 1: where a step's time goes (diagnostic, separate loop) --------------------------------
    breakdown = None
    if world > 1:
        t_r = max_over_ranks(timed_loop(render_my_share, 3)) / 3
        t_g = max_over_ranks(timed_loop(close_frame, 3)) / 3
        breakdown = {"render_shard_ms_max_over_ranks": t_r, ("frame_barrier_ms" if mode == "p2p" else "framebuffer_reduce_ms"): t_g}
        barrier()

    # ---- N > 1: the gathered frame must be bit-identical to the single-GPU render ------------------
    image_ok, single_crc = None, None
    if world > 1:
        with torch.cuda.stream(stream):
            step()
        barrier()
        if rank == 0:
            multi_fb = frame_from_device(0)
            single_fb = r.render(cam, W, H, spp=spp, seed=1984, jitter=True).framebuffer()
            image_ok = bool(np.array_equal(multi_fb, single_fb))
            single_crc = crc32(single_fb)
        barrier()

    # ---- e2e: the reference's full frame through the public API with HOST buffers -----------------------
    # Every rank uploads the frame's vertices from its own pinned buffer over its own PCIe link and rebuilds locally
    # (the build is deterministic, so the trees are identical and no broadcast is needed: 0.19 ms against 36 MB of
    # NVLink traffic per frame), renders its share into rank 0's frame buffer and rank 0 copies the frame to pinned host
    # memory.  The loop is software-pipelined the way a frame loop is: frame k+1's upload and frame k-1's download run on
    # copy streams while frame k is traced (two vertex buffers, two halves of the shared framebuffer).
    can_pipe = mode in ("single", "p2p")
    if rank != 0:
        r.load_models(pinned_tri)
        r.build()
        r.sync()
    barrier()
    host_fb = [torch.empty((H, W), dtype=torch.int32).pin_memory() for _ in range(2)] if rank == 0 else None
    dev_tri = [torch.empty(pinned_tri.shape, dtype=torch.float32, device=dev) for _ in range(2)]
    copy_in, copy_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def e2e_serial_step():
        r.update_vertices(pinned_tri)                    # H2D, pinned (every rank, own link)
        r.build()
        step()
        if rank == 0:
            if mode == "p2p":
                fb2 = torch.as_tensor(multi._CudaView(peer_ptr, (2, H, W), "<i4"), device=dev)
                host_fb[0].copy_(fb2[0], non_blocking=True)
                stream.synchronize()
            else:
                r.framebuffer(out=host_fb[0])               # D2H, pinned; synchronises

    upload_mode = os.environ.get("BIHRT_BENCH_E2E_UPLOAD", "one")

    def e2e_pipelined(k_frames):
        """k_frames frames through the pipeline; returns this rank's ms (events on the launching stream, the last
        frame's download included)."""
        fb2 = torch.as_tensor(multi._CudaView(peer_ptr, (2, H, W), "<i4"), device=dev) if rank == 0 else None
        ev_in = [torch.cuda.Event() for _ in range(2)]
        ev_free = [torch.cuda.Event() for _ in range(2)]

        ev_rend = [torch.cuda.Event() for _ in range(2)]
        ev_out = [None, None]
        with torch.cuda.stream(stream):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            copy_in.wait_stream(stream)
            copy_out.wait_stream(stream)
            dbg = os.environ.get("BIHRT_BENCH_E2E_DEBUG") and k_frames > 4
            marks, host_t = [], []
            for k in range(k_frames):
                b = k & 1
                if dbg:
                    host_t.append(time.perf_counter())
                    m = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
                    marks.append(m); m[0].record(stream)
                # "one" (default): the frame's vertices cross PCIe ONCE -- rank k % N uploads them over its own link (every link
                # carries one upload every N frames; rank 0's is left to the framebuffer download) and hands them to the others with one
                # 36 MB NCCL broadcast over NVLink on the launching stream (0.24 ms of the 8-GPU frame).  "each": every rank uploads
                # its own copy on its copy stream.  Measured at 8 GPUs (BIHRT_BENCH_E2E_DEBUG=1): the broadcast disappears from the
                # launching stream, but DMA traffic next to the kernels slows them -- build 0.20 -> 0.32 ms, trace 1.47 -> 1.54 ms,
                # rank 0 (download + upload) build 0.64 ms -- and the frame takes 2.26-2.36 ms against 2.11-2.21 with "one".
                # Also measured: the broadcast issued a frame ahead on its own stream and communicator.  The receivers' NCCL kernels
                # then sit on a few SMs until the sender's trace kernel has drained, and the build's cooperative k_front cannot
                # become co-resident next to them: the frame period DOUBLES (2 GPUs: 6.0 -> 11.8 ms).  Left as it was.
                if upload_mode == "each" or rank == k % world:
                    with torch.cuda.stream(copy_in):
                        if k >= 2:
                            copy_in.wait_event(ev_free[b])       # frame k-2's build input has been consumed
                        dev_tri[b].copy_(pinned_tri, non_blocking=True)      # H2D on the copy stream
                        ev_in[b].record(copy_in)
                    stream.wait_event(ev_in[b])
                if world > 1 and upload_mode != "each":
                    dist.broadcast(dev_tri[b], src=k % world)
                r.update_vertices(dev_tri[b])                    # device -> the context's input array (36 MB D2D)
                ev_free[b].record(stream)
                if dbg: marks[-1][1].record(stream)
                r.build()
                if dbg: marks[-1][2].record(stream)
                render_my_share(b)
                if dbg: marks[-1][3].record(stream)
                # peers store into half b of rank 0's buffer: rank 0 joins the barrier of frame k only once its download of
                # frame k-1 is done, so when a peer passes this barrier the half it writes NEXT frame is free
                if rank == 0 and ev_out[b ^ 1] is not None:
                    stream.wait_event(ev_out[b ^ 1])
                if world > 1:
                    multi.frame_barrier(dist, token)
                if dbg: marks[-1][4].record(stream)
                if rank == 0:
                    ev_rend[b].record(stream)
                    with torch.cuda.stream(copy_out):
                        copy_out.wait_event(ev_rend[b])
                        if not os.environ.get("BIHRT_BENCH_E2E_NO_D2H"):
                            host_fb[b].copy_(fb2[b], non_blocking=True)      # D2H on the copy stream
                        ev_out[b] = torch.cuda.Event()
                        ev_out[b].record(copy_out)
            if rank == 0:
                for e in ev_out:
                    if e is not None:
                        stream.wait_event(e)
            e1.record(stream)
            host_end = time.perf_counter()
            e1.synchronize()
            if dbg:
                seg = np.array([[m[i].elapsed_time(m[i + 1]) for i in range(4)] + [marks[j][0].elapsed_time(marks[j + 1][0]) if j + 1 < len(marks) else float('nan')] for j, m in enumerate(marks)])
                log("rank %d e2e pipeline (ms, median over frames): wait+upload->input %.3f  build %.3f  trace %.3f  barrier(+download wait) %.3f  | frame period %.3f | host enqueue per frame %.3f" % (
                    (rank,) + tuple(np.nanmedian(seg, axis=0)) + ((host_end - host_t[0]) / k_frames * 1e3,)))
            return e0.elapsed_time(e1)

    e2e_steps = max(2, min(args.steps, 5))
    with torch.cuda.stream(stream):
        e2e_serial_step()
    barrier()
    ms_e2e_serial = max_over_ranks(timed_loop(e2e_serial_step, e2e_steps)) / e2e_steps
    barrier()
    ms_e2e, e2e_frames, e2e_crc = ms_e2e_serial, e2e_steps, None
    if can_pipe:
        e2e_frames = max(6, 2 * e2e_steps)
        e2e_pipelined(4)
        barrier()
        ms_e2e = max_over_ranks(e2e_pipelined(e2e_frames)) / e2e_frames
        barrier()
        if rank == 0:
            e2e_crc = crc32(host_fb[(e2e_frames - 1) & 1].numpy().view(np.uint32))
    e2e_val = rays_total / (ms_e2e * 1e-3) / 1e6

    # ---- N > 1: BASELINE config 5 at N GPUs: animated 1 M-triangle scene, rebuild + 1080p x 1 spp trace per frame --------
    # (a) rank 0 rebuilds and broadcasts the BIH, (b) every rank rebuilds locally (deterministic build => identical
    # trees, no broadcast); both end with the fused gather into rank 0's framebuffer + frame barrier
    animated = None
    if world > 1 and mode == "p2p" and args.scene == "1m":
        try:
            aw, ah = 1920, 1080
            acam = scenes.pinhole_camera(aspect=aw / ah)
            r.sync()
            barrier()

            def frame_bcast():
                if rank == 0:
                    r.build()
                multi.replicate_bih_inplace(r, dist, n_tri, src=0)
                r.render_interleaved_to(acam, aw, ah, 1, rank, world, target_ptr=peer_ptr, seed=1984, jitter=False)
                multi.frame_barrier(dist, token)

            def frame_local():
                r.build()
                r.render_interleaved_to(acam, aw, ah, 1, rank, world, target_ptr=peer_ptr, seed=1984, jitter=False)
                multi.frame_barrier(dist, token)

            def trace_only():
                r.render_interleaved_to(acam, aw, ah, 1, rank, world, target_ptr=peer_ptr, seed=1984, jitter=False)
                multi.frame_barrier(dist, token)

            res = {}
            for nm, fn in (("frame_ms_bih_broadcast", frame_bcast), ("frame_ms_local_rebuild", frame_local), ("trace_ms", trace_only)):
                with torch.cuda.stream(stream):
                    for _ in range(3):
                        fn()
                barrier()
                res[nm] = max_over_ranks(timed_loop(fn, 5)) / 5
                barrier()
            # the frame of the local-rebuild variant must equal the single-GPU render
            with torch.cuda.stream(stream):
                frame_local()
            barrier()
            if rank == 0:
                fb2 = torch.as_tensor(multi._CudaView(peer_ptr, (2 * H * W,), "<i4"), device=dev)
                torch.cuda.synchronize(dev)
                mfb = fb2[:aw * ah].cpu().numpy().view(np.uint32).reshape(ah, aw)
                sfb = r.render(acam, aw, ah, spp=1, seed=1984, jitter=False).framebuffer()
                res["image_bit_identical_to_single_gpu"] = bool(np.array_equal(mfb, sfb))
                res["frame_crc32"] = crc32(mfb)
                res["single_gpu_frame_crc32"] = crc32(sfb)
                res["what"] = "config 5 at %d GPUs: 1 M triangles rebuilt every frame + 1920x1080 x 1 spp primary rays; max over ranks, L2 flushed" % world
            barrier()
            animated = res
        except Exception as ex:       # noqa
            animated = {"error": repr(ex)[:200]}

    # ---- N > 1: BASELINE config 4 as written: the 10 M-triangle mesh at 3840x2160 x 16 spp over N GPUs, BIH built on
    # rank 0 and replicated by ONE broadcast (640 MB) over NVLink, gather fused into the trace kernel -------------------
    config4 = None
    if world > 1 and mode == "p2p" and not args.no_config4 and (W, H, spp) == (3840, 2160, 16):
        try:
            n10 = 2 * scenes.SPHERE_NSEG["10m"] ** 2
            if rank == 0:
                t10 = scenes.displaced_sphere(scenes.SPHERE_NSEG["10m"])
                r.load_models(torch.from_numpy(t10).to(dev))
                r.build()
                r.sync()
            barrier()

            def bcast10():
                multi.replicate_bih_inplace(r, dist, n10, src=0)

            with torch.cuda.stream(stream):
                bcast10()
            barrier()
            t_b = max_over_ranks(timed_loop(bcast10, 3)) / 3
            barrier()
            with torch.cuda.stream(stream):
                for _ in range(2):
                    step()
            barrier()
            k4 = 3
            t_f = max_over_ranks(timed_loop(step, k4)) / k4
            barrier()
            res = {"triangles": n10, "rays_per_frame": rays_total, "trace_ms_max_over_ranks": t_f,
                   "mrays_s": rays_total / (t_f * 1e-3) / 1e6, "bih_broadcast_ms": t_b,
                   "bih_blob_bytes": 64 + n10 * (NODE_BYTES + 48), "bih_broadcast_gb_s": (64 + n10 * (NODE_BYTES + 48)) / (t_b * 1e-3) / 1e9,
                   "mrays_s_with_one_broadcast_per_frame": rays_total / ((t_f + t_b) * 1e-3) / 1e6,
                   "what": "BASELINE config 4: 9 999 392-triangle mesh, 3840x2160 x 16 spp, unit interleave over %d GPUs, BIH built on rank 0 and "
                           "replicated in place by one NCCL broadcast; L2 flushed; max over ranks" % world}
            if rank == 0:
                mfb = frame_from_device(0)
                res["frame_crc32"] = crc32(mfb)
                sfb = r.render(cam, W, H, spp=spp, seed=1984, jitter=True).framebuffer()
                res["single_gpu_frame_crc32"] = crc32(sfb)
                res["image_bit_identical_to_single_gpu"] = bool(np.array_equal(mfb, sfb))
            barrier()
            config4 = res
        except Exception as ex:       # noqa
            config4 = {"error": repr(ex)[:300]}
        # back to the bench scene on rank 0 (the remaining sections use it)
        if rank == 0:
            r.load_models(pinned_tri)
            r.build()
            r.sync()
        barrier()

    out = None
    if rank == 0:
        peak, peak_src = peaks()
        info = r.build_info()
        # ---- build ms/Mtri (device events), L2 flushed before each build
        r.build(); r.sync()
        tb = []
        for _ in range(max(args.steps, 5)):
            tb.append(timed_loop(lambda: r.build(), 1))
        build_ms = float(np.median(tb))
        # ---- algorithmic bytes per ray for the roofline (SURVEY.md 8(d), DESIGN.md): instrumented
        # kernel over the same frame at 1 spp (same camera, same jitter stream)
        cnt = r.render_counted(cam, W, H, spp=1, seed=1984, jitter=True)
        v_n, v_t = cnt["nodes"] / cnt["rays"], cnt["tris"] / cnt["rays"]
        bytes_per_ray = v_n * NODE_BYTES + v_t * 48 + 4.0 / spp
        if world == 1:
            kern_s = ms_per_step * 1e-3
            achieved = bytes_per_ray * rays_total / kern_s / 1e9
            # the honest limiter of this kernel is instruction issue, not bytes: quote it next to the node-fetch fraction.
            # Software counters (instrumented kernel, this run): SIMD efficiency of the two phases at the bench's lane layout;
            # hardware counters: the committed ncu capture of this very kernel source, or nothing.
            cs = r.render_counted(cam, W, H, spp=spp, seed=1984, jitter=True)
            wn, wl = r.get_stat("trace_warp_node_steps"), r.get_stat("trace_warp_leaf_steps")
            hw = ncu_counters("bench_4k16spp_1m")
            sm_hz = (clocks or {}).get("sm_mhz") or 0
            issue_frac = None
            if hw and "warp_inst_per_ray" in hw and sm_hz:
                issue_frac = hw["warp_inst_per_ray"] * rays_total / (r.get_stat("sm_count") * 4 * sm_hz * 1e6 * kern_s)
            roofline = {"bound": "hbm", "kernel": "k_trace<render>", "achieved": achieved, "peak": peak, "unit": "GB/s",
                        "frac": achieved / peak, "traffic": (hw or {}).get("dram_bytes_per_launch"), "peak_source": peak_src,
                        "algorithmic_bytes_per_ray": bytes_per_ray, "nodes_per_ray": v_n, "tris_per_ray": v_t,
                        "issue_frac": issue_frac,
                        "lanes_active": (hw or {}).get("lanes_active"), "l1_hit": (hw or {}).get("l1_hit"), "l2_hit": (hw or {}).get("l2_hit"),
                        "hw_counters_source": (hw or {}).get("source") or (hw or {}).get("stale"),
                        "simd_efficiency_node_phase": cs["nodes"] / (32.0 * wn) if wn else None,
                        "simd_efficiency_leaf_phase": cs["tris"] / (32.0 * wl) if wl else None,
                        "note": "frac = node + triangle fetch bytes of the shipped traversal order over the measured HBM peak (the north star's "
                                "fraction).  It is NOT a bound here: the scene (62 MB) is L2-resident and a warp's rays share nodes in L1, so DRAM "
                                "traffic is ~1000x below the algorithmic bytes and frac can exceed 1.  The limiter is instruction issue: issue_frac = "
                                "warp instructions (ncu, same kernel source) / (SMs x 4 schedulers x SM clock x kernel time); useful work = issue_frac x "
                                "lanes_active / 32"}
        else:
            roofline = None
        out = {"metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
               "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
               "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "config": {"workload": name, "triangles": n_tri, "leaves": info["nu"], "rays_per_step": rays_total,
                          "l2": "flushed before every timed step (256 MiB write)", "parallelism": "%s%d" % (mode, world),
                          "scheduling": "launches of 64 k .. 48 M rays per GPU (scenes of >= 10 k triangles) start the tiles whose longest unit was slow in the previous frame of the "
                                        "same geometry first (costs measured by the kernel itself; warm-up frames provide the first order)",
                          "sharding": {"single": "one GPU",
                                       "p2p": "every rank walks every 32x32 tile and owns every N-th 32-ray unit; the trace kernel stores the finished "
                                              "pixels straight into rank 0's framebuffer over NVLink (CUDA IPC mapping), one-element all-reduce as frame barrier",
                                       "interleave": "every rank walks every 32x32 tile and owns every N-th 32-ray unit (hit counts, reduce, resolve)",
                                       "samples": "samples of every pixel split over ranks (hit counts, reduce, resolve)",
                                       "tiles": "32x32-pixel tiles round-robin over ranks"}[mode] + "; BIH broadcast once" + ("" if mode in ("single", "p2p") else "; framebuffer reduce per step")},
               "frame_crc32": frame_crc, "oracle_tile_check": tile_check,
               "build_ms_per_mtri": build_ms / (n_tri / 1e6), "build_ms": build_ms,
               "build_roofline": {"bound": "hbm", "algorithmic_bytes_per_triangle": 320, "achieved": n_tri * 320 / (build_ms * 1e-3) / 1e9,
                                  "peak": peak, "unit": "GB/s", "frac": n_tri * 320 / (build_ms * 1e-3) / 1e9 / peak},
               "e2e": {"value": e2e_val, "unit": "Mrays/s", "h2d_bytes_per_step": n_tri * 36 if (can_pipe and upload_mode == "one") else n_tri * 36 * world, "d2h_bytes_per_step": W * H * 4,
                       "ms_per_step": ms_e2e, "frames_timed": e2e_frames, "frame_crc32": e2e_crc,
                       "serial_value": rays_total / (ms_e2e_serial * 1e-3) / 1e6, "serial_ms_per_step": ms_e2e_serial,
                       "upload": upload_mode if can_pipe else "each",
                       "what": ("per frame: vertices H2D from pinned host memory (36 MB%s) + bihrt_build on every rank (local, "
                                "deterministic: identical trees, no BIH broadcast) + every rank's share of the frame stored into rank 0's framebuffer%s; rank 0: framebuffer D2H to "
                                "pinned memory.  Pipelined frame loop: the upload of frame k+1 and the download of frame k-1 run on copy streams while frame k is traced (value); "
                                "serial_value = every rank uploads its own copy, nothing overlapped" % (
                                    (", by every rank over its own PCIe link" if upload_mode == "each" else ", by rank frame %% %d over its own PCIe link, then one NVLink broadcast" % world) if world > 1 else "",
                                    " over NVLink + frame barrier" if world > 1 else "")) if can_pipe else
                               "vertices H2D (pinned) + bihrt_build + render + framebuffer reduce + D2H (pinned), per frame, serial"},
               "gpu_launches": int(launches), "clocks": clocks}
        if animated:
            out["animated_frame_1080p_1spp"] = animated
        if config4:
            out["config4_10m_4k_16spp"] = config4
        if breakdown:
            out["breakdown"] = breakdown
            out["multi_gpu_image_bit_identical_to_single_gpu"] = image_ok
            out["single_gpu_frame_crc32"] = single_crc
        if roofline:
            out["roofline"] = roofline

    # ---- N=1 extras: the other BASELINE configs / sizes and the baselines -------------------------
    if rank == 0 and world == 1 and not args.no_extras:
        def med(fn, k=5):
            fn(); r.sync()
            return float(np.median([timed_loop(fn, 1) for _ in range(k)]))

        def primary(c2, w, h, s_):
            return w * h * s_ / (med(lambda: r.render(c2, w, h, spp=s_, jitter=s_ > 1)) * 1e-3) / 1e6

        def shadow_pass(c3, w, h, s_, light, label):
            """BASELINE's metric names primary + shadow rays: one frame = primary hits per sample -> shadow rays to a point
            light generated on the device -> occlusion trace.  Everything is timed; rates and the node-fetch fraction of
            the combined pass."""
            jit = s_ > 1
            db, _src = r.secondary_rays(c3, w, h, spp=s_, kind="shadow", light=light, jitter=jit)
            blk = torch.empty(len(db), dtype=torch.int32, device=dev)
            n_p, n_s = w * h * s_, len(db)
            t_p = med(lambda: r.render(c3, w, h, spp=s_, jitter=jit))
            t_gen = med(lambda: r.secondary_rays(c3, w, h, spp=s_, kind="shadow", light=light, jitter=jit), 3)   # primary hit buffers + generation
            t_s = med(lambda: r.trace_any(db, tmax=1.0, blocker=blk))
            t_c = med(lambda: (r.secondary_rays(c3, w, h, spp=s_, kind="shadow", light=light, jitter=jit), r.trace_any(db, tmax=1.0, blocker=blk)), 3)
            cp = r.render_counted(c3, w, h, spp=s_, jitter=jit)
            _t, _s, _p, cq = r.trace(db, counted=True)
            # (the occlusion query visits fewer nodes than the closest-hit trace the counters come from: upper bound on its bytes)
            bytes_p = cp["nodes"] * NODE_BYTES + cp["tris"] * 48 + n_p * 12
            bytes_s = cq["nodes"] * NODE_BYTES + cq["tris"] * 48 + n_s * 28
            pk = peaks()[0]
            return {"what": label, "primary_rays": n_p, "shadow_rays": n_s,
                    "primary_mrays_s": n_p / (t_p * 1e-3) / 1e6, "shadow_occlusion_mrays_s": n_s / (t_s * 1e-3) / 1e6,
                    "hits_plus_shadow_generation_ms": t_gen, "frame_ms": t_c,
                    "primary_plus_shadow_mrays_s": (n_p + n_s) / (t_c * 1e-3) / 1e6,
                    "roofline_frac": (bytes_p + bytes_s) / (t_c * 1e-3) / 1e9 / pk,
                    "shadow_nodes_per_ray_closest_hit": cq["nodes"] / max(n_s, 1), "shadow_tris_per_ray_closest_hit": cq["tris"] / max(n_s, 1)}

        configs = {}
        try:
            # the metric's other half on the bench scene: primary + shadow rays, 1080p x 4 spp
            out["primary_plus_shadow"] = shadow_pass(scenes.pinhole_camera(aspect=1920 / 1080), 1920, 1080, 4, (2.0, 3.0, -3.0),
                                                     "bench scene (1 M triangles), 1920x1080 x 4 spp jittered: per-sample primary hits -> shadow rays to a point light "
                                                     "(generated on the device) -> occlusion query; all three timed together (frame_ms)")
        except Exception as ex:           # noqa
            out["primary_plus_shadow"] = {"error": repr(ex)[:200]}
        try:
            # config 1: Cornell box, 512x512, 1 spp
            r.load_models(torch.from_numpy(scenes.cornell_box()).to(dev)); r.build()
            configs["config1_cornell_32tri_512x512_1spp"] = {"primary_mrays_s": primary(scenes.cornell_camera(), 512, 512, 1)}
            # sizes: build ms/Mtri and 1080p primary rays on the displaced spheres of configs 2/4/5
            c2 = scenes.pinhole_camera(aspect=1920 / 1080)
            for key, label in (("70k", "config2_70k_1080p"), ("260k", "sphere_260k_1080p"), ("1m", "config5_1m_1080p"), ("10m", "config4_10m")):
                t2 = scenes.displaced_sphere(scenes.SPHERE_NSEG[key])
                d = torch.from_numpy(t2).to(dev)
                r.load_models(d)
                bms = med(lambda: r.build())
                e = {"triangles": len(t2), "leaves": r.build_info()["nu"], "build_ms": bms, "build_ms_per_mtri": bms / (len(t2) / 1e6),
                     "build_roofline_frac": len(t2) * 320 / (bms * 1e-3) / 1e9 / peaks()[0],
                     "primary_mrays_s_1080p_1spp": primary(c2, 1920, 1080, 1), "primary_mrays_s_1080p_4spp": primary(c2, 1920, 1080, 4)}
                cc = r.render_counted(c2, 1920, 1080, spp=1)
                bpr = cc["nodes"] / cc["rays"] * NODE_BYTES + cc["tris"] / cc["rays"] * 48 + 4.0
                pk = peaks()[0]
                e.update({"nodes_per_ray": cc["nodes"] / cc["rays"], "tris_per_ray": cc["tris"] / cc["rays"], "algorithmic_bytes_per_ray": bpr,
                          "roofline_frac_1080p_1spp": e["primary_mrays_s_1080p_1spp"] * 1e6 * bpr / (pk * 1e9),
                          "roofline_frac_1080p_4spp": e["primary_mrays_s_1080p_4spp"] * 1e6 * bpr / (pk * 1e9)})
                if key == "1m":      # config 5: animated frame = rebuild + trace, 1080p
                    tms = med(lambda: r.render(c2, 1920, 1080, spp=1))
                    fms = med(lambda: (r.build(), r.render(c2, 1920, 1080, spp=1)))
                    rms = med(lambda: r.refit())
                    r.build()
                    e["animated_frame_1080p_1spp"] = {"build_ms": bms, "trace_ms": tms, "frame_ms": fms, "fps": 1e3 / fms,
                                                      "refit_ms_nonparity": rms}
                    e["moving_camera_1080p_1spp"] = moving_camera(r, scenes, timed_loop, 1920, 1080)
                if key in ("1m", "10m"):
                    # quality mode (SURVEY.md 8(f) f4; NOT a parity path, reported separately): 63-bit Morton keys, leaves capped at 4
                    try:
                        r.set_option("morton_bits", 63); r.set_option("leaf_cap", 4)
                        qb = med(lambda: r.build())
                        cq = r.render_counted(c2, 1920, 1080, spp=1)
                        e["quality_mode_63bit_cap4"] = {
                            "parity": False, "leaves": r.build_info()["nu"], "build_ms_per_mtri": qb / (len(t2) / 1e6),
                            "primary_mrays_s_1080p_1spp": primary(c2, 1920, 1080, 1), "primary_mrays_s_1080p_4spp": primary(c2, 1920, 1080, 4),
                            "nodes_per_ray": cq["nodes"] / cq["rays"], "tris_per_ray": cq["tris"] / cq["rays"],
                            "what": "non-parity tree: 21-bit grid per axis, ties broken by position, subtrees of <= 4 triangles collapsed into leaves; hits == brute force "
                                    "(tests/test_gpu_quality.py)"}
                    except Exception as ex:       # noqa
                        e["quality_mode_63bit_cap4"] = {"error": repr(ex)[:200]}
                    r.set_option("morton_bits", 30)
                    r.build()
                if key == "10m":     # config 4: 4K x 16 spp
                    c4 = scenes.pinhole_camera(aspect=3840 / 2160)
                    e["primary_mrays_s_4k_16spp"] = 3840 * 2160 * 16 / (med(lambda: r.render(c4, 3840, 2160, spp=16, jitter=True), 3) * 1e-3) / 1e6
                configs[label] = e
                del d
            # config 3: atrium, 1080p primary + shadow rays to a point light + one diffuse bounce (ray lists on the device)
            ta = scenes.atrium()
            r.load_models(torch.from_numpy(ta).to(dev))
            bms = med(lambda: r.build())
            ca = scenes.atrium_camera(1920 / 1080)
            e = {"triangles": len(ta), "build_ms_per_mtri": bms / (len(ta) / 1e6), "primary_mrays_s_1080p_1spp": primary(ca, 1920, 1080, 1)}
            # shadow rays to a point light and one cosine-weighted bounce, generated on the device from the
            # primary hits (bihrt_secondary_rays), traced as ray lists
            for nm, kind in (("shadow", "shadow"), ("bounce", "diffuse")):
                db, _src = r.secondary_rays(ca, 1920, 1080, spp=1, kind=kind, light=(0.0, 0.8, 0.0))
                ot = torch.empty(len(db), dtype=torch.float32, device=dev)
                os_ = torch.empty(len(db), dtype=torch.int32, device=dev)
                ms_b = med(lambda: r.trace(db, t=ot, slot=os_, prim=os_))
                e[nm + "_mrays_s"] = len(db) / (ms_b * 1e-3) / 1e6
                if nm == "shadow":      # occlusion query: is the light (t = 1) hidden -- ends at the first blocker
                    ms_o = med(lambda: r.trace_any(db, tmax=1.0, blocker=os_))
                    e["shadow_occlusion_mrays_s"] = len(db) / (ms_o * 1e-3) / 1e6
                if nm == "bounce":      # incoherent batch: traced through the origin-cell / octant permutation (sort included in the time)
                    r.set_option("trace_sort_rays", 1)
                    ms_s = med(lambda: r.trace(db, t=ot, slot=os_, prim=os_))
                    r.set_option("trace_sort_rays", 0)
                    e["bounce_sorted_mrays_s"] = len(db) / (ms_s * 1e-3) / 1e6
                e[nm + "_rays"] = len(db)
                e[nm + "_generation_ms"] = med(lambda: r.secondary_rays(ca, 1920, 1080, spp=1, kind=kind, light=(0.0, 0.8, 0.0)), 3)
            e["primary_plus_shadow"] = shadow_pass(ca, 1920, 1080, 1, (0.0, 0.8, 0.0), "atrium, 1920x1080 x 1 spp: primary hits -> shadow rays -> occlusion query")
            configs["config3_atrium_262k_1080p"] = e
        except Exception as ex:           # noqa
            configs["error"] = repr(ex)[:200]
        out["configs"] = configs
        out["cpu_baseline"] = cpu_baseline(args, tri, cam)
        out["reference_kernels_b200"] = reference_kernels_baseline(args, tri, cam)
    if rank == 0:
        emit(out)
    if peer_opened:
        r.framebuffer_ipc_close(peer_ptr)
    if world > 1:
        barrier()
    r.close()
    if world > 1:
        dist.destroy_process_group()


def moving_camera(r, scenes, timed_loop, w, h, frames=60):
    """The tile schedule is learnt from the PREVIOUS frame: check it on a camera that moves.  A 60-frame orbit (6 degrees
    per frame) around the mesh at 1 spp, traced with the cost-ordered schedule and in scan order."""
    res = {}
    cams = []
    for k in range(frames):
        a = 2 * np.pi * k / frames
        cams.append(scenes.look_at_camera((3.0 * np.sin(a) + 0.1, 0.2, -3.0 * np.cos(a)), (0.0, 0.0, 0.0), 0.45, w / h))
    for nm, opt in (("tile_order_on", 1), ("tile_order_off", 0)):
        r.set_option("trace_tile_order", opt)
        for c in cams[:3]:
            r.render(c, w, h, spp=1)
        r.sync()
        it = iter(cams)
        ms = timed_loop(lambda: r.render(next(it), w, h, spp=1), frames)
        res[nm + "_ms_per_frame"] = ms / frames
        res[nm + "_mrays_s"] = w * h / (ms / frames * 1e-3) / 1e6
    r.set_option("trace_tile_order", 1)
    res["what"] = "%d-frame orbit, 6 degrees per frame, %dx%d x 1 spp; every frame's tile order comes from the previous (different) view" % (frames, w, h)
    return res


def cpu_baseline(args, tri, cam):
    """The oracle (port of the reference algorithm) on the box's host cores, bounded sample."""
    from oracle import oracle as O
    t0 = time.perf_counter()
    ob = O.Bih(tri)
    build_s = time.perf_counter() - t0
    w, h = cpu_sample(args, 4)
    rays = O.camera_rays(cam, w, h)
    cores = host_cores()
    t0 = time.perf_counter()
    ob.trace(rays, "ref", threads=cores)
    dt = time.perf_counter() - t0
    t0 = time.perf_counter()
    ob.trace(rays, "proper", threads=cores)
    dt_p = time.perf_counter() - t0
    r1 = np.ascontiguousarray(rays[::16])
    t0 = time.perf_counter()
    ob.trace(r1, "ref", threads=1)
    dt_1 = time.perf_counter() - t0
    # the reference's own default workload: 640x480 x 4 spp (R/src/Constants.h:4-8), jittered, its camera model
    rd = O.camera_rays(scenes_default_camera(), 640, 480, spp=4, jitter=True)
    t0 = time.perf_counter()
    ob.trace(rd, "ref", threads=cores)
    dt_d = time.perf_counter() - t0
    return {"value": len(rays) / dt / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port",
            "one_thread_mrays_s": len(r1) / dt_1 / 1e6,
            "reference_default_640x480x4spp": {"mrays_s": len(rd) / dt_d / 1e6, "frame_ms": dt_d * 1e3, "cores": cores,
                                               "what": "the reference's compile-time workload (R/src/Constants.h:4-8) on this scene, config-2 camera at 4:3"},
            "sample": "%dx%d pixel-centre primary rays of the same camera and scene (%d rays), literal reference traversal "
                      "semantics, OpenMP %d threads" % (w, h, len(rays), cores),
            "pruned_traversal_mrays_s": len(rays) / dt_p / 1e6,
            "build_ms_per_mtri": build_s * 1e3 / (len(tri) / 1e6), "build_threads": 1}


def scenes_default_camera():
    from bihrt import scenes
    return scenes.pinhole_camera(aspect=640 / 480)


def reference_kernels_baseline(args, tri, cam):
    """The reference's own BuildTree / FindClipPlanes / TraverseTree (+ the thrust calls of its Render),
    compiled unmodified for sm_100a (oracle/_ref, built in the dev container), on this GPU: a reported
    baseline next to the CPU one (BASELINE.md section 2), 1 GPU only."""
    try:
        from oracle import oracle as O
        from oracle import ref_harness
        if not ref_harness.available():
            log("!!! oracle/_ref/libref_harness.so is MISSING on this box: the reference-kernel pin and baseline did not run "
                "(it is built by __graft_entry__.build() where /root/reference exists and travels with the snapshot)")
            return {"unavailable": "oracle/_ref/libref_harness.so not built (reference tree absent at build time)", "LOUD": True}
        ob = O.Bih(tri)
        ref = ref_harness.RefScene(ob)
        ref.build()
        bms = []
        for _ in range(5):
            ref.build(); bms.append(ref.build_ms())
        w, h = cpu_sample(args, 4)
        rays = O.camera_rays(cam, w, h)
        _, _, ms = ref.trace(rays, reps=3)
        ref.close()
        return {"build_ms_per_mtri": float(np.median(bms)) / (len(tri) / 1e6), "trace_mrays_s": len(rays) / (ms * 1e-3) / 1e6,
                "sample": "%dx%d pixel-centre primary rays, reference TraverseTree kernel, 64-thread blocks; build = thrust transform/"
                          "sequence/stable_sort_by_key/reduce_by_key/unique_by_key_copy + BuildTree + FindClipPlanes with the "
                          "reference's cudaDeviceSynchronize after each step" % (w, h)}
    except Exception as ex:           # noqa
        return {"unavailable": repr(ex)[:200]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scene", default="1m", choices=["70k", "260k", "1m", "10m"])
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--spp", type=int, default=16)
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-config4", action="store_true", help="N > 1: skip the 10 M-triangle config-4 section")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the framebuffer of the last timed step to DIR/framebuffer.npy (float32, packed r | g<<8 | b<<16)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus:
        log("note: WORLD_SIZE=%d, --gpus=%d; using WORLD_SIZE" % (world, args.gpus))
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
