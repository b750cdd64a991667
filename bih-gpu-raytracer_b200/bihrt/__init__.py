"""Host-side mirror of the reference's interface for the BIH hot path, on top of libbihrt.so.

The reference exposes the path through three C++ classes; this module keeps their names and the
meaning of their entry points so that tests read like calls into the reference:

    App::LoadModels(path)                R/src/App.cpp:65-167      -> Renderer.load_models(tri9 | path)
    Renderer::Render(GPUArrayManager&)   R/src/Renderer.cpp:415-672 -> Renderer.build() + Renderer.render(...)
    GPUArrayManager getters              R/src/GPUArrayManager.h:18-38 -> Renderer.reference_view()
    Launch_cudaRender / TraverseTree     R/src/CUDAKernels.cu:227-447 -> Renderer.trace(rays)
    m_cudaDestResource                   R/src/Renderer.h:46       -> Renderer.framebuffer()

Everything goes through the C ABI in include/bihrt.h (ctypes); torch is used only for device
buffers, streams and torch.distributed.  There is no CPU fallback: importing works anywhere, but
constructing a Renderer without libbihrt.so or without a B200-class GPU raises.
"""
import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(_PKG, "libbihrt.so")

OK = 0
RENDER_JITTER = 1


class BihrtError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("bihrt error %d: %s" % (code, msg))
        self.code = code


class Config(C.Structure):
    _fields_ = [("device", C.c_int32), ("flags", C.c_uint32), ("reserved", C.c_int32 * 6)]


class Camera(C.Structure):
    _fields_ = [("origin", C.c_float * 3), ("lower_left", C.c_float * 3),
                ("horizontal", C.c_float * 3), ("vertical", C.c_float * 3)]

    @staticmethod
    def from_array(cam12):
        cam12 = np.asarray(cam12, np.float32).reshape(12)
        c = Camera()
        C.memmove(C.byref(c), cam12.ctypes.data, 48)
        return c


class RefView(C.Structure):
    _fields_ = [("n", C.c_int64), ("nu", C.c_int64), ("scene_lo", C.c_float * 3), ("scene_hi", C.c_float * 3),
                ("morton_codes", C.c_void_p), ("tris_indexes", C.c_void_p), ("unique_morton_codes", C.c_void_p),
                ("duplicates_cnts", C.c_void_p), ("first_idxs", C.c_void_p), ("clip_planes", C.c_void_p),
                ("axis", C.c_void_p), ("is_leaf", C.c_void_p), ("children", C.c_void_p), ("parent", C.c_void_p),
                ("leaf_parents", C.c_void_p)]


class BuildInfo(C.Structure):
    _fields_ = [("n", C.c_int64), ("nu", C.c_int64), ("node_bytes", C.c_int64), ("tri_bytes", C.c_int64),
                ("last_build_ms", C.c_float), ("sort_passes", C.c_int32), ("reserved", C.c_int32 * 6)]


class Hits(C.Structure):
    """bihrt_hits: where bihrt_intersect writes each part of the hit record (NULL = not wanted)."""
    _fields_ = [("t", C.c_void_p), ("u", C.c_void_p), ("v", C.c_void_p), ("slot", C.c_void_p), ("prim", C.c_void_p),
                ("ng", C.c_void_p)]


class Closest(C.Structure):
    """bihrt_closest: where bihrt_closest_point writes each part of the record (NULL = not wanted)."""
    _fields_ = [("d2", C.c_void_p), ("u", C.c_void_p), ("v", C.c_void_p), ("slot", C.c_void_p), ("prim", C.c_void_p),
                ("q", C.c_void_p), ("ng", C.c_void_p)]


INTERSECT_ANY = 1
INTERSECT_TWO_SIDED = 4
HIT_OUTPUTS = ("t", "u", "v", "slot", "prim", "ng")
CLOSEST_OUTPUTS = ("d2", "u", "v", "slot", "prim", "q", "ng")


def interval_rays(rays6, tmin=0.0, tmax=np.inf):
    """(N,8) float32 rays o.xyz tmin d.xyz tmax for Renderer.intersect, from (N,6) rays o.xyz d.xyz and a scalar or per-ray
    (N,) tmin / tmax.  numpy in -> numpy out; torch in -> torch out on the same device."""
    if isinstance(rays6, np.ndarray):
        r = np.asarray(rays6, np.float32).reshape(-1, 6)
        out = np.empty((r.shape[0], 8), np.float32)
    else:
        import torch
        r = rays6.reshape(-1, 6).to(torch.float32)
        out = torch.empty((r.shape[0], 8), dtype=torch.float32, device=r.device)
    out[:, 0:3] = r[:, 0:3]
    out[:, 4:7] = r[:, 3:6]
    out[:, 3] = tmin
    out[:, 7] = tmax
    return out


def point_queries(points3, rmax=np.inf):
    """(N,4) float32 queries p.xyz rmax for Renderer.closest_point, from (N,3) points and a scalar or per-point (N,) search
    radius.  numpy in -> numpy out; torch in -> torch out on the same device."""
    if isinstance(points3, np.ndarray):
        p = np.asarray(points3, np.float32).reshape(-1, 3)
        out = np.empty((p.shape[0], 4), np.float32)
    else:
        import torch
        p = points3.reshape(-1, 3).to(torch.float32)
        out = torch.empty((p.shape[0], 4), dtype=torch.float32, device=p.device)
    out[:, 0:3] = p
    out[:, 3] = rmax
    return out


# every symbol include/bihrt.h declares (tests check that the library exports all of them)
ABI_SYMBOLS = [
    "bihrt_version", "bihrt_create", "bihrt_destroy", "bihrt_last_error", "bihrt_set_stream", "bihrt_get_stream", "bihrt_sync",
    "bihrt_set_option", "bihrt_get_stat", "bihrt_scene_load_triangles", "bihrt_scene_update_vertices", "bihrt_scene_load_obj",
    "bihrt_build", "bihrt_refit", "bihrt_get_build_info", "bihrt_export_reference_view", "bihrt_trace", "bihrt_trace_any", "bihrt_intersect", "bihrt_closest_point", "bihrt_winding_number", "bihrt_trace_counted",
    "bihrt_render", "bihrt_render_counted", "bihrt_render_shard", "bihrt_render_samples", "bihrt_render_interleaved", "bihrt_render_interleaved_to", "bihrt_framebuffer_ipc_export", "bihrt_framebuffer_ipc_open", "bihrt_framebuffer_ipc_close", "bihrt_framebuffer_ipc_unexport", "bihrt_bih_region", "bihrt_bih_adopt", "bihrt_bih_copy", "bihrt_framebuffer_resolve", "bihrt_render_hits", "bihrt_secondary_rays", "bihrt_framebuffer", "bihrt_framebuffer_read",
    "bihrt_bih_blob_bytes", "bihrt_bih_export", "bihrt_bih_import",
    "bihrt_create_multi", "bihrt_destroy_multi", "bihrt_multi_size", "bihrt_multi_nccl_version", "bihrt_multi_broadcast",
    "bihrt_multi_render", "bihrt_multi_sync",
]

_lib = None


def load_library(path=None):
    """dlopen libbihrt.so (no CUDA call is made).  Raises if the library has not been built."""
    global _lib
    if _lib is None or path:
        p = path or os.environ.get("BIHRT_LIB") or LIB_PATH
        if not os.path.exists(p):
            raise BihrtError(-100, "%s not found: build it with `make -C %s` (there is no CPU fallback)" % (p, _PKG))
        lib = C.CDLL(p)
        lib.bihrt_last_error.restype = C.c_char_p
        lib.bihrt_last_error.argtypes = [C.c_void_p]
        lib.bihrt_destroy.restype = None
        lib.bihrt_destroy.argtypes = [C.c_void_p]
        lib.bihrt_destroy_multi.restype = None
        lib.bihrt_multi_broadcast.argtypes = [C.c_void_p]
        lib.bihrt_multi_sync.argtypes = [C.c_void_p]
        _lib = lib
    return _lib


def _ptr(x):
    """Pointer of a numpy array (host), a torch tensor (host or device), an int address, or None."""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        return C.c_void_p(x.ctypes.data)
    if isinstance(x, int):
        return C.c_void_p(x)
    if hasattr(x, "data_ptr"):
        return C.c_void_p(x.data_ptr())
    raise TypeError("unsupported buffer type %r" % type(x))


class Renderer:
    """One context = one GPU.  Mirrors the call order of the reference's frame:
    load_models -> build -> render/trace -> framebuffer."""

    def __init__(self, device=0, stream=None):
        self._lib = load_library()
        self._ctx = C.c_void_p()
        cfg = Config(device=device, flags=0)
        rc = self._lib.bihrt_create(C.byref(self._ctx), C.byref(cfg))
        if rc != OK:
            self._ctx = C.c_void_p()
            raise BihrtError(rc, "bihrt_create failed (no sm_100-class GPU visible? there is no CPU fallback)")
        self.device = device
        self.n = 0
        if stream is not None:
            self.set_stream(stream)

    # -- plumbing -----------------------------------------------------------------------------
    def _check(self, rc):
        if rc != OK:
            raise BihrtError(rc, self._lib.bihrt_last_error(self._ctx).decode())

    def close(self):
        if getattr(self, "_ctx", None) and self._ctx.value:
            self._lib.bihrt_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream):
        """Run on a caller-owned stream: an int cudaStream_t with CUDA's meaning (0 = the legacy default stream, which is
        what torch.cuda.current_stream().cuda_stream is on torch's default stream), or None / "own" for the context's
        private stream."""
        own = cuda_stream is None or cuda_stream == "own"
        h = C.c_void_p(-1) if own else C.c_void_p(int(cuda_stream))
        self._check(self._lib.bihrt_set_stream(self._ctx, h))

    def stream_handle(self):
        """The cudaStream_t (int) the context launches on."""
        p = C.c_void_p()
        self._check(self._lib.bihrt_get_stream(self._ctx, C.byref(p)))
        return p.value or 0

    # Ordering with torch work.  The library launches on the context's stream; torch tensors handed in were produced,
    # and tensors handed out will be consumed, on torch's CURRENT stream.  When the two differ they are ordered with
    # events (no host synchronisation): wait_torch() before a call that reads torch memory, torch_wait() after a call
    # that wrote it.  Both are no-ops when the context already runs on torch's current stream.
    def _torch_streams(self):
        import torch
        cur = torch.cuda.current_stream(self.device)
        h = self.stream_handle()
        if h == cur.cuda_stream:
            return None, None
        return torch.cuda.ExternalStream(h, device=self.device), cur

    def wait_torch(self):
        """The context's stream waits for the work enqueued so far on torch's current stream."""
        ext, cur = self._torch_streams()
        if ext is not None:
            ext.wait_stream(cur)

    def torch_wait(self):
        """torch's current stream waits for the work enqueued so far on the context's stream."""
        ext, cur = self._torch_streams()
        if ext is not None:
            cur.wait_stream(ext)

    def sync(self):
        self._check(self._lib.bihrt_sync(self._ctx))

    def set_option(self, name, value):
        self._check(self._lib.bihrt_set_option(self._ctx, name.encode(), C.c_int64(int(value))))

    def get_stat(self, name):
        v = C.c_int64()
        self._check(self._lib.bihrt_get_stat(self._ctx, name.encode(), C.byref(v)))
        return v.value

    # -- App::LoadModels ------------------------------------------------------------------------
    def load_models(self, src):
        """src: path of a Wavefront .obj, or (N,9) float32 triangles (numpy / torch, host or device)."""
        if isinstance(src, (str, bytes, os.PathLike)):
            self._check(self._lib.bihrt_scene_load_obj(self._ctx, os.fsencode(src)))
            self.n = None
            return self
        if isinstance(src, np.ndarray):
            src = np.ascontiguousarray(src, dtype=np.float32)
            n = src.size // 9
        else:
            n = src.numel() // 9
        self._keep = src
        if getattr(src, "is_cuda", False):
            self.wait_torch()
        self._check(self._lib.bihrt_scene_load_triangles(self._ctx, _ptr(src), C.c_int64(n)))
        self.n = n
        return self

    def update_vertices(self, src):
        if isinstance(src, np.ndarray):
            src = np.ascontiguousarray(src, dtype=np.float32)
            n = src.size // 9
        else:
            n = src.numel() // 9
        self._keep = src
        if getattr(src, "is_cuda", False):
            self.wait_torch()
        self._check(self._lib.bihrt_scene_update_vertices(self._ctx, _ptr(src), C.c_int64(n)))

    # -- first half of Renderer::Render -----------------------------------------------------------
    def build(self):
        self._check(self._lib.bihrt_build(self._ctx))
        return self

    def refit(self):
        """Non-parity fast update after update_vertices: same topology, new clip planes (bihrt_refit)."""
        self._check(self._lib.bihrt_refit(self._ctx))
        return self

    def build_info(self):
        bi = BuildInfo()
        self._check(self._lib.bihrt_get_build_info(self._ctx, C.byref(bi)))
        return {"n": bi.n, "nu": bi.nu, "node_bytes": bi.node_bytes, "tri_bytes": bi.tri_bytes,
                "last_build_ms": bi.last_build_ms, "sort_passes": bi.sort_passes}

    def reference_view(self):
        """The reference's device arrays (SURVEY.md 2.3) as numpy arrays, trimmed to n / Nu."""
        info = self.build_info()
        n, m = info["n"], max(info["n"], 1)
        out = {
            "morton_codes": np.zeros(m, np.uint32), "tris_indexes": np.zeros(m, np.uint32),
            "unique_morton_codes": np.zeros(m, np.uint32), "duplicates_cnts": np.zeros(m, np.uint32),
            "first_idxs": np.zeros(m, np.int32), "clip_planes": np.zeros((m, 2), np.float32),
            "axis": np.zeros(m, np.int32), "is_leaf": np.zeros((m, 2), np.uint8),
            "children": np.zeros((m, 2), np.int32), "parent": np.zeros(m, np.int32),
            "leaf_parents": np.zeros(m, np.int32)}
        v = RefView()
        for k, a in out.items():
            setattr(v, k, a.ctypes.data)
        self._check(self._lib.bihrt_export_reference_view(self._ctx, C.byref(v)))
        nu, ni = v.nu, max(v.nu - 1, 0)
        trim = {"morton_codes": n, "tris_indexes": n, "unique_morton_codes": nu, "duplicates_cnts": nu,
                "first_idxs": nu, "leaf_parents": nu, "clip_planes": ni, "axis": ni, "is_leaf": ni,
                "children": ni, "parent": ni}
        res = {k: out[k][:trim[k]] for k in out}
        res.update(n=n, nu=nu, scene_lo=np.array(list(v.scene_lo), np.float32),
                   scene_hi=np.array(list(v.scene_hi), np.float32))
        return res

    # -- Launch_cudaRender / TraverseTree -----------------------------------------------------------
    def trace(self, rays, t=None, slot=None, prim=None, counted=False):
        """rays: (N,6) float32 o.xyz d.xyz (numpy or torch, host or device).  With numpy input the
        outputs are numpy arrays; with torch input they are torch tensors on the rays' device unless
        given.  Returns (t, slot, prim[, counters])."""
        if isinstance(rays, np.ndarray):
            rays = np.ascontiguousarray(rays, dtype=np.float32)
            n = rays.size // 6
            t = np.empty(n, np.float32) if t is None else t
            slot = np.empty(n, np.int32) if slot is None else slot
            prim = np.empty(n, np.int32) if prim is None else prim
        else:
            import torch
            n = rays.numel() // 6
            t = torch.empty(n, dtype=torch.float32, device=rays.device) if t is None else t
            slot = torch.empty(n, dtype=torch.int32, device=rays.device) if slot is None else slot
            prim = torch.empty(n, dtype=torch.int32, device=rays.device) if prim is None else prim
        on_dev = any(getattr(x, "is_cuda", False) for x in (rays, t, slot, prim))
        if on_dev:
            self.wait_torch()            # rays (and recycled output blocks) were last touched on torch's current stream
        if counted:
            cnt = (C.c_uint64 * 4)()
            self._check(self._lib.bihrt_trace_counted(self._ctx, _ptr(rays), C.c_int64(n), _ptr(t), _ptr(slot), _ptr(prim), cnt))
            return t, slot, prim, {"nodes": cnt[0], "tris": cnt[1], "max_stack": cnt[2], "rays": cnt[3]}
        self._check(self._lib.bihrt_trace(self._ctx, _ptr(rays), C.c_int64(n), _ptr(t), _ptr(slot), _ptr(prim)))
        if on_dev:
            self.torch_wait()            # device outputs are written asynchronously on the context's stream
        return t, slot, prim

    def trace_any(self, rays, tmax=1.0, blocker=None):
        """Occlusion query: blocker[i] >= 0 iff ray i hits something with 0 < t < tmax (bihrt_trace_any)."""
        if isinstance(rays, np.ndarray):
            rays = np.ascontiguousarray(rays, dtype=np.float32)
            n = rays.size // 6
            blocker = np.empty(n, np.int32) if blocker is None else blocker
        else:
            import torch
            n = rays.numel() // 6
            blocker = torch.empty(n, dtype=torch.int32, device=rays.device) if blocker is None else blocker
        on_dev = any(getattr(x, "is_cuda", False) for x in (rays, blocker))
        if on_dev:
            self.wait_torch()
        self._check(self._lib.bihrt_trace_any(self._ctx, _ptr(rays), C.c_int64(n), C.c_float(tmax), _ptr(blocker)))
        if on_dev:
            self.torch_wait()
        return blocker

    def intersect(self, rays8, any_hit=False, two_sided=False, outputs=HIT_OUTPUTS):
        """Ray queries with per-ray intervals (bihrt_intersect).  rays8: (N,8) float32 o.xyz tmin d.xyz tmax (numpy or torch,
        host or device; interval_rays builds it).  A triangle counts when max(tmin,0) < t < min(tmax,FLT_MAX); any_hit ends a
        ray at the first one (occlusion).  two_sided accepts back faces too (BIHRT_INTERSECT_TWO_SIDED): dot(d, ng) > 0 marks
        a back-face hit.  Returns {name: array} for the requested outputs of
        t (N,), u (N,), v (N,), slot (N,), prim (N,), ng (N,3): numpy for numpy input, torch tensors on the rays' device for
        torch input.  A miss reads t = FLT_MAX, slot = prim = -1, u = v = ng = 0."""
        unknown = set(outputs) - set(HIT_OUTPUTS)
        if unknown:
            raise ValueError("unknown outputs %s (known: %s)" % (sorted(unknown), ", ".join(HIT_OUTPUTS)))
        shapes = {"t": (), "u": (), "v": (), "slot": (), "prim": (), "ng": (3,)}
        if isinstance(rays8, np.ndarray):
            rays8 = np.ascontiguousarray(rays8, dtype=np.float32)
            n = rays8.size // 8
            res = {k: np.empty((n,) + shapes[k], np.int32 if k in ("slot", "prim") else np.float32) for k in outputs}
        else:
            import torch
            rays8 = rays8.contiguous()
            n = rays8.numel() // 8
            res = {k: torch.empty((n,) + shapes[k], dtype=torch.int32 if k in ("slot", "prim") else torch.float32, device=rays8.device)
                   for k in outputs}
        hits = Hits(**{k: _ptr(res[k]) for k in res})
        flags = (INTERSECT_ANY if any_hit else 0) | (INTERSECT_TWO_SIDED if two_sided else 0)
        on_dev = getattr(rays8, "is_cuda", False)
        if on_dev:
            self.wait_torch()            # rays (and recycled output blocks) were last touched on torch's current stream
        self._check(self._lib.bihrt_intersect(self._ctx, _ptr(rays8), C.c_int64(n), C.c_uint32(flags), C.byref(hits)))
        if on_dev:
            self.torch_wait()            # device outputs are written asynchronously on the context's stream
        return res

    def closest_point(self, queries4, outputs=CLOSEST_OUTPUTS):
        """Closest-point queries (bihrt_closest_point).  queries4: (N,4) float32 p.xyz rmax (numpy or torch, host or device;
        point_queries builds it).  A triangle counts when its squared distance d2 <= min(rmax^2, FLT_MAX); the result is the
        one with the smallest (d2, slot).  Returns {name: array} for the requested outputs of d2 (N,), u (N,), v (N,),
        slot (N,), prim (N,), q (N,3), ng (N,3): numpy for numpy input, torch tensors on the points' device for torch input.
        A miss reads d2 = FLT_MAX, slot = prim = -1, u = v = q = ng = 0."""
        unknown = set(outputs) - set(CLOSEST_OUTPUTS)
        if unknown:
            raise ValueError("unknown outputs %s (known: %s)" % (sorted(unknown), ", ".join(CLOSEST_OUTPUTS)))
        shapes = {"d2": (), "u": (), "v": (), "slot": (), "prim": (), "q": (3,), "ng": (3,)}
        if isinstance(queries4, np.ndarray):
            queries4 = np.ascontiguousarray(queries4, dtype=np.float32)
            n = queries4.size // 4
            res = {k: np.empty((n,) + shapes[k], np.int32 if k in ("slot", "prim") else np.float32) for k in outputs}
        else:
            import torch
            queries4 = queries4.contiguous()
            n = queries4.numel() // 4
            res = {k: torch.empty((n,) + shapes[k], dtype=torch.int32 if k in ("slot", "prim") else torch.float32,
                                  device=queries4.device) for k in outputs}
        rec = Closest(**{k: _ptr(res[k]) for k in res})
        on_dev = getattr(queries4, "is_cuda", False)
        if on_dev:
            self.wait_torch()            # points (and recycled output blocks) were last touched on torch's current stream
        self._check(self._lib.bihrt_closest_point(self._ctx, _ptr(queries4), C.c_int64(n), C.byref(rec)))
        if on_dev:
            self.torch_wait()            # device outputs are written asynchronously on the context's stream
        return res

    def winding_number(self, queries4, beta=2.0):
        """Generalized winding numbers (bihrt_winding_number): (1/4pi) x the signed solid angle of the mesh at each point, 1 inside
        and 0 outside a closed outward-wound mesh.  queries4: (N,4) float32 p.xyz rmax as for closest_point (rmax is not read;
        numpy or torch, host or device).  beta > 1 sets the accuracy of the far-field expansion (2 recommended; np.inf: the
        exact sum, O(n) per point).  Returns (N,) float32: numpy for numpy input, a torch tensor on the points' device for
        torch input."""
        beta = float(beta)
        if not beta > 1.0:
            raise ValueError("beta must be > 1 or inf (got %r)" % beta)
        if isinstance(queries4, np.ndarray):
            queries4 = np.ascontiguousarray(queries4, dtype=np.float32)
            n = queries4.size // 4
            w = np.empty(n, np.float32)
        else:
            import torch
            queries4 = queries4.contiguous()
            n = queries4.numel() // 4
            w = torch.empty(n, dtype=torch.float32, device=queries4.device)
        on_dev = getattr(queries4, "is_cuda", False)
        if on_dev:
            self.wait_torch()            # points (and recycled output blocks) were last touched on torch's current stream
        self._check(self._lib.bihrt_winding_number(self._ctx, _ptr(queries4), C.c_int64(n), C.c_float(beta), _ptr(w)))
        if on_dev:
            self.torch_wait()            # device outputs are written asynchronously on the context's stream
        return w

    def signed_distance(self, queries4, beta=2.0, outputs=("sd",)):
        """Signed distance from the two queries on the same points: sd = -sqrt(d2) where the winding number w > 0.5 (inside),
        +sqrt(d2) otherwise; a point whose search radius rmax reaches no triangle gets -inf / +inf.  outputs: "sd", "w" and any
        of CLOSEST_OUTPUTS.  Returns {name: array} as closest_point does."""
        unknown = set(outputs) - set(("sd", "w") + CLOSEST_OUTPUTS)
        if unknown:
            raise ValueError("unknown outputs %s (known: sd, w, %s)" % (sorted(unknown), ", ".join(CLOSEST_OUTPUTS)))
        closest = self.closest_point(queries4, outputs=tuple(dict.fromkeys(("d2", "slot") + tuple(k for k in outputs if k in CLOSEST_OUTPUTS))))
        w = self.winding_number(queries4, beta)
        res = {k: v for k, v in closest.items() if k in outputs}
        if "w" in outputs:
            res["w"] = w
        if "sd" in outputs:
            if isinstance(w, np.ndarray):
                dist = np.where(closest["slot"] >= 0, np.sqrt(closest["d2"]), np.float32(np.inf)).astype(np.float32)
                res["sd"] = np.where(w > 0.5, -dist, dist).astype(np.float32)
            else:
                import torch
                dist = torch.where(closest["slot"] >= 0, torch.sqrt(closest["d2"]), torch.full_like(closest["d2"], float("inf")))
                res["sd"] = torch.where(w > 0.5, -dist, dist)
        return res

    def render(self, camera, w, h, spp=1, seed=1984, jitter=False, shard=(0, 1)):
        cam = camera if isinstance(camera, Camera) else Camera.from_array(camera)
        self._check(self._lib.bihrt_render_shard(self._ctx, C.byref(cam), C.c_int32(w), C.c_int32(h), C.c_int32(spp),
                                                 C.c_uint64(seed), C.c_uint32(RENDER_JITTER if jitter else 0),
                                                 C.c_int32(shard[0]), C.c_int32(shard[1])))
        return self

    def render_samples(self, camera, w, h, spp, sample_begin, sample_end, seed=1984, jitter=True):
        """Multi-GPU sample sharding: hit counts of samples [sample_begin, sample_end) into the framebuffer."""
        cam = camera if isinstance(camera, Camera) else Camera.from_array(camera)
        self._check(self._lib.bihrt_render_samples(self._ctx, C.byref(cam), C.c_int32(w), C.c_int32(h), C.c_int32(spp),
                                                   C.c_uint64(seed), C.c_uint32(RENDER_JITTER if jitter else 0),
                                                   C.c_int32(sample_begin), C.c_int32(sample_end)))
        return self

    def render_interleaved(self, camera, w, h, spp, index, count, seed=1984, jitter=True):
        """Multi-GPU unit interleave: hit counts of every count-th 32-ray unit of every tile (bihrt_render_interleaved)."""
        cam = camera if isinstance(camera, Camera) else Camera.from_array(camera)
        self._check(self._lib.bihrt_render_interleaved(self._ctx, C.byref(cam), C.c_int32(w), C.c_int32(h), C.c_int32(spp),
                                                       C.c_uint64(seed), C.c_uint32(RENDER_JITTER if jitter else 0),
                                                       C.c_int32(index), C.c_int32(count)))
        return self

    def render_interleaved_to(self, camera, w, h, spp, index, count, target_ptr=None, seed=1984, jitter=True):
        """Multi-GPU unit interleave fused with the gather: the final colours of this rank's pixels are stored by the
        trace kernel straight into the framebuffer at `target_ptr` (another GPU's, over NVLink; None = own)."""
        cam = camera if isinstance(camera, Camera) else Camera.from_array(camera)
        self._check(self._lib.bihrt_render_interleaved_to(self._ctx, C.byref(cam), C.c_int32(w), C.c_int32(h), C.c_int32(spp),
                                                          C.c_uint64(seed), C.c_uint32(RENDER_JITTER if jitter else 0),
                                                          C.c_int32(index), C.c_int32(count), C.c_void_p(target_ptr)))
        return self

    def framebuffer_ipc_export(self, w, h):
        """64-byte CUDA IPC handle of this context's w x h framebuffer (allocated if needed)."""
        buf = C.create_string_buffer(64)
        self._check(self._lib.bihrt_framebuffer_ipc_export(self._ctx, C.c_int32(w), C.c_int32(h), buf))
        return buf.raw

    def framebuffer_ipc_open(self, handle):
        """Map another process's framebuffer; returns the device pointer to pass as target_ptr."""
        p = C.c_void_p()
        self._check(self._lib.bihrt_framebuffer_ipc_open(self._ctx, C.c_char_p(bytes(handle)), C.byref(p)))
        return p.value

    def framebuffer_ipc_close(self, ptr):
        self._check(self._lib.bihrt_framebuffer_ipc_close(self._ctx, C.c_void_p(ptr)))

    def framebuffer_ipc_unexport(self):
        """The peers have closed their mappings: the framebuffer may be reallocated again."""
        self._check(self._lib.bihrt_framebuffer_ipc_unexport(self._ctx))

    def framebuffer_resolve(self, spp):
        self._check(self._lib.bihrt_framebuffer_resolve(self._ctx, C.c_int32(spp)))
        return self

    def render_counted(self, camera, w, h, spp=1, seed=1984, jitter=False):
        cam = camera if isinstance(camera, Camera) else Camera.from_array(camera)
        cnt = (C.c_uint64 * 4)()
        self._check(self._lib.bihrt_render_counted(self._ctx, C.byref(cam), C.c_int32(w), C.c_int32(h), C.c_int32(spp),
                                                   C.c_uint64(seed), C.c_uint32(RENDER_JITTER if jitter else 0), cnt))
        return {"nodes": cnt[0], "tris": cnt[1], "max_stack": cnt[2], "rays": cnt[3]}

    def render_hits(self, camera, w, h, spp=1, seed=1984, jitter=False):
        cam = camera if isinstance(camera, Camera) else Camera.from_array(camera)
        n = w * h * spp
        t, slot, prim = np.empty(n, np.float32), np.empty(n, np.int32), np.empty(n, np.int32)
        self._check(self._lib.bihrt_render_hits(self._ctx, C.byref(cam), C.c_int32(w), C.c_int32(h), C.c_int32(spp),
                                                C.c_uint64(seed), C.c_uint32(RENDER_JITTER if jitter else 0),
                                                _ptr(t), _ptr(slot), _ptr(prim)))
        return t, slot, prim

    def secondary_rays(self, camera, w, h, spp=1, kind="shadow", light=(0.0, 0.0, 0.0), seed=1984, jitter=False):
        """Device-side shadow / diffuse-bounce rays from the primary hits of a camera frame.
        Returns (rays (M,6) float32 CUDA tensor, sample index (M,) int32 CUDA tensor)."""
        import torch
        cam = camera if isinstance(camera, Camera) else Camera.from_array(camera)
        n = w * h * spp
        dev = "cuda:%d" % self.device
        rays = torch.empty((n, 6), dtype=torch.float32, device=dev)
        src = torch.empty(n, dtype=torch.int32, device=dev)
        cnt = C.c_int64()
        lt = (C.c_float * 3)(*[float(x) for x in light])
        self.wait_torch()                # the fresh tensors may recycle blocks last used on torch's current stream
        self._check(self._lib.bihrt_secondary_rays(self._ctx, C.byref(cam), C.c_int32(w), C.c_int32(h), C.c_int32(spp), C.c_uint64(seed),
                                                   C.c_uint32(RENDER_JITTER if jitter else 0), C.c_int32({"shadow": 0, "diffuse": 1}[kind]),
                                                   lt, _ptr(rays), _ptr(src), C.byref(cnt)))
        return rays[:cnt.value], src[:cnt.value]

    # -- m_cudaDestResource ---------------------------------------------------------------------------
    def framebuffer_ptr(self):
        p, w, h = C.c_void_p(), C.c_int32(), C.c_int32()
        self._check(self._lib.bihrt_framebuffer(self._ctx, C.byref(p), C.byref(w), C.byref(h)))
        return p.value, w.value, h.value

    def framebuffer(self, out=None):
        """Packed r | g<<8 | b<<16 pixels, row 0 = bottom, as a (h, w) uint32 host array."""
        _, w, h = self.framebuffer_ptr()
        if out is None:
            out = np.empty((h, w), np.uint32)
        self._check(self._lib.bihrt_framebuffer_read(self._ctx, _ptr(out)))
        return out

    # -- BIH replication ---------------------------------------------------------------------------
    def bih_blob_bytes(self):
        b = C.c_uint64()
        self._check(self._lib.bihrt_bih_blob_bytes(self._ctx, C.byref(b)))
        return b.value

    def bih_export(self, dev_buffer, nbytes):
        self._check(self._lib.bihrt_bih_export(self._ctx, _ptr(dev_buffer), C.c_uint64(nbytes)))

    def bih_region(self, n):
        """(device pointer, bytes) of the whole blob of an n-triangle scene, laid out (and allocated) for n."""
        p, b = C.c_void_p(), C.c_uint64()
        self._check(self._lib.bihrt_bih_region(self._ctx, C.c_int64(n), C.byref(p), C.byref(b)))
        return p.value, b.value

    def bih_adopt(self, n):
        self._check(self._lib.bihrt_bih_adopt(self._ctx, C.c_int64(n)))

    def bih_import(self, dev_buffer, nbytes):
        self._check(self._lib.bihrt_bih_import(self._ctx, _ptr(dev_buffer), C.c_uint64(nbytes)))


class MultiRenderer:
    """Several GPUs of ONE process behind the C ABI (bihrt_create_multi: N contexts + one in-library NCCL communicator).
    .ctx[0] is the builder / gatherer and behaves like a Renderer; broadcast() replicates its BIH, render() traces one
    frame over all devices into ctx[0]'s framebuffer."""

    def __init__(self, ngpu):
        self._lib = load_library()
        self._arr = (C.c_void_p * ngpu)()
        self.ngpu = ngpu
        rc = self._lib.bihrt_create_multi(self._arr, C.c_int32(ngpu))
        if rc != OK:
            raise BihrtError(rc, "bihrt_create_multi(%d) failed (fewer GPUs, no peer access, or libnccl.so.2 missing)" % ngpu)
        self.ctx = []
        for i in range(ngpu):
            r = Renderer.__new__(Renderer)
            r._lib, r._ctx, r.device, r.n = self._lib, C.c_void_p(self._arr[i]), i, 0
            r.close = lambda: None              # released by the group
            self.ctx.append(r)

    def _check(self, rc):
        self.ctx[0]._check(rc)

    def nccl_version(self):
        return self._lib.bihrt_multi_nccl_version()

    def broadcast(self):
        self._check(self._lib.bihrt_multi_broadcast(self.ctx[0]._ctx))
        return self

    def render(self, camera, w, h, spp=1, seed=1984, jitter=False):
        cam = camera if isinstance(camera, Camera) else Camera.from_array(camera)
        self._check(self._lib.bihrt_multi_render(self.ctx[0]._ctx, C.byref(cam), C.c_int32(w), C.c_int32(h), C.c_int32(spp),
                                                 C.c_uint64(seed), C.c_uint32(RENDER_JITTER if jitter else 0)))
        return self

    def sync(self):
        self._check(self._lib.bihrt_multi_sync(self.ctx[0]._ctx))

    def framebuffer(self):
        return self.ctx[0].framebuffer()

    def close(self):
        if getattr(self, "_arr", None) is not None and self._arr[0]:
            self._lib.bihrt_destroy_multi(self._arr, C.c_int32(self.ngpu))
            for r in self.ctx:
                r._ctx = C.c_void_p()
            self._arr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


from . import multi  # noqa: E402  (bihrt.multi: torch.distributed plumbing)
