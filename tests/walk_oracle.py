"""The CPU restatement every GPU trace test is pinned to, and the helpers those tests share.

tests/walk_oracle.c restates the walk of every trace entry point (csrc/trace.cu, k_trace) on the blob bihrt_bih_export
writes, for the oracle's parity tree and for the quality-mode tree alike.  The `tree` fixture compiles it once per session
and builds a Tree from an oracle.Bih (parity) or from triangles and a leaf cap (quality); Tree.walk and Tree.brute run it.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.join(os.path.dirname(HERE), "oracle")
FLT_MAX = np.float32(np.finfo(np.float32).max)
EXITS = {"closest": 0, "first": 1, "any": 2}
OUTS = ("t", "u", "v", "slot", "prim", "ng")


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class Tree:
    """A tree as the exported blob holds it: header (16 words), node slots ((nn, 16) words, nn = nu - 1 for a parity tree and
    n - 1 for a quality tree; `reach` marks the ones the tree uses) and triangle records ((n, 12) words).  A quality tree also
    has its sorted keys and its depth in nodes."""

    def __init__(self, lib, src, cap=None):
        self.lib = lib
        if cap is None:                                     # src: an oracle.Bih
            ob = src
            self.tri9, self.n, self.nu = ob.tri9, ob.n, ob.nu
            nn = max(ob.nu - 1, 0)
            self.hdr, self.nodes = np.zeros(16, np.uint32), np.zeros((max(nn, 1), 16), np.uint32)
            self.tris = np.zeros((max(ob.n, 1), 12), np.uint32)
            keep = [np.ascontiguousarray(x) for x in (ob.tris_idx, ob.cnt, ob.first, ob.clip, ob.axis, ob.is_leaf, ob.children)]
            lib.orc_parity_blob(_p(ob.tri9), C.c_int64(ob.n), C.c_int64(ob.nu), *[_p(k) for k in keep], _p(ob.scene_lo),
                                _p(ob.scene_hi), _p(self.hdr), _p(self.nodes), _p(self.tris))
            self.nodes, self.tris, self.reach = self.nodes[:nn], self.tris[:ob.n], np.ones(nn, bool)
            return
        self.tri9 = np.ascontiguousarray(src, np.float32).reshape(-1, 9)
        n = self.n = len(self.tri9)
        self.cap = cap
        self.hdr = np.zeros(16, np.uint32)
        self.nodes = np.zeros((max(n - 1, 1), 16), np.uint32)
        self.reach = np.zeros(max(n - 1, 1), np.uint8)
        self.tris = np.zeros((max(n, 1), 12), np.uint32)
        self.keys = np.zeros(max(n, 1), np.uint64)
        self.depth = lib.orc_q_build(_p(self.tri9), C.c_int64(n), C.c_int(cap), _p(self.hdr), _p(self.nodes), _p(self.reach),
                                     _p(self.tris), _p(self.keys))
        self.nodes, self.reach = self.nodes[:max(n - 1, 0)], self.reach[:max(n - 1, 0)].astype(bool)
        self.tris, self.keys = self.tris[:n], self.keys[:n]
        self.nu = int(self.hdr[1])

    def walk(self, rays, exit="closest", tmin=0.0, tmax=np.inf, two_sided=False, ht_max=FLT_MAX):
        """rays: (N,6) with the interval (tmin, tmax), or (N,8).  h.t starts at min(tmax, ht_max): FLT_MAX as bihrt_intersect,
        bihrt_trace and the renders start it; np.inf for tmax as given, as bihrt_trace_any does.  Returns the record
        {t, u, v, slot, prim, ng} and counters (total nodes, triangle tests, deepest stack) and stack (each ray's deepest)."""
        return self._run(False, rays, exit, tmin, tmax, two_sided, ht_max)

    def brute(self, rays, tmin=0.0, tmax=np.inf, two_sided=False, ht_max=FLT_MAX):
        """Every slot in slot order, the closest accepted triangle; arguments and result as walk's."""
        return self._run(True, rays, "closest", tmin, tmax, two_sided, ht_max)

    def _run(self, brute, rays, exit, tmin, tmax, two_sided, ht_max):
        r8 = np.ascontiguousarray(rays, np.float32)
        r8 = r8 if r8.ndim == 2 and r8.shape[1] == 8 else rays8(r8, tmin, tmax)
        nr = len(r8)
        r = {"t": np.empty(nr, np.float32), "u": np.empty(nr, np.float32), "v": np.empty(nr, np.float32),
             "slot": np.empty(nr, np.int32), "prim": np.empty(nr, np.int32), "ng": np.empty((nr, 3), np.float32),
             "stack": np.empty(nr, np.int32)}
        cnt = np.zeros(3, np.uint64)
        self.lib.orc_walk(_p(self.tri9), _p(self.hdr), _p(self.nodes), _p(self.tris), C.c_int(int(brute)), C.c_int(EXITS[exit]),
                          C.c_int(int(two_sided)), C.c_float(ht_max), _p(r8), C.c_int64(nr),
                          *[_p(r[k]) for k in OUTS + ("stack",)], _p(cnt), C.c_int(0))
        r["counters"] = {"nodes": int(cnt[0]), "tris": int(cnt[1]), "max_stack": int(cnt[2])}
        return r


@pytest.fixture(scope="session")
def tree(tmp_path_factory):
    """Builds tests/walk_oracle.c (the oracle's source plus both blob builders and the walk) into a temporary directory;
    returns tree(bih) -> the parity Tree of an oracle.Bih, tree(tri, cap) -> the quality Tree of `tri` at leaf cap `cap`."""
    out = str(tmp_path_factory.mktemp("walk_oracle") / "libwalk_oracle.so")
    cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
    subprocess.check_call([cc, "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-fvisibility=hidden", "-std=c11",
                           "-shared", "-I" + ORACLE_DIR, "-o", out, os.path.join(HERE, "walk_oracle.c"), "-lm"])
    lib = C.CDLL(out)
    lib.orc_q_build.restype = C.c_int
    return lambda src, cap=None: Tree(lib, src, cap)


# ------------------------------------------------------------------------------------------------ rays and records

def rays8(rays6, tmin=0.0, tmax=np.inf):
    """(N,8) o.xyz tmin d.xyz tmax from (N,6) rays and scalar or per-ray bounds (bihrt.interval_rays on numpy arrays)."""
    from bihrt import interval_rays
    return interval_rays(np.asarray(rays6, np.float32), tmin, tmax)


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32) if a.dtype == np.float32 else a


def assert_records_equal(got, want, outputs=OUTS, msg=""):
    for k in outputs:
        np.testing.assert_array_equal(bits(got[k]), bits(want[k]), err_msg="%s %s" % (msg, k))


def mt(tri9, prim, rays6, two_sided=False):
    """Moller-Trumbore of ray i against triangle prim[i] in numpy binary32, the reference's operation order
    (R/src/CUDAKernels.cu:17-50), with the det test det >= 1e-6 or, two-sided, |det| >= 1e-6: returns ok, det, t, u, v -- an
    independent restatement of what a hit record holds."""
    f = np.float32
    tri = tri9.reshape(-1, 9)[prim].astype(f)
    v0, v1, v2 = tri[:, 0:3], tri[:, 3:6], tri[:, 6:9]
    o, d = rays6[:, 0:3].astype(f), rays6[:, 3:6].astype(f)
    e1, e2 = v1 - v0, v2 - v0

    def cross(a, b):
        return np.stack([a[:, 1] * b[:, 2] - b[:, 1] * a[:, 2], a[:, 2] * b[:, 0] - b[:, 2] * a[:, 0],
                         a[:, 0] * b[:, 1] - b[:, 0] * a[:, 1]], 1)

    def dot(a, b):
        return (a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1]) + a[:, 2] * b[:, 2]
    p = cross(d, e2)
    det = dot(e1, p)
    ok = (np.abs(det.astype(np.float64)) if two_sided else det.astype(np.float64)) >= 1e-6
    with np.errstate(all="ignore"):
        inv = (1.0 / det.astype(np.float64)).astype(f)
        tv = o - v0
        u = dot(tv, p) * inv
        q = cross(tv, e1)
        v = dot(d, q) * inv
        t = dot(e2, q) * inv
    ok &= ~((u < 0) | (u > 1) | (v < 0) | ((u + v) > 1))
    return ok, det, t, u, v


def degenerate_rays(scenes, rng=None):
    """Zero direction components, origins on grid planes and on the scene box, diagonal directions, on the Cornell box plus a
    small sphere: returns tri, rays.  The rays are drawn from `rng` (default: seeded with 7)."""
    tri = np.concatenate([scenes.cornell_box(), scenes.displaced_sphere(24) * 0.3])
    rng = np.random.default_rng(7) if rng is None else rng
    n = 20000
    o = rng.uniform(-1.2, 1.2, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    which = rng.integers(0, 7, n)
    d[which == 0, 0] = 0.0
    d[which == 1, 1] = 0.0
    d[which == 2, 2] = 0.0
    d[which == 3, :2] = 0.0
    o[which == 4] = np.round(o[which == 4] * 4) / 4
    d[which == 5] = np.sign(d[which == 5])
    o[which == 6, 0] = -1.0
    d[(which == 3) & (d[:, 2] == 0), 2] = 1.0
    return tri, np.concatenate([o, d], 1).astype(np.float32)


def assorted_intervals(t0, seed):
    """Per-ray (tmin, tmax) drawn from: tmin in {0, a random fraction of the closest t, exactly the closest t, negative},
    tmax in {+inf, FLT_MAX, random, below the hit, NaN, <= tmin}; plus NaN tmin on a few rays."""
    rng = np.random.default_rng(seed)
    n = len(t0)
    hit = t0 < FLT_MAX
    ref = np.where(hit, t0, np.float32(4.0)).astype(np.float32)         # a scale for the misses
    k = rng.integers(0, 4, n)
    tmin = np.select([k == 0, k == 1, k == 2, k == 3],
                     [np.zeros(n), rng.uniform(0, 1, n) * ref, ref, -rng.uniform(0, 10, n)]).astype(np.float32)
    j = rng.integers(0, 6, n)
    tmax = np.select([j == 0, j == 1, j == 2, j == 3, j == 4, j == 5],
                     [np.full(n, np.inf), np.full(n, FLT_MAX), rng.uniform(0, 3, n) * ref, ref * np.float32(0.999),
                      np.full(n, np.nan), tmin - rng.uniform(0, 1, n) * (rng.integers(0, 2, n))]).astype(np.float32)
    tmin[rng.random(n) < 0.01] = np.nan
    return tmin, tmax


# ------------------------------------------------------------------------------------------------ blobs

def blob_of(renderer):
    """The exported BIH blob as host uint32 words."""
    import torch
    nbytes = renderer.bih_blob_bytes()
    blob = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    renderer.bih_export(blob, nbytes)
    renderer.sync()
    return blob.cpu().numpy().view(np.uint32)


def assert_blob_equals(words, tree, what=""):
    """Header, every node the tree reaches and every triangle record equal the restatement: bytes, except the scene box, the
    planes and the children boxes, which compare as floats (==, so that -0 and +0, which no ray tells apart, are equal)."""
    n, nn = tree.n, len(tree.nodes)
    assert len(words) == 16 + 16 * nn + 12 * n, what
    hdr, nodes, tris = words[:16], words[16:16 + 16 * nn].reshape(nn, 16), words[16 + 16 * nn:].reshape(n, 12)
    np.testing.assert_array_equal(hdr[[0, 1, 8, 9, 10]], tree.hdr[[0, 1, 8, 9, 10]], err_msg="%s header" % what)
    np.testing.assert_array_equal(hdr[2:8].view(np.float32), tree.hdr[2:8].view(np.float32), err_msg="%s scene box" % what)
    got, want = nodes[tree.reach], tree.nodes[tree.reach]
    np.testing.assert_array_equal(got[:, 2:4], want[:, 2:4], err_msg="%s child references" % what)
    fl = [0, 1] + list(range(4, 16))
    np.testing.assert_array_equal(got[:, fl].view(np.float32), want[:, fl].view(np.float32), err_msg="%s planes / boxes" % what)
    np.testing.assert_array_equal(tris, tree.tris, err_msg="%s triangle records" % what)
