"""The CPU restatement the GPU winding-number tests are pinned to (tests/winding_oracle.c).

The `winding` fixture compiles it once per session and returns a Winding: winding.table(tree) is the far-field table of a tree
that holds the exported blob's words (a walk_oracle Tree or closest_oracle.blob_tree), winding(tree, queries4, beta) the walk
(or with brute=True the exact sum over every slot in slot order), winding.f64(tri9, points) the float64 solid-angle sum over
the input triangles, and winding.atan2 the library's atan2 on arrays.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
WREC = 32          # floats per child record of the table (csrc/bihrt_internal.cuh WTAB_FLOATS)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def build_lib(out_dir):
    """Compiles tests/winding_oracle.c into out_dir; returns the loaded library."""
    out = os.path.join(str(out_dir), "libwinding_oracle.so")
    cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
    subprocess.check_call([cc, "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-fvisibility=hidden", "-std=c11", "-shared",
                           "-o", out, os.path.join(HERE, "winding_oracle.c"), "-lm"])
    lib = C.CDLL(out)
    lib.orc_atan2.restype = C.c_float
    lib.orc_atan2.argtypes = [C.c_float, C.c_float]
    return lib


def _words(tree):
    hdr, nodes, tris = (np.ascontiguousarray(x, np.uint32) for x in (tree.hdr, tree.nodes, tree.tris))
    return hdr, (nodes if nodes.size else np.zeros((1, 16), np.uint32)), (tris if tris.size else np.zeros((1, 12), np.uint32))


class Winding:
    def __init__(self, lib):
        self.lib = lib
        self._tables = {}

    def table(self, tree):
        """(node slots, 2, WREC) float32: per node slot, the records of its two children (zeros where the tree does not
        reach).  Cached per tree object."""
        key = id(tree)
        if key not in self._tables or self._tables[key][0] is not tree:
            hdr, nodes, tris = _words(tree)
            tab = np.zeros((len(nodes), 2, WREC), np.float32)
            self.lib.orc_wtab(_p(hdr), _p(nodes), _p(tris), _p(tab))
            self._tables[key] = (tree, tab)
        return self._tables[key][1]

    def __call__(self, tree, queries4, beta=2.0, brute=False):
        """Winding numbers of queries4 ((N,4) p.xyz, rmax ignored) on tree's blob words.  Returns (w (N,) float32, counters
        {nodes, far, exact}: totals of internal nodes stepped, far-field terms and exact triangle terms)."""
        q4 = np.ascontiguousarray(queries4, np.float32).reshape(-1, 4)
        hdr, nodes, tris = _words(tree)
        tab = self.table(tree)
        w = np.empty(len(q4), np.float32)
        cnt = np.zeros(3, np.uint64)
        b2 = np.float32(beta) * np.float32(beta) if np.isfinite(beta) else np.float32(np.inf)
        self.lib.orc_winding(_p(hdr), _p(nodes), _p(tris), _p(tab), C.c_int(int(brute)), C.c_float(b2), _p(q4),
                             C.c_int64(len(q4)), _p(w), _p(cnt), C.c_int(0))
        return w, {"nodes": int(cnt[0]), "far": int(cnt[1]), "exact": int(cnt[2])}

    def f64(self, tri9, points):
        """float64 winding numbers of points (N,3) from the input triangles tri9 (M,9)"""
        t = np.ascontiguousarray(tri9, np.float32).reshape(-1, 9)
        p = np.ascontiguousarray(points, np.float32).reshape(-1, 3)
        out = np.empty(len(p), np.float64)
        self.lib.orc_winding64(_p(t), C.c_int64(len(t)), _p(p), C.c_int64(len(p)), _p(out), C.c_int(0))
        return out

    def atan2(self, y, x):
        y, x = np.ascontiguousarray(y, np.float32), np.ascontiguousarray(x, np.float32)
        out = np.empty(len(y), np.float32)
        self.lib.orc_atan2_many(_p(y), _p(x), _p(out), C.c_int64(len(y)))
        return out


@pytest.fixture(scope="session")
def winding(tmp_path_factory):
    """A Winding on the session's build of tests/winding_oracle.c."""
    return Winding(build_lib(tmp_path_factory.mktemp("winding_oracle")))
