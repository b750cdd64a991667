"""The CPU restatement the GPU multi-hit ray query tests are pinned to (tests/intersect_k_oracle.c).

The `intersect_k` fixture compiles it once per session and returns intersect_k(tree, rays8, k, total=False, two_sided=False,
brute=False), which runs the kernel's walk with its list (or brute force over every slot) on any tree that holds the exported
blob's words, as walk_oracle's Tree.walk does.  With total=True the walk cuts at the interval's upper end only and counts every
accepted triangle, as the kernel does when its caller asks for the total.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from walk_oracle import ORACLE_DIR, OUTS

HERE = os.path.dirname(os.path.abspath(__file__))
K_OUTS = OUTS + ("count", "total")
K_MAX = 64                      # include/bihrt.h: BIHRT_INTERSECT_K_MAX


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def build_lib(out_dir):
    """Compiles tests/intersect_k_oracle.c (which includes walk_oracle.c) into out_dir; returns the loaded library."""
    out = os.path.join(str(out_dir), "libintersect_k_oracle.so")
    cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
    subprocess.check_call([cc, "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-fvisibility=hidden", "-std=c11", "-shared",
                           "-I", HERE, "-I", ORACLE_DIR, "-o", out, os.path.join(HERE, "intersect_k_oracle.c"), "-lm"])
    return C.CDLL(out)


def run_intersect_k(lib, tree, rays8, k, total=False, two_sided=False, brute=False):
    """Multi-hit ray queries (bihrt_intersect_k) on tree's blob words: rays8 (N,8) o.xyz tmin d.xyz tmax, 0 <= k <= K_MAX.
    Returns the rows {t, u, v, slot, prim (N,k), ng (N,k,3)}, count (N,), total (N,) when total=True, and counters (total node
    fetches, triangle tests, deepest stack)."""
    r8 = np.ascontiguousarray(rays8, np.float32).reshape(-1, 8)
    nr = len(r8)
    r = {o: np.empty((nr, k), np.int32 if o in ("slot", "prim") else np.float32) for o in ("t", "u", "v", "slot", "prim")}
    r.update(ng=np.empty((nr, k, 3), np.float32), count=np.empty(nr, np.int32))
    if total:
        r["total"] = np.empty(nr, np.int32)
    cnt = np.zeros(3, np.uint64)
    tri9 = np.ascontiguousarray(tree.tri9, np.float32)
    hdr, nodes, tris = (np.ascontiguousarray(x, np.uint32) for x in (tree.hdr, tree.nodes, tree.tris))
    nodes = nodes if nodes.size else np.zeros(16, np.uint32)
    lib.orc_walk_k(_p(tri9), _p(hdr), _p(nodes), _p(tris), C.c_int(int(brute)), C.c_int(int(two_sided)), C.c_int(k),
                   C.c_int(int(total)), _p(r8), C.c_int64(nr), *[_p(r.get(o)) for o in K_OUTS], _p(cnt), C.c_int(0))
    r["counters"] = {"nodes": int(cnt[0]), "tris": int(cnt[1]), "max_stack": int(cnt[2])}
    return r


@pytest.fixture(scope="session")
def intersect_k(tmp_path_factory):
    """intersect_k(tree, rays8, k, total=False, two_sided=False, brute=False) -> run_intersect_k on the session's build of
    tests/intersect_k_oracle.c."""
    lib = build_lib(tmp_path_factory.mktemp("intersect_k_oracle"))
    return lambda tree, rays8, k, total=False, two_sided=False, brute=False: run_intersect_k(
        lib, tree, rays8, k, total, two_sided, brute)
