"""The CPU restatement the GPU k-nearest-triangle tests are pinned to (tests/closest_k_oracle.c).

The `closest_k` fixture compiles it once per session and returns closest_k(tree, queries4, k, total=False, brute=False,
margin_scale=CLOSEST_EPS), which runs the kernel's walk (or brute force over every slot) on any tree that holds the exported
blob's words, as closest_oracle's `closest` does.  With total=True the walk prunes at the radius only and counts every
candidate, as the kernel does when its caller asks for the total.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from closest_oracle import CLOSEST_EPS, CLOSEST_OUTS

HERE = os.path.dirname(os.path.abspath(__file__))
CLOSEST_K_OUTS = CLOSEST_OUTS + ("count", "total")
K_MAX = 64                      # include/bihrt.h: BIHRT_CLOSEST_K_MAX


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def build_lib(out_dir):
    """Compiles tests/closest_k_oracle.c (which includes closest_oracle.c) into out_dir; returns the loaded library."""
    out = os.path.join(str(out_dir), "libclosest_k_oracle.so")
    cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
    subprocess.check_call([cc, "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-fvisibility=hidden", "-std=c11", "-shared",
                           "-I", HERE, "-o", out, os.path.join(HERE, "closest_k_oracle.c"), "-lm"])
    return C.CDLL(out)


def run_closest_k(lib, tree, queries4, k, total=False, brute=False, margin_scale=CLOSEST_EPS):
    """k-nearest-triangle queries (bihrt_closest_k) on tree's blob words: queries4 (N,4) p.xyz rmax, 0 <= k <= K_MAX.
    Returns the rows {d2, u, v, slot, prim (N,k), q, ng (N,k,3)}, count (N,), total (N,) when total=True, and counters (total
    node fetches, distance evaluations, deepest stack)."""
    q4 = np.ascontiguousarray(queries4, np.float32).reshape(-1, 4)
    nq = len(q4)
    r = {o: np.empty((nq, k), np.int32 if o in ("slot", "prim") else np.float32) for o in ("d2", "u", "v", "slot", "prim")}
    r.update(q=np.empty((nq, k, 3), np.float32), ng=np.empty((nq, k, 3), np.float32), count=np.empty(nq, np.int32))
    if total:
        r["total"] = np.empty(nq, np.int32)
    cnt = np.zeros(3, np.uint64)
    hdr, nodes, tris = (np.ascontiguousarray(x, np.uint32) for x in (tree.hdr, tree.nodes, tree.tris))
    nodes = nodes if nodes.size else np.zeros(16, np.uint32)
    lib.orc_closest_k(_p(hdr), _p(nodes), _p(tris), C.c_int(int(brute)), C.c_float(margin_scale), C.c_int(k), _p(q4),
                      C.c_int64(nq), *[_p(r.get(o)) for o in CLOSEST_K_OUTS], _p(cnt), C.c_int(0))
    r["counters"] = {"nodes": int(cnt[0]), "tris": int(cnt[1]), "max_stack": int(cnt[2])}
    return r


@pytest.fixture(scope="session")
def closest_k(tmp_path_factory):
    """closest_k(tree, queries4, k, total=False, brute=False, margin_scale=CLOSEST_EPS) -> run_closest_k on the session's build
    of tests/closest_k_oracle.c."""
    lib = build_lib(tmp_path_factory.mktemp("closest_k_oracle"))
    return lambda tree, queries4, k, total=False, brute=False, margin_scale=CLOSEST_EPS: run_closest_k(
        lib, tree, queries4, k, total, brute, margin_scale)
