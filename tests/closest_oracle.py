"""The CPU restatement the GPU closest-point tests are pinned to (tests/closest_oracle.c).

The `closest` fixture compiles it once per session and returns closest(tree, queries4, brute=False, margin_scale=CLOSEST_EPS),
which runs the kernel's walk (or brute force over every slot) on any tree that holds the exported blob's words: a walk_oracle
Tree (the parity tree of an oracle.Bih or the quality tree of a leaf cap) or an exported blob itself (blob_tree).
"""
import ctypes as C
import os
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
CLOSEST_OUTS = ("d2", "u", "v", "slot", "prim", "q", "ng")
CLOSEST_EPS = 2.0 ** -16        # csrc/closest.cu: the boxes' margin is this times the query's largest coordinate magnitude


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def build_lib(out_dir):
    """Compiles tests/closest_oracle.c into out_dir; returns the loaded library."""
    out = os.path.join(str(out_dir), "libclosest_oracle.so")
    cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
    subprocess.check_call([cc, "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-fvisibility=hidden", "-std=c11", "-shared",
                           "-o", out, os.path.join(HERE, "closest_oracle.c"), "-lm"])
    return C.CDLL(out)


def run_closest(lib, tree, queries4, brute=False, margin_scale=CLOSEST_EPS):
    """Closest-point queries (bihrt_closest_point) on tree's blob words (hdr, nodes, tris): queries4 (N,4) p.xyz rmax.
    brute=False is the kernel's walk (its margin unless margin_scale says otherwise), brute=True every slot in slot order.
    Returns the record {d2, u, v, slot, prim, q, ng} and counters (total node fetches, distance evaluations, deepest stack)."""
    q4 = np.ascontiguousarray(queries4, np.float32).reshape(-1, 4)
    nq = len(q4)
    r = {"d2": np.empty(nq, np.float32), "u": np.empty(nq, np.float32), "v": np.empty(nq, np.float32),
         "slot": np.empty(nq, np.int32), "prim": np.empty(nq, np.int32), "q": np.empty((nq, 3), np.float32),
         "ng": np.empty((nq, 3), np.float32)}
    cnt = np.zeros(3, np.uint64)
    hdr, nodes, tris = (np.ascontiguousarray(x, np.uint32) for x in (tree.hdr, tree.nodes, tree.tris))
    nodes = nodes if nodes.size else np.zeros(16, np.uint32)
    lib.orc_closest(_p(hdr), _p(nodes), _p(tris), C.c_int(int(brute)), C.c_float(margin_scale), _p(q4), C.c_int64(nq),
                    *[_p(r[k]) for k in CLOSEST_OUTS], _p(cnt), C.c_int(0))
    r["counters"] = {"nodes": int(cnt[0]), "tris": int(cnt[1]), "max_stack": int(cnt[2])}
    return r


def blob_tree(words):
    """The header, node slots and triangle records of exported blob words (n from the header)."""
    words = np.asarray(words, np.uint32)
    n = int(words[0])
    nn = (len(words) - 16 - 12 * n) // 16
    return SimpleNamespace(hdr=words[:16].copy(), nodes=words[16:16 + 16 * nn].reshape(nn, 16).copy(),
                           tris=words[16 + 16 * nn:].reshape(n, 12).copy(), n=n, nu=int(words[1]))


@pytest.fixture(scope="session")
def closest(tmp_path_factory):
    """closest(tree, queries4, brute=False, margin_scale=CLOSEST_EPS) -> run_closest on the session's build of
    tests/closest_oracle.c."""
    lib = build_lib(tmp_path_factory.mktemp("closest_oracle"))
    return lambda tree, queries4, brute=False, margin_scale=CLOSEST_EPS: run_closest(lib, tree, queries4, brute, margin_scale)
