"""Closest-point queries (bihrt_closest_point, csrc/closest.cu k_closest) on the GPU: the exported blob equals the CPU
restatement's word for word, and the kernel's records equal the restatement's walk (tests/closest_oracle.c) bit for
bit in all seven outputs, on parity and quality trees -- the walk itself equals brute force (tests/test_closest_oracle.py).
"""
import ctypes as C

import numpy as np
import pytest

from test_closest_oracle import (CAPS, SCENE_NAMES, assert_closest_equal, camera_for, identical, point_set, queries, radius_cases,
                                 scene_set)
from closest_oracle import CLOSEST_OUTS, blob_tree, closest  # noqa: F401  (closest: fixture)
from walk_oracle import FLT_MAX, assert_blob_equals, blob_of, tree  # noqa: F401  (tree: fixture)

pytestmark = pytest.mark.gpu


def build(renderer, tri, cap):
    """Builds tri in renderer as the parity tree (cap None) or the quality tree at leaf cap `cap`."""
    renderer.set_option("morton_bits", 30 if cap is None else 63)
    if cap is not None:
        renderer.set_option("leaf_cap", cap)
    renderer.load_models(tri).build()
    return renderer


def restated(tri, cap, oracle, tree):
    return tree(oracle.Bih(tri)) if cap is None else tree(tri, cap)


@pytest.mark.parametrize("name", SCENE_NAMES)
@pytest.mark.parametrize("cap", (None,) + CAPS)
def test_kernel_equals_walk(renderer, oracle, scenes, tree, closest, name, cap):
    tri = scene_set(scenes)[name]
    pt = restated(tri, cap, oracle, tree)
    build(renderer, tri, cap)
    assert_blob_equals(blob_of(renderer), pt, "%s %s" % (name, cap))
    pts = point_set(tri, pt, oracle, camera_for(name, scenes))
    q = queries(pts)
    assert_closest_equal(renderer.closest_point(q), closest(pt, q), "%s %s unbounded" % (name, cap))
    fin = np.isfinite(pts).all(1)
    full = closest(pt, q[fin], brute=True)
    rmax, _ = radius_cases(full["d2"], np.random.default_rng(4))
    q = queries(pts[fin], rmax)
    assert_closest_equal(renderer.closest_point(q), closest(pt, q), "%s %s radii" % (name, cap))


def test_large_scene(renderer, oracle, scenes, tree, closest):
    """1 M-triangle sphere, 200 k points (uniform in 1.2x the box, and near the surface), both tree kinds."""
    tri = scenes.displaced_sphere(scenes.SPHERE_NSEG["1m"])
    rng = np.random.default_rng(8)
    v = tri.reshape(-1, 3)
    lo, hi = v.min(0), v.max(0)
    c, ext = (lo + hi) * 0.5, hi - lo
    uni = rng.uniform(c - 0.6 * ext, c + 0.6 * ext, (100000, 3))
    t = tri.reshape(-1, 9)[rng.integers(0, len(tri), 100000)]
    w = rng.dirichlet((1, 1, 1), 100000)
    near = np.einsum("kj,kjc->kc", w, t.reshape(-1, 3, 3)) + rng.normal(scale=1e-3, size=(100000, 3))
    pts = np.concatenate([uni, near]).astype(np.float32)
    rmax = np.where(rng.random(len(pts)) < 0.5, np.inf, 0.01).astype(np.float32)
    for cap in (None, 4):
        pt = restated(tri, cap, oracle, tree)
        build(renderer, tri, cap)
        assert_blob_equals(blob_of(renderer), pt, "1m %s" % cap)
        q = queries(pts, rmax)
        got, want = renderer.closest_point(q), closest(pt, q)
        assert_closest_equal(got, want, "1m %s" % cap)
        assert (got["slot"] >= 0).mean() > 0.5


@pytest.mark.parametrize("case", ["one_triangle", "one_cell_parity", "one_leaf_quality"])
def test_single_leaf(renderer, oracle, scenes, tree, closest, case):
    tri, cap = {"one_triangle": (scenes.dodecahedron()[:1], None), "one_cell_parity": (identical(40), None),
                "one_leaf_quality": (scenes.dodecahedron()[:12], 16)}[case]
    pt = restated(tri, cap, oracle, tree)
    assert pt.nu == 1
    build(renderer, tri, cap)
    assert_blob_equals(blob_of(renderer), pt, case)
    rng = np.random.default_rng(1)
    pts = rng.uniform(-2, 2, (3000, 3)).astype(np.float32)
    rmax = np.where(rng.random(3000) < 0.5, np.inf, rng.uniform(0, 2, 3000)).astype(np.float32)
    q = queries(pts, rmax)
    got = renderer.closest_point(q)
    assert_closest_equal(got, closest(pt, q), case)
    assert_closest_equal(got, closest(pt, q, brute=True), case)


def test_refit_equals_brute_force_on_the_moved_mesh(renderer, oracle, scenes, tree, closest):
    """bihrt_refit (a parity-tree operation) keeps the topology and recomputes boxes and records: the query still equals brute
    force over the moved mesh's records."""
    tri = scenes.displaced_sphere(96)
    moved = scenes.displaced_sphere(96, phase=0.7)
    pt = restated(tri, None, oracle, tree)
    build(renderer, tri, None)
    assert_blob_equals(blob_of(renderer), pt, "before the refit")
    renderer.update_vertices(moved)
    renderer.refit()
    words = blob_of(renderer)
    bt = blob_tree(words)
    rec = bt.tris.view(np.float32)
    np.testing.assert_array_equal(rec[:, 0:3], moved.reshape(-1, 9)[bt.tris[:, 9], 0:3])     # the records hold the moved mesh
    rng = np.random.default_rng(6)
    pts = np.concatenate([rng.uniform(-1.5, 1.5, (3000, 3)), moved.reshape(-1, 3)[rng.integers(0, 3 * len(moved), 2000)]])
    q = queries(pts.astype(np.float32))
    got = renderer.closest_point(q)
    assert_closest_equal(got, closest(bt, q, brute=True), "refit")
    assert_closest_equal(got, closest(bt, q), "refit walk")


def test_replicas(renderer, oracle, scenes, tree, closest):
    import torch
    import bihrt
    tri = scenes.atrium(0.15)
    rng = np.random.default_rng(2)
    q = queries(rng.uniform(-1.5, 1.5, (20000, 3)).astype(np.float32))
    build(renderer, tri, 4)
    want = renderer.closest_point(q)
    nbytes = renderer.bih_blob_bytes()
    blob = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    renderer.bih_export(blob, nbytes)
    renderer.sync()
    r2 = bihrt.Renderer(0)
    r2.bih_import(blob, nbytes)
    assert_closest_equal(r2.closest_point(q), want, "imported")
    r2.close()
    # a replica adopted in place by a context that was not told the kind is refused
    r3 = bihrt.Renderer(0)
    ptr, nb = r3.bih_region(len(tri))
    src_ptr, _ = renderer.bih_region(len(tri))
    t_src = torch.as_tensor(bihrt.multi._CudaView(src_ptr, (nb,), "|u1"), device="cuda")
    t_dst = torch.as_tensor(bihrt.multi._CudaView(ptr, (nb,), "|u1"), device="cuda")
    renderer.sync()
    t_dst.copy_(t_src)
    torch.cuda.synchronize()
    r3.bih_adopt(len(tri))
    with pytest.raises(bihrt.BihrtError) as e:
        r3.closest_point(q)
    assert e.value.code == -4
    r3.set_option("morton_bits", 63)
    r3.bih_adopt(len(tri))
    assert_closest_equal(r3.closest_point(q), want, "adopted")
    r3.close()


def _raw(renderer, q4, outs, n=None):
    """bihrt_closest_point through ctypes with caller-owned outputs: returns the code"""
    import bihrt
    rec = bihrt.Closest(**{k: (bihrt._ptr(v) if v is not None else None) for k, v in outs.items()})
    n = len(q4) if n is None else n
    return renderer._lib.bihrt_closest_point(renderer._ctx, bihrt._ptr(q4), C.c_int64(n), C.byref(rec))


def test_watchdog_leaves_host_outputs_untouched(renderer, scenes):
    import bihrt
    tri = scenes.displaced_sphere(64)
    q = queries(np.random.default_rng(0).uniform(-1, 1, (4000, 3)).astype(np.float32))
    renderer.load_models(tri).build()
    want = renderer.closest_point(q)
    renderer.set_option("debug_trip_watchdog", 2)
    renderer.build()
    outs = {"d2": np.full(4000, 7.0, np.float32), "slot": np.full(4000, -7, np.int32), "q": np.full((4000, 3), 7.0, np.float32)}
    assert _raw(renderer, q, outs) == -6
    assert np.all(outs["d2"] == 7.0) and np.all(outs["slot"] == -7) and np.all(outs["q"] == 7.0)
    with pytest.raises(bihrt.BihrtError) as e:
        renderer.closest_point(q)
    assert e.value.code == -6
    renderer.set_option("debug_trip_watchdog", 0)
    renderer.build()
    renderer.sync()
    assert_closest_equal(renderer.closest_point(q), want)


def test_inputs_outputs_and_errors(renderer, scenes, oracle, tree, closest):
    import torch
    import bihrt
    tri = scenes.cornell_box()
    pt = tree(oracle.Bih(tri))
    rng = np.random.default_rng(3)
    pts = rng.uniform(-1.2, 1.2, (5000, 3)).astype(np.float32)
    rmax = np.where(rng.random(5000) < 0.5, np.inf, 0.3).astype(np.float32)
    q = bihrt.point_queries(pts, rmax)
    # no BIH yet
    with pytest.raises(bihrt.BihrtError) as e:
        renderer.closest_point(q)
    assert e.value.code == -4
    renderer.load_models(tri).build()
    want = closest(pt, q)
    # numpy in, numpy out
    assert_closest_equal(renderer.closest_point(q), want, "host")
    # torch in (device), torch out on the device; point_queries on torch
    qd = bihrt.point_queries(torch.from_numpy(pts).cuda(), torch.from_numpy(rmax).cuda())
    assert torch.equal(qd.cpu(), torch.from_numpy(q))
    got = renderer.closest_point(qd)
    for k in CLOSEST_OUTS:
        assert got[k].is_cuda
    assert_closest_equal({k: v.cpu().numpy() for k, v in got.items()}, want, "device")
    # on a side stream of torch's: ordered by wait_torch / torch_wait
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        qs = bihrt.point_queries(torch.from_numpy(pts).cuda(), torch.from_numpy(rmax).cuda())
        got = renderer.closest_point(qs, outputs=("d2", "slot"))
        d2 = got["d2"].cpu().numpy()
    np.testing.assert_array_equal(d2.view(np.uint32), want["d2"].view(np.uint32))
    # each output alone; host points with device outputs and device points with host outputs
    qd_c = qd.contiguous()
    for k in CLOSEST_OUTS:
        r = renderer.closest_point(q, outputs=(k,))
        assert list(r) == [k]
        np.testing.assert_array_equal(np.ascontiguousarray(r[k]).view(np.uint32) if r[k].dtype == np.float32 else r[k],
                                      want[k].view(np.uint32) if want[k].dtype == np.float32 else want[k], err_msg=k)
        dev = torch.empty(want[k].shape, dtype=torch.int32 if k in ("slot", "prim") else torch.float32, device="cuda")
        assert _raw(renderer, q, {k: dev}) == 0
        renderer.sync()
        host = np.empty_like(want[k])
        assert _raw(renderer, qd_c, {k: host}) == 0
        np.testing.assert_array_equal(dev.cpu().numpy(), host, err_msg=k)
        np.testing.assert_array_equal(host.view(np.uint32) if host.dtype == np.float32 else host,
                                      want[k].view(np.uint32) if want[k].dtype == np.float32 else want[k], err_msg=k)
    with pytest.raises(ValueError):
        renderer.closest_point(q, outputs=("t",))
    # errors
    lib, ctx = renderer._lib, renderer._ctx
    assert lib.bihrt_closest_point(ctx, bihrt._ptr(q), C.c_int64(10), None) == -1                      # out == NULL
    assert _raw(renderer, q, {"d2": np.empty(10, np.float32)}, n=-1) == -1                          # n < 0
    assert lib.bihrt_closest_point(ctx, None, C.c_int64(10), C.byref(bihrt.Closest())) == -1        # pts == NULL, n > 0
    assert lib.bihrt_closest_point(ctx, None, C.c_int64(0), C.byref(bihrt.Closest())) == 0          # nothing to do
    assert _raw(renderer, q, {}, n=(1 << 32) - (1 << 24)) == -1                                      # 32-bit work counter
    flat = torch.zeros(4 * 64 + 1, dtype=torch.float32, device="cuda")
    assert lib.bihrt_closest_point(ctx, C.c_void_p(flat.data_ptr() + 4), C.c_int64(64), C.byref(bihrt.Closest())) == -1   # misaligned
    assert "aligned" in lib.bihrt_last_error(ctx).decode()
    # a miss record
    r = renderer.closest_point(bihrt.point_queries(np.array([[5.0, 5.0, 5.0], [0.0, 0.0, 0.0]], np.float32), np.array([0.1, np.nan], np.float32)))
    assert np.all(r["d2"] == FLT_MAX) and np.all(r["slot"] == -1) and np.all(r["prim"] == -1)
    assert np.all(r["u"] == 0) and np.all(r["v"] == 0) and np.all(r["q"] == 0) and np.all(r["ng"] == 0)
