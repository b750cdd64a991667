"""k-nearest-triangle queries (bihrt_closest_k, csrc/closest.cu k_closest_k) on the GPU: the kernel's rows, counts and totals
equal the restatement's walk (tests/closest_k_oracle.c) bit for bit, on parity and quality trees, for k in {1, 3, 8, 64}, with
and without the total -- the walk itself equals brute force (tests/test_closest_k_oracle.py).  At k = 1 the rows are
bihrt_closest_point's records.
"""
import ctypes as C

import numpy as np
import pytest

from closest_k_oracle import CLOSEST_K_OUTS, K_MAX, closest_k  # noqa: F401  (closest_k: fixture)
from closest_oracle import CLOSEST_OUTS, blob_tree
from test_closest_k_oracle import KS, RADIUS_COLUMN, assert_k_equal, k_points
from test_closest_oracle import CAPS, SCENE_NAMES, camera_for, identical, queries, radius_cases, scene_set
from test_gpu_closest import build, restated
from walk_oracle import FLT_MAX, assert_blob_equals, bits, blob_of, tree  # noqa: F401  (tree: fixture)

pytestmark = pytest.mark.gpu

ROWS = CLOSEST_OUTS + ("count",)


def gpu_k(renderer, q, k, total=False):
    return renderer.closest_k(q, k, outputs=ROWS + (("total",) if total else ()))


@pytest.mark.parametrize("name", SCENE_NAMES)
@pytest.mark.parametrize("cap", (None,) + CAPS)
def test_kernel_equals_walk(renderer, oracle, scenes, tree, closest_k, name, cap):
    tri = scene_set(scenes)[name]
    pt = restated(tri, cap, oracle, tree)
    build(renderer, tri, cap)
    assert_blob_equals(blob_of(renderer), pt, "%s %s" % (name, cap))
    pts = k_points(tri, pt, oracle, camera_for(name, scenes))
    q = queries(pts)
    fin = np.isfinite(pts).all(1)
    nearest = closest_k(pt, q[fin], RADIUS_COLUMN + 1)["d2"][:, RADIUS_COLUMN]
    rmax, _ = radius_cases(nearest, np.random.default_rng(4))
    for case, qq in (("unbounded", q), ("radii", queries(pts[fin], rmax))):
        for k in KS:
            for total in (False, True):
                assert_k_equal(gpu_k(renderer, qq, k, total), closest_k(pt, qq, k, total=total),
                               "%s %s %s k=%d total=%s" % (name, cap, case, k, total))


@pytest.mark.parametrize("name", ["cornell", "sphere", "needles", "identical", "coplanar"])
def test_k1_rows_are_closest_point_records(renderer, oracle, scenes, tree, name):
    tri = scene_set(scenes)[name]
    for cap in (None, 4):
        pt = restated(tri, cap, oracle, tree)
        build(renderer, tri, cap)
        pts = k_points(tri, pt, oracle, camera_for(name, scenes), seed=2)
        rmax = np.where(np.random.default_rng(1).random(len(pts)) < 0.5, np.inf, 0.05).astype(np.float32)
        for qq in (queries(pts), queries(pts, rmax)):
            a, b = renderer.closest_k(qq, 1), renderer.closest_point(qq)
            for o in CLOSEST_OUTS:
                np.testing.assert_array_equal(bits(a[o][:, 0]), bits(b[o]), err_msg="%s %s %s" % (name, cap, o))
            np.testing.assert_array_equal(a["count"], (b["slot"] >= 0).astype(np.int32))


def test_large_scene(renderer, oracle, scenes, tree, closest_k):
    """1 M-triangle sphere, 200 k points (uniform in 1.2x the box, and near the surface), both tree kinds: k = 16 with half the
    radii unbounded and half 0.01; k = 64 with the total at rmax = 0.01 (an unbounded total would visit every leaf)."""
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
        got = gpu_k(renderer, q, 16)
        assert_k_equal(got, closest_k(pt, q, 16), "1m %s k=16" % cap)
        assert (got["count"] == 16).mean() > 0.4
        q = queries(pts, 0.01)
        got = gpu_k(renderer, q, 64, total=True)
        assert_k_equal(got, closest_k(pt, q, 64, total=True), "1m %s k=64 total" % cap)
        assert (got["total"] > 0).mean() > 0.4


@pytest.mark.parametrize("case", ["one_triangle", "one_cell_parity", "one_leaf_quality"])
def test_single_leaf(renderer, oracle, scenes, tree, closest_k, case):
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
    for k in (1, 8):
        for total in (False, True):
            got = gpu_k(renderer, q, k, total)
            assert_k_equal(got, closest_k(pt, q, k, total=total), "%s k=%d total=%s walk" % (case, k, total))
            assert_k_equal(got, closest_k(pt, q, k, total=True, brute=True), "%s k=%d total=%s brute" % (case, k, total))


def test_refit_equals_brute_force_on_the_moved_mesh(renderer, oracle, scenes, tree, closest_k):
    tri = scenes.displaced_sphere(96)
    moved = scenes.displaced_sphere(96, phase=0.7)
    build(renderer, tri, None)
    renderer.update_vertices(moved)
    renderer.refit()
    bt = blob_tree(blob_of(renderer))
    np.testing.assert_array_equal(bt.tris.view(np.float32)[:, 0:3], moved.reshape(-1, 9)[bt.tris[:, 9], 0:3])
    rng = np.random.default_rng(6)
    pts = np.concatenate([rng.uniform(-1.5, 1.5, (3000, 3)), moved.reshape(-1, 3)[rng.integers(0, 3 * len(moved), 2000)]])
    rmax = np.where(rng.random(len(pts)) < 0.5, np.inf, 0.05).astype(np.float32)
    q = queries(pts.astype(np.float32), rmax)
    for k in (1, 8):
        for total in (False, True):
            assert_k_equal(gpu_k(renderer, q, k, total), closest_k(bt, q, k, total=True, brute=True),
                           "refit k=%d total=%s" % (k, total))


def test_replicas(renderer, scenes):
    import torch
    import bihrt
    tri = scenes.atrium(0.15)
    rng = np.random.default_rng(2)
    q = queries(rng.uniform(-1.5, 1.5, (20000, 3)).astype(np.float32), 0.2)
    build(renderer, tri, 4)
    want = gpu_k(renderer, q, 8, total=True)
    nbytes = renderer.bih_blob_bytes()
    blob = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    renderer.bih_export(blob, nbytes)
    renderer.sync()
    r2 = bihrt.Renderer(0)
    r2.bih_import(blob, nbytes)
    assert_k_equal(gpu_k(r2, q, 8, total=True), want, "imported")
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
        gpu_k(r3, q, 8, total=True)
    assert e.value.code == -4
    r3.set_option("morton_bits", 63)
    r3.bih_adopt(len(tri))
    assert_k_equal(gpu_k(r3, q, 8, total=True), want, "adopted")
    r3.close()


def _raw(renderer, q4, k, outs, n=None):
    """bihrt_closest_k through ctypes with caller-owned outputs: returns the code"""
    import bihrt
    rec = bihrt.Closest(**{o: bihrt._ptr(v) for o, v in outs.items() if o in CLOSEST_OUTS})
    n = len(q4) if n is None else n
    return renderer._lib.bihrt_closest_k(renderer._ctx, bihrt._ptr(q4), C.c_int64(n), C.c_int32(k), C.byref(rec),
                                         bihrt._ptr(outs.get("count")), bihrt._ptr(outs.get("total")))


def test_watchdog_leaves_host_outputs_untouched(renderer, scenes):
    import bihrt
    tri = scenes.displaced_sphere(64)
    q = queries(np.random.default_rng(0).uniform(-1, 1, (4000, 3)).astype(np.float32), 0.3)
    renderer.load_models(tri).build()
    want = gpu_k(renderer, q, 4, total=True)
    renderer.set_option("debug_trip_watchdog", 2)
    renderer.build()
    outs = {"d2": np.full((4000, 4), 7.0, np.float32), "slot": np.full((4000, 4), -7, np.int32),
            "q": np.full((4000, 4, 3), 7.0, np.float32), "count": np.full(4000, -7, np.int32), "total": np.full(4000, -7, np.int32)}
    assert _raw(renderer, q, 4, outs) == -6
    assert np.all(outs["d2"] == 7.0) and np.all(outs["slot"] == -7) and np.all(outs["q"] == 7.0)
    assert np.all(outs["count"] == -7) and np.all(outs["total"] == -7)
    with pytest.raises(bihrt.BihrtError) as e:
        renderer.closest_k(q, 4)
    assert e.value.code == -6
    renderer.set_option("debug_trip_watchdog", 0)
    renderer.build()
    renderer.sync()
    assert_k_equal(gpu_k(renderer, q, 4, total=True), want)


def test_inputs_outputs_and_errors(renderer, scenes, oracle, tree, closest_k):
    import torch
    import bihrt
    tri = scenes.cornell_box()
    pt = tree(oracle.Bih(tri))
    rng = np.random.default_rng(3)
    pts = rng.uniform(-1.2, 1.2, (5000, 3)).astype(np.float32)
    rmax = np.where(rng.random(5000) < 0.5, np.inf, 0.3).astype(np.float32)
    q = bihrt.point_queries(pts, rmax)
    k = 5
    # no BIH yet
    with pytest.raises(bihrt.BihrtError) as e:
        renderer.closest_k(q, k)
    assert e.value.code == -4
    renderer.load_models(tri).build()
    want = closest_k(pt, q, k, total=True)
    # numpy in, numpy out; the default outputs leave out the total
    got = renderer.closest_k(q, k)
    assert set(got) == set(ROWS)
    assert got["d2"].shape == (5000, k) and got["q"].shape == (5000, k, 3) and got["count"].shape == (5000,)
    assert_k_equal(got, want, "host")
    # torch in (device), torch out on the device
    qd = bihrt.point_queries(torch.from_numpy(pts).cuda(), torch.from_numpy(rmax).cuda())
    got = renderer.closest_k(qd, k, outputs=CLOSEST_K_OUTS)
    for o in CLOSEST_K_OUTS:
        assert got[o].is_cuda
    assert_k_equal({o: v.cpu().numpy() for o, v in got.items()}, want, "device")
    # on a side stream of torch's: ordered by wait_torch / torch_wait
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        qs = bihrt.point_queries(torch.from_numpy(pts).cuda(), torch.from_numpy(rmax).cuda())
        got = renderer.closest_k(qs, k, outputs=("d2", "total"))
        d2, total = got["d2"].cpu().numpy(), got["total"].cpu().numpy()
    np.testing.assert_array_equal(d2.view(np.uint32), want["d2"].view(np.uint32))
    np.testing.assert_array_equal(total, want["total"])
    # each output alone; host points with device outputs and device points with host outputs
    qd_c = qd.contiguous()
    for o in CLOSEST_K_OUTS:
        r = renderer.closest_k(q, k, outputs=(o,))
        assert list(r) == [o]
        np.testing.assert_array_equal(bits(r[o]), bits(want[o]), err_msg=o)
        dev = torch.empty(want[o].shape, dtype=torch.float32 if want[o].dtype == np.float32 else torch.int32, device="cuda")
        assert _raw(renderer, q, k, {o: dev}) == 0
        renderer.sync()
        host = np.empty_like(want[o])
        assert _raw(renderer, qd_c, k, {o: host}) == 0
        np.testing.assert_array_equal(bits(dev.cpu().numpy()), bits(host), err_msg=o)
        np.testing.assert_array_equal(bits(host), bits(want[o]), err_msg=o)
    # host rows next to device counts in one call
    host_d2, dev_total = np.empty((5000, k), np.float32), torch.empty(5000, dtype=torch.int32, device="cuda")
    assert _raw(renderer, q, k, {"d2": host_d2, "total": dev_total}) == 0
    renderer.sync()
    np.testing.assert_array_equal(bits(host_d2), bits(want["d2"]))
    np.testing.assert_array_equal(dev_total.cpu().numpy(), want["total"])
    # k = 0: counts only
    r = renderer.closest_k(q, 0, outputs=CLOSEST_K_OUTS)
    assert r["d2"].shape == (5000, 0) and np.all(r["count"] == 0)
    np.testing.assert_array_equal(r["total"], want["total"])
    with pytest.raises(ValueError):
        renderer.closest_k(q, k, outputs=("t",))
    with pytest.raises(ValueError):
        renderer.closest_k(q, K_MAX + 1)
    # errors
    lib, ctx = renderer._lib, renderer._ctx
    empty = C.byref(bihrt.Closest())
    assert lib.bihrt_closest_k(ctx, bihrt._ptr(q), C.c_int64(10), C.c_int32(k), None, None, None) == -1          # rec == NULL
    assert lib.bihrt_closest_k(ctx, bihrt._ptr(q), C.c_int64(10), C.c_int32(-1), empty, None, None) == -1         # k < 0
    assert lib.bihrt_closest_k(ctx, bihrt._ptr(q), C.c_int64(10), C.c_int32(K_MAX + 1), empty, None, None) == -1  # k > max
    assert lib.bihrt_closest_k(ctx, bihrt._ptr(q), C.c_int64(10), C.c_int32(K_MAX), empty, None, None) == 0
    assert _raw(renderer, q, k, {"count": np.empty(10, np.int32)}, n=-1) == -1                                     # n < 0
    assert lib.bihrt_closest_k(ctx, None, C.c_int64(10), C.c_int32(k), empty, None, None) == -1                    # pts == NULL
    assert lib.bihrt_closest_k(ctx, None, C.c_int64(0), C.c_int32(k), empty, None, None) == 0                      # nothing to do
    assert _raw(renderer, q, k, {}, n=(1 << 32) - (1 << 24)) == -1                                                 # 32-bit work counter
    flat = torch.zeros(4 * 64 + 1, dtype=torch.float32, device="cuda")
    assert lib.bihrt_closest_k(ctx, C.c_void_p(flat.data_ptr() + 4), C.c_int64(64), C.c_int32(k), empty, None, None) == -1
    assert "aligned" in lib.bihrt_last_error(ctx).decode()
    # host rows of 2^32 - 2^24 - 1 points x 64 (1.1 TB): the staging buffer cannot be allocated, nothing is launched
    assert _raw(renderer, qd_c, K_MAX, {"d2": np.empty(1, np.float32)}, n=(1 << 32) - (1 << 24) - 1) == -3
    assert_k_equal(renderer.closest_k(q, k, outputs=CLOSEST_K_OUTS), want, "after NOMEM")
    # a miss record
    r = renderer.closest_k(bihrt.point_queries(np.array([[5.0, 5.0, 5.0], [0.0, 0.0, 0.0]], np.float32),
                                               np.array([0.1, np.nan], np.float32)), 3, outputs=CLOSEST_K_OUTS)
    assert np.all(r["d2"] == FLT_MAX) and np.all(r["slot"] == -1) and np.all(r["prim"] == -1)
    assert np.all(r["u"] == 0) and np.all(r["v"] == 0) and np.all(r["q"] == 0) and np.all(r["ng"] == 0)
    assert np.all(r["count"] == 0) and np.all(r["total"] == 0)
