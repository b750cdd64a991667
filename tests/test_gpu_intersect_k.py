"""Multi-hit ray queries (bihrt_intersect_k, csrc/trace.cu k_trace MODE 5 and 6) on the GPU: the kernel's rows, counts and
totals equal the restatement's walk (tests/intersect_k_oracle.c) bit for bit, on parity and quality trees, for k in
{1, 3, 8, 64}, with and without the total, one- and two-sided -- the walk itself is tied to the closest-hit walk and to brute
force in tests/test_intersect_k_oracle.py.  At k = 1 the rows are bihrt_intersect's records (up to exact-t ties).
"""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest

from closest_oracle import blob_tree
from intersect_k_oracle import K_MAX, K_OUTS, intersect_k  # noqa: F401  (intersect_k: fixture)
from test_closest_oracle import CAPS
from test_gpu_closest import build, restated
from test_gpu_golden_scenes import SCENES as GOLDEN
from test_intersect_k_oracle import KS, assert_k_equal, intervals
from walk_oracle import FLT_MAX, OUTS, assert_blob_equals, bits, blob_of, rays8, tree  # noqa: F401  (tree: fixture)

pytestmark = pytest.mark.gpu

ROWS = OUTS + ("count",)


def gpu_k(renderer, r8, k, total=False, two_sided=False):
    return renderer.intersect_k(r8, k, two_sided=two_sided, outputs=ROWS + (("total",) if total else ()))


def check_all(renderer, ik, pt, r8, msg, ks=KS):
    """ik: the intersect_k fixture"""
    for two_sided in (False, True):
        for k in ks:
            for total in (False, True):
                assert_k_equal(gpu_k(renderer, r8, k, total, two_sided), ik(pt, r8, k, total, two_sided),
                               "%s k=%d total=%s two_sided=%s" % (msg, k, total, two_sided))


@pytest.mark.parametrize("name", list(GOLDEN))
@pytest.mark.parametrize("cap", (None,) + CAPS)
def test_kernel_equals_walk(renderer, oracle, scenes, tree, intersect_k, name, cap):
    tri, cam, w, h = GOLDEN[name](scenes)
    pt = restated(tri, cap, oracle, tree)
    build(renderer, tri, cap)
    assert_blob_equals(blob_of(renderer), pt, "%s %s" % (name, cap))
    rays = oracle.camera_rays(cam, w, h)
    check_all(renderer, intersect_k, pt, intervals(rays, pt, 17), "%s %s" % (name, cap))


@pytest.mark.parametrize("name", list(GOLDEN))
def test_k1_rows_are_intersect_records(renderer, oracle, scenes, name):
    tri, cam, w, h = GOLDEN[name](scenes)
    rays = oracle.camera_rays(cam, w, h)
    for cap in (None, 4):
        build(renderer, tri, cap)
        r8 = rays8(rays)
        for two_sided in (False, True):
            a, b = renderer.intersect_k(r8, 1, two_sided=two_sided), renderer.intersect(r8, two_sided=two_sided)
            np.testing.assert_array_equal(bits(a["t"][:, 0]), bits(b["t"]))
            np.testing.assert_array_equal(a["count"], (b["slot"] >= 0).astype(np.int32))
            tie = a["slot"][:, 0] != b["slot"]
            assert np.all(a["slot"][tie, 0] < b["slot"][tie])          # exact-t ties: the smaller slot
            for o in ("u", "v", "prim", "ng"):
                np.testing.assert_array_equal(bits(a[o][~tie, 0]), bits(b[o][~tie]), err_msg="%s %s %s" % (name, cap, o))


def test_large_scene(renderer, oracle, scenes, tree, intersect_k):
    """1 M-triangle sphere, 200 k rays, both tree kinds: 100 k from a camera inside the sphere (two-sided: the exit hits) and
    100 k camera rays from outside (entry and exit, two-sided); the atrium's camera with its many layers."""
    tri = scenes.displaced_sphere(scenes.SPHERE_NSEG["1m"])
    rng = np.random.default_rng(8)
    d = rng.normal(size=(100000, 3))
    inside = np.concatenate([rng.normal(scale=0.05, size=(100000, 3)), d], 1).astype(np.float32)
    outside = oracle.camera_rays(scenes.pinhole_camera(), 400, 250)
    r8 = rays8(np.concatenate([inside, outside]))
    for cap in (None, 4):
        pt = restated(tri, cap, oracle, tree)
        build(renderer, tri, cap)
        assert_blob_equals(blob_of(renderer), pt, "1m %s" % cap)
        for k in (1, 4, 16):
            for total in (False, True):
                got = gpu_k(renderer, r8, k, total, two_sided=True)
                assert_k_equal(got, intersect_k(pt, r8, k, total, two_sided=True), "1m %s k=%d total=%s" % (cap, k, total))
        assert (got["total"][:100000] % 2 == 1).mean() > 0.999        # a closed mesh seen from inside: odd crossings (rays
                                                                      # through a shared edge may count it twice)
        got = gpu_k(renderer, r8, 4)
        assert_k_equal(got, intersect_k(pt, r8, 4), "1m %s one-sided" % cap)
    tri = scenes.atrium(0.3)
    rays = oracle.camera_rays(scenes.atrium_camera(), 320, 180)
    for cap in (None, 4):
        pt = restated(tri, cap, oracle, tree)
        build(renderer, tri, cap)
        check_all(renderer, intersect_k, pt, rays8(rays), "atrium %s" % cap, ks=(4, 64))


@pytest.mark.parametrize("case", ["one_triangle", "one_cell_parity", "one_leaf_quality"])
def test_single_leaf(renderer, oracle, scenes, tree, intersect_k, case):
    from test_closest_oracle import identical
    tri, cap = {"one_triangle": (scenes.dodecahedron()[:1], None), "one_cell_parity": (identical(40), None),
                "one_leaf_quality": (scenes.dodecahedron()[:12], 16)}[case]
    pt = restated(tri, cap, oracle, tree)
    assert pt.nu == 1
    build(renderer, tri, cap)
    assert_blob_equals(blob_of(renderer), pt, case)
    rng = np.random.default_rng(1)
    o = rng.uniform(-2, 2, (3000, 3))
    d = rng.uniform(-0.5, 0.5, (3000, 3)) - o
    r8 = rays8(np.concatenate([o, d], 1).astype(np.float32))
    check_all(renderer, intersect_k, pt, r8, case, ks=(1, 8))
    for total in (False, True):
        assert_k_equal(gpu_k(renderer, r8, 8, total), intersect_k(pt, r8, 8, True, brute=True), "%s brute" % case,
                       ROWS)


def test_refit_equals_restatement(renderer, oracle, scenes, intersect_k):
    tri = scenes.displaced_sphere(96)
    moved = scenes.displaced_sphere(96, phase=0.7)
    build(renderer, tri, None)
    renderer.update_vertices(moved)
    renderer.refit()
    bt = blob_tree(blob_of(renderer))
    bt = SimpleNamespace(tri9=moved.reshape(-1, 9), hdr=bt.hdr, nodes=bt.nodes, tris=bt.tris)
    rng = np.random.default_rng(6)
    o = rng.uniform(-1.5, 1.5, (5000, 3))
    d = rng.uniform(-0.5, 0.5, (5000, 3)) - o
    check_all(renderer, intersect_k, bt, rays8(np.concatenate([o, d], 1).astype(np.float32)), "refit", ks=(1, 8))


def test_replicas(renderer, scenes, oracle):
    import torch
    import bihrt
    tri = scenes.atrium(0.15)
    r8 = rays8(oracle.camera_rays(scenes.atrium_camera(), 160, 90))
    build(renderer, tri, 4)
    want = gpu_k(renderer, r8, 8, total=True, two_sided=True)
    nbytes = renderer.bih_blob_bytes()
    blob = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    renderer.bih_export(blob, nbytes)
    renderer.sync()
    r2 = bihrt.Renderer(0)
    r2.bih_import(blob, nbytes)
    assert_k_equal(gpu_k(r2, r8, 8, total=True, two_sided=True), want, "imported")
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
        gpu_k(r3, r8, 8, total=True, two_sided=True)
    assert e.value.code == -4
    r3.set_option("morton_bits", 63)
    r3.bih_adopt(len(tri))
    assert_k_equal(gpu_k(r3, r8, 8, total=True, two_sided=True), want, "adopted")
    r3.close()


def _raw(renderer, r8, k, outs, n=None, flags=0):
    """bihrt_intersect_k through ctypes with caller-owned outputs: returns the code"""
    import bihrt
    rec = bihrt.Hits(**{o: bihrt._ptr(v) for o, v in outs.items() if o in OUTS})
    n = len(r8) if n is None else n
    return renderer._lib.bihrt_intersect_k(renderer._ctx, bihrt._ptr(r8), C.c_int64(n), C.c_int32(k), C.c_uint32(flags),
                                           C.byref(rec), bihrt._ptr(outs.get("count")), bihrt._ptr(outs.get("total")))


def test_watchdog_leaves_host_outputs_untouched(renderer, scenes, oracle):
    import bihrt
    tri = scenes.displaced_sphere(64)
    r8 = rays8(oracle.camera_rays(scenes.pinhole_camera(), 80, 50))
    n = len(r8)
    renderer.load_models(tri).build()
    want = gpu_k(renderer, r8, 4, total=True)
    renderer.set_option("debug_trip_watchdog", 2)
    renderer.build()
    outs = {"t": np.full((n, 4), 7.0, np.float32), "slot": np.full((n, 4), -7, np.int32),
            "ng": np.full((n, 4, 3), 7.0, np.float32), "count": np.full(n, -7, np.int32), "total": np.full(n, -7, np.int32)}
    assert _raw(renderer, r8, 4, outs) == -6
    assert np.all(outs["t"] == 7.0) and np.all(outs["slot"] == -7) and np.all(outs["ng"] == 7.0)
    assert np.all(outs["count"] == -7) and np.all(outs["total"] == -7)
    with pytest.raises(bihrt.BihrtError) as e:
        renderer.intersect_k(r8, 4)
    assert e.value.code == -6
    renderer.set_option("debug_trip_watchdog", 0)
    renderer.build()
    renderer.sync()
    assert_k_equal(gpu_k(renderer, r8, 4, total=True), want)


def test_inputs_outputs_and_errors(renderer, scenes, oracle, tree, intersect_k):
    import torch
    import bihrt
    tri = scenes.cornell_box()
    pt = tree(oracle.Bih(tri))
    rays = oracle.camera_rays(scenes.cornell_camera(), 80, 60)
    r8 = intervals(rays, pt, 3)
    n, k = len(r8), 5
    lib, ctx = renderer._lib, renderer._ctx
    empty = C.byref(bihrt.Hits())
    # no BIH yet
    with pytest.raises(bihrt.BihrtError) as e:
        renderer.intersect_k(r8, k)
    assert e.value.code == -4
    renderer.load_models(tri).build()
    want = intersect_k(pt, r8, k, total=True)
    # numpy in, numpy out; the default outputs leave out the total
    got = renderer.intersect_k(r8, k)
    assert set(got) == set(ROWS)
    assert got["t"].shape == (n, k) and got["ng"].shape == (n, k, 3) and got["count"].shape == (n,)
    assert_k_equal(got, want, "host")
    # torch in (device), torch out on the device
    rd = torch.from_numpy(r8).cuda()
    got = renderer.intersect_k(rd, k, outputs=K_OUTS)
    for o in K_OUTS:
        assert got[o].is_cuda
    assert_k_equal({o: v.cpu().numpy() for o, v in got.items()}, want, "device")
    # on a side stream of torch's, behind a long kernel: ordered by wait_torch / torch_wait
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(50_000_000)
        rs = torch.from_numpy(r8).cuda() * 1.0
        got = renderer.intersect_k(rs, k, outputs=("t", "total"))
        t, total = got["t"].cpu().numpy(), got["total"].cpu().numpy()
    np.testing.assert_array_equal(bits(t), bits(want["t"]))
    np.testing.assert_array_equal(total, want["total"])
    # each output alone; host rays with device outputs and device rays with host outputs
    for o in K_OUTS:
        r = renderer.intersect_k(r8, k, outputs=(o,))
        assert list(r) == [o]
        np.testing.assert_array_equal(bits(r[o]), bits(want[o]), err_msg=o)
        dev = torch.empty(want[o].shape, dtype=torch.float32 if want[o].dtype == np.float32 else torch.int32, device="cuda")
        assert _raw(renderer, r8, k, {o: dev}) == 0
        renderer.sync()
        host = np.empty_like(want[o])
        assert _raw(renderer, rd, k, {o: host}) == 0
        np.testing.assert_array_equal(bits(dev.cpu().numpy()), bits(host), err_msg=o)
        np.testing.assert_array_equal(bits(host), bits(want[o]), err_msg=o)
    # two-sided through the raw call
    host_t = np.empty((n, k), np.float32)
    assert _raw(renderer, r8, k, {"t": host_t}, flags=bihrt.INTERSECT_TWO_SIDED) == 0
    np.testing.assert_array_equal(bits(host_t), bits(intersect_k(pt, r8, k, two_sided=True)["t"]))
    # k = 0: counts only
    r = renderer.intersect_k(r8, 0, outputs=K_OUTS)
    assert r["t"].shape == (n, 0) and np.all(r["count"] == 0)
    np.testing.assert_array_equal(r["total"], want["total"])
    with pytest.raises(ValueError):
        renderer.intersect_k(r8, k, outputs=("d2",))
    with pytest.raises(ValueError):
        renderer.intersect_k(r8, K_MAX + 1)
    # errors
    rp = bihrt._ptr(r8)
    assert lib.bihrt_intersect_k(ctx, rp, C.c_int64(10), C.c_int32(k), C.c_uint32(0), None, None, None) == -1   # rec NULL
    assert lib.bihrt_intersect_k(ctx, rp, C.c_int64(10), C.c_int32(-1), C.c_uint32(0), empty, None, None) == -1  # k < 0
    assert lib.bihrt_intersect_k(ctx, rp, C.c_int64(10), C.c_int32(K_MAX + 1), C.c_uint32(0), empty, None, None) == -1
    assert lib.bihrt_intersect_k(ctx, rp, C.c_int64(10), C.c_int32(K_MAX), C.c_uint32(0), empty, None, None) == 0
    for flags in (bihrt.INTERSECT_ANY, bihrt.INTERSECT_ANY | bihrt.INTERSECT_TWO_SIDED, 2, 8):                       # ANY, unknown bits
        assert lib.bihrt_intersect_k(ctx, rp, C.c_int64(10), C.c_int32(k), C.c_uint32(flags), empty, None, None) == -1
    assert _raw(renderer, r8, k, {"count": np.empty(10, np.int32)}, n=-1) == -1                                    # n < 0
    assert lib.bihrt_intersect_k(ctx, None, C.c_int64(10), C.c_int32(k), C.c_uint32(0), empty, None, None) == -1     # rays NULL
    assert lib.bihrt_intersect_k(ctx, None, C.c_int64(0), C.c_int32(k), C.c_uint32(0), empty, None, None) == 0      # nothing to do
    assert _raw(renderer, r8, k, {}, n=(1 << 32) - (1 << 24)) == -1                                                 # work counter
    flat = torch.zeros(8 * 64 + 1, dtype=torch.float32, device="cuda")
    assert lib.bihrt_intersect_k(ctx, C.c_void_p(flat.data_ptr() + 4), C.c_int64(64), C.c_int32(k), C.c_uint32(0), empty,
                                 None, None) == -1
    assert "aligned" in lib.bihrt_last_error(ctx).decode()
    # host rows of 2^32 - 2^24 - 1 rays x 64 (1.1 TB): the staging buffer cannot be allocated, nothing is launched
    assert _raw(renderer, rd, K_MAX, {"t": np.empty(1, np.float32)}, n=(1 << 32) - (1 << 24) - 1) == -3
    assert_k_equal(renderer.intersect_k(r8, k, outputs=K_OUTS), want, "after NOMEM")
    # miss records: a ray past the scene, a NaN interval
    r = renderer.intersect_k(rays8(np.array([[5, 5, 5, 1, 1, 1], [0, 0, -3, 0, 0, 1]], np.float32), np.array([0, np.nan],
                                   np.float32)), 3, outputs=K_OUTS)
    assert np.all(r["t"] == FLT_MAX) and np.all(r["slot"] == -1) and np.all(r["prim"] == -1)
    assert np.all(r["u"] == 0) and np.all(r["v"] == 0) and np.all(r["ng"] == 0)
    assert np.all(r["count"] == 0) and np.all(r["total"] == 0)
