"""Winding-number queries (bihrt_winding_number, csrc/winding.cu k_winding) on the GPU: the kernel's w equals the CPU
restatement's walk (tests/winding_oracle.c) bit for bit on parity and quality trees at every beta tested, the far-field table
is rebuilt whenever the BIH changes, and signed_distance composes the two queries as documented.  The restatement itself is
held to brute force and to float64 in tests/test_winding_oracle.py.
"""
import ctypes as C

import numpy as np
import pytest

from test_closest_oracle import CAPS, SCENE_NAMES, camera_for, point_set, queries, scene_set
from test_winding_oracle import BETA_TOL, sample_points
from closest_oracle import blob_tree, closest  # noqa: F401  (closest: fixture)
from walk_oracle import assert_blob_equals, bits, blob_of, tree  # noqa: F401  (tree: fixture)
from winding_oracle import winding  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu

BETAS = (1.5, 2.0, 4.0, np.inf)


def build(renderer, tri, cap):
    """Builds tri in renderer as the parity tree (cap None) or the quality tree at leaf cap `cap`."""
    renderer.set_option("morton_bits", 30 if cap is None else 63)
    if cap is not None:
        renderer.set_option("leaf_cap", cap)
    renderer.load_models(tri).build()
    return renderer


def restated(tri, cap, oracle, tree):
    return tree(oracle.Bih(tri)) if cap is None else tree(tri, cap)


def assert_bits(a, b, msg=""):
    np.testing.assert_array_equal(bits(np.asarray(a)), bits(np.asarray(b)), err_msg=msg)


@pytest.mark.parametrize("name", SCENE_NAMES)
@pytest.mark.parametrize("cap", (None,) + CAPS)
def test_kernel_equals_walk(renderer, oracle, scenes, tree, winding, name, cap):
    tri = scene_set(scenes)[name]
    pt = restated(tri, cap, oracle, tree)
    build(renderer, tri, cap)
    assert_blob_equals(blob_of(renderer), pt, "%s %s" % (name, cap))
    q = queries(point_set(tri, pt, oracle, camera_for(name, scenes)))
    for beta in BETAS:
        assert_bits(renderer.winding_number(q, beta), winding(pt, q, beta)[0], "%s %s beta %s" % (name, cap, beta))


def sphere_points(tri, rng, k):
    v = tri.reshape(-1, 3)
    lo, hi = v.min(0), v.max(0)
    c, ext = (lo + hi) * 0.5, hi - lo
    uni = rng.uniform(c - 0.6 * ext, c + 0.6 * ext, (k, 3))
    t = tri.reshape(-1, 9)[rng.integers(0, len(tri), k)]
    w = rng.dirichlet((1, 1, 1), k)
    near = np.einsum("kj,kjc->kc", w, t.reshape(-1, 3, 3)) + rng.normal(scale=1e-3, size=(k, 3))
    return np.concatenate([uni, near]).astype(np.float32)


def test_large_scene(renderer, oracle, scenes, tree, closest, winding):  # noqa: F811
    """1 M-triangle sphere, 200 k points (uniform in 1.2x the box, and near the surface), beta 2, both tree kinds; a sampled
    subset away from the surface also against float64."""
    tri = scenes.displaced_sphere(scenes.SPHERE_NSEG["1m"])
    pts = sphere_points(tri, np.random.default_rng(8), 100000)
    q = queries(pts)
    sub = np.random.default_rng(9).permutation(len(pts))[:200]
    w64 = winding.f64(tri, pts[sub])
    for cap in (None, 4):
        pt = restated(tri, cap, oracle, tree)
        build(renderer, tri, cap)
        assert_blob_equals(blob_of(renderer), pt, "1m %s" % cap)
        got = renderer.winding_number(q, 2.0)
        assert_bits(got, winding(pt, q, 2.0)[0], "1m %s" % cap)
        lo, hi = tri.reshape(-1, 3).min(0), tri.reshape(-1, 3).max(0)
        far = np.sqrt(closest(pt, q[sub])["d2"].astype(np.float64)) >= 1e-4 * np.linalg.norm(hi - lo)
        assert np.abs(got[sub][far] - w64[far]).max() <= BETA_TOL[2.0]
        np.testing.assert_array_equal(np.round(got[sub][far]), np.round(w64[far]))
        assert set(np.round(w64[far]).astype(int)) == {0, 1}


def test_table_follows_the_bih(renderer, oracle, scenes, tree, winding):
    """The table is rebuilt after every change of the BIH: refit, a rebuild of another mesh with the same n, a quality build
    over a parity build's stale node slots, and replicas (import, adopt, copy)."""
    import torch
    import bihrt
    rng = np.random.default_rng(6)
    tri = scenes.displaced_sphere(96)
    q = queries(sample_points(tri, rng, 3000))

    def check(r, what):
        words = blob_of(r)
        bt = blob_tree(words)
        for beta in (2.0, 4.0):
            assert_bits(r.winding_number(q, beta), winding(bt, q, beta)[0], "%s beta %s" % (what, beta))

    build(renderer, tri, None)
    check(renderer, "first build")
    renderer.update_vertices(scenes.displaced_sphere(96, phase=0.7))
    renderer.refit()
    check(renderer, "refit")
    other = (scenes.displaced_sphere(96, seed=11) * np.float32(0.7)).astype(np.float32)     # another mesh, the same n
    renderer.load_models(other).build()
    check(renderer, "rebuild, same n")
    build(renderer, tri, 4)                                       # quality tree over the parity tree's node slots
    check(renderer, "quality over parity")
    want = renderer.winding_number(q, 2.0)
    nbytes = renderer.bih_blob_bytes()
    blob = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    renderer.bih_export(blob, nbytes)
    renderer.sync()
    r2 = bihrt.Renderer(0)
    r2.load_models(other).build()
    r2.winding_number(q, 2.0)                                     # a table of the other mesh first
    r2.bih_import(blob, nbytes)
    assert_bits(r2.winding_number(q, 2.0), want, "imported")
    r2.close()
    r3 = bihrt.Renderer(0)
    r3.set_option("morton_bits", 63)
    r3.load_models(other).build()
    r3.winding_number(q, 2.0)
    ptr, nb = r3.bih_region(len(tri))
    src_ptr, _ = renderer.bih_region(len(tri))
    t_src = torch.as_tensor(bihrt.multi._CudaView(src_ptr, (nb,), "|u1"), device="cuda")
    t_dst = torch.as_tensor(bihrt.multi._CudaView(ptr, (nb,), "|u1"), device="cuda")
    renderer.sync()
    t_dst.copy_(t_src)
    torch.cuda.synchronize()
    r3.bih_adopt(len(tri))
    assert_bits(r3.winding_number(q, 2.0), want, "adopted")
    r3.close()
    r4 = bihrt.Renderer(0)
    r4.load_models(other).build()
    r4.winding_number(q, 2.0)
    assert r4._lib.bihrt_bih_copy(r4._ctx, renderer._ctx) == 0
    assert_bits(r4.winding_number(q, 2.0), want, "copied")
    r4.close()


def test_replica_of_the_other_kind_and_watchdog(renderer, scenes):
    import torch
    import bihrt
    tri = scenes.atrium(0.15)
    q = queries(np.random.default_rng(2).uniform(-1.5, 1.5, (4000, 3)).astype(np.float32))
    build(renderer, tri, 4)
    r3 = bihrt.Renderer(0)                                       # adopts a quality tree without being told the kind
    ptr, nb = r3.bih_region(len(tri))
    src_ptr, _ = renderer.bih_region(len(tri))
    t_src = torch.as_tensor(bihrt.multi._CudaView(src_ptr, (nb,), "|u1"), device="cuda")
    t_dst = torch.as_tensor(bihrt.multi._CudaView(ptr, (nb,), "|u1"), device="cuda")
    renderer.sync()
    t_dst.copy_(t_src)
    torch.cuda.synchronize()
    r3.bih_adopt(len(tri))
    with pytest.raises(bihrt.BihrtError) as e:
        r3.winding_number(q)
    assert e.value.code == -4
    r3.close()
    build(renderer, tri, None)
    want = renderer.winding_number(q)
    renderer.set_option("debug_trip_watchdog", 2)
    renderer.build()
    w = np.full(4000, 7.0, np.float32)
    assert renderer._lib.bihrt_winding_number(renderer._ctx, bihrt._ptr(q), C.c_int64(4000), C.c_float(2.0), bihrt._ptr(w)) == -6
    assert np.all(w == 7.0)
    with pytest.raises(bihrt.BihrtError) as e:
        renderer.winding_number(q)
    assert e.value.code == -6
    renderer.set_option("debug_trip_watchdog", 0)
    renderer.build()
    renderer.sync()
    assert_bits(renderer.winding_number(q), want)


def test_inputs_outputs_and_errors(renderer, scenes, oracle, tree, winding):
    import torch
    import bihrt
    tri = scenes.cornell_box()
    pt = tree(oracle.Bih(tri))
    pts = np.random.default_rng(3).uniform(-1.2, 1.2, (5000, 3)).astype(np.float32)
    q = bihrt.point_queries(pts)
    with pytest.raises(bihrt.BihrtError) as e:                   # no BIH yet
        renderer.winding_number(q)
    assert e.value.code == -4
    renderer.load_models(tri).build()
    want = winding(pt, q, 2.0)[0]
    assert_bits(renderer.winding_number(q), want, "host")
    qd = torch.from_numpy(q).cuda()
    got = renderer.winding_number(qd)
    assert got.is_cuda and got.dtype == torch.float32 and got.shape == (5000,)
    assert_bits(got.cpu().numpy(), want, "device")
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):                                   # on a side stream of torch's
        qs = torch.from_numpy(q).cuda()
        w = renderer.winding_number(qs).cpu().numpy()
    assert_bits(w, want, "side stream")
    lib, ctx = renderer._lib, renderer._ctx

    def raw(pts_, n, beta, out):
        return lib.bihrt_winding_number(ctx, bihrt._ptr(pts_), C.c_int64(n), C.c_float(beta), bihrt._ptr(out))
    dev = torch.empty(5000, dtype=torch.float32, device="cuda")
    assert raw(q, 5000, 2.0, dev) == 0                           # host points, device output
    renderer.sync()
    host = np.empty(5000, np.float32)
    assert raw(qd, 5000, 2.0, host) == 0                         # device points, host output
    assert_bits(dev.cpu().numpy(), want)
    assert_bits(host, want)
    assert raw(q, 10, 2.0, None) == -1                            # w == NULL
    assert raw(q, -1, 2.0, host) == -1                            # n < 0
    assert raw(None, 10, 2.0, host) == -1                         # pts == NULL, n > 0
    assert raw(None, 0, 2.0, host) == 0                           # nothing to do
    assert raw(q, (1 << 32) - (1 << 24), 2.0, host) == -1         # 32-bit work counter
    for beta in (1.0, 0.5, -1.0, float("nan"), float("-inf")):
        assert raw(q, 10, beta, host) == -1, beta
    flat = torch.zeros(4 * 64 + 1, dtype=torch.float32, device="cuda")
    assert lib.bihrt_winding_number(ctx, C.c_void_p(flat.data_ptr() + 4), C.c_int64(64), C.c_float(2.0), bihrt._ptr(host)) == -1
    assert "aligned" in lib.bihrt_last_error(ctx).decode()
    bad = bihrt.point_queries(np.array([[np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf]], np.float32))
    np.testing.assert_array_equal(renderer.winding_number(bad), 0.0)
    renderer.load_models(np.zeros((0, 9), np.float32)).build()   # an empty scene
    np.testing.assert_array_equal(renderer.winding_number(q[:100]), 0.0)


@pytest.mark.parametrize("case", ["one_triangle", "one_leaf_quality"])
def test_single_leaf(renderer, oracle, scenes, tree, winding, case):
    tri, cap = {"one_triangle": (scenes.dodecahedron()[:1], None), "one_leaf_quality": (scenes.dodecahedron()[:12], 16)}[case]
    pt = restated(tri, cap, oracle, tree)
    assert pt.nu == 1
    build(renderer, tri, cap)
    q = queries(np.random.default_rng(1).uniform(-2, 2, (3000, 3)).astype(np.float32))
    for beta in BETAS:
        assert_bits(renderer.winding_number(q, beta), winding(pt, q, brute=True)[0], "%s %s" % (case, beta))


def test_signed_distance(renderer, scenes):
    import torch
    import bihrt
    tri = np.concatenate([scenes.displaced_sphere(64), scenes.box([-0.3, -0.3, 1.5], [0.3, 0.3, 2.1], n=2)]).astype(np.float32)
    renderer.load_models(tri).build()
    rng = np.random.default_rng(12)
    pts = rng.uniform(-1.4, 2.3, (20000, 3)).astype(np.float32)
    rmax = np.where(rng.random(20000) < 0.8, np.inf, 0.05).astype(np.float32)
    q = bihrt.point_queries(pts, rmax)
    cp = renderer.closest_point(q)
    w = renderer.winding_number(q, 2.0)
    dist = np.where(cp["slot"] >= 0, np.sqrt(cp["d2"]), np.float32(np.inf)).astype(np.float32)
    want = np.where(w > 0.5, -dist, dist).astype(np.float32)
    got = renderer.signed_distance(q, outputs=("sd", "w", "slot", "q"))
    assert set(got) == {"sd", "w", "slot", "q"}
    assert_bits(got["sd"], want)
    assert_bits(got["w"], w)
    np.testing.assert_array_equal(got["slot"], cp["slot"])
    assert_bits(got["q"], cp["q"])
    assert (want < 0).sum() > 1000 and (want > 0).sum() > 1000 and np.isinf(want).sum() > 100
    assert np.isneginf(want).sum() > 0                           # a miss inside the mesh is -inf
    gd = renderer.signed_distance(torch.from_numpy(q).cuda(), beta=4.0)
    assert list(gd) == ["sd"] and gd["sd"].is_cuda
    w4 = renderer.winding_number(q, 4.0)
    assert_bits(gd["sd"].cpu().numpy(), np.where(w4 > 0.5, -dist, dist).astype(np.float32))
    with pytest.raises(ValueError):
        renderer.signed_distance(q, outputs=("t",))
