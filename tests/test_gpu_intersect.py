"""Ray queries with per-ray intervals and full hit records (bihrt_intersect, csrc/trace.cu MODE 3).

tests/walk_oracle.c restates the query on the CPU: its walk over the parity tree's blob is the oracle's "box" traversal
(what the shipped kernel does) with the ray's interval, and its brute force tests every slot over the interval.  The CPU
tests tie the walk back to "box" (over (0, inf) it is "box", counters included: the anchor of every GPU trace test) and to
brute force; the GPU tests hold the exported parity blob to the restated one word for word, the kernel to the walk bit for
bit in all six outputs (t, u, v, slot, prim, ng) and to bihrt_trace / bihrt_trace_any where the interval is the one those
calls use.

Tie tolerance: where a test compares two different walks (the BIH against brute force), primitive ids may differ on exact-t
ties, the class DESIGN.md section 2 documents, on at most ID_MISMATCH_MAX of the rays.  Each such comparison is
marked "tie tolerance" below; every other comparison is exact.
"""
import ctypes as C

import numpy as np
import pytest

from test_gpu_golden_scenes import SCENES as GOLDEN
from walk_oracle import (FLT_MAX, OUTS, assert_blob_equals, assert_records_equal, assorted_intervals, bits, blob_of,
                         degenerate_rays, mt, rays8, tree)  # noqa: F401  (tree: fixture)

ID_MISMATCH_MAX = 1e-4


# ------------------------------------------------------------------------------------------------ CPU: the restatement

@pytest.mark.parametrize("name", list(GOLDEN))
def test_full_interval_equals_box_on_golden_scenes(oracle, scenes, tree, name):
    tri, cam, w, h = GOLDEN[name](scenes)
    ob = oracle.Bih(tri)
    pt = tree(ob)
    rays = oracle.camera_rays(cam, w, h)
    t3, s3, p3, c3 = ob.trace(rays, "box", want_counters=True)
    for tmax in (FLT_MAX, np.inf):
        r = pt.walk(rays8(rays, 0.0, tmax))
        np.testing.assert_array_equal(bits(r["t"]), bits(t3))
        np.testing.assert_array_equal(r["slot"], s3)
        np.testing.assert_array_equal(r["prim"], p3)
        assert r["counters"] == c3


def test_full_interval_equals_box_on_degenerate_rays(oracle, scenes, tree):
    tri, rays = degenerate_rays(scenes)
    ob = oracle.Bih(tri)
    pt = tree(ob)
    t3, s3, p3, c3 = ob.trace(rays, "box", want_counters=True)
    r = pt.walk(rays8(rays))
    np.testing.assert_array_equal(bits(r["t"]), bits(t3))
    np.testing.assert_array_equal(r["slot"], s3)
    assert r["counters"] == c3
    assert (s3 >= 0).sum() > 1000


@pytest.mark.parametrize("name", ["cornell", "sphere187", "atrium", "soup"])
def test_tmax_cut_hits_iff_box_t_below_tmax(oracle, scenes, tree, name):
    tri, cam, w, h = GOLDEN[name](scenes)
    ob = oracle.Bih(tri)
    pt = tree(ob)
    rays = oracle.camera_rays(cam, w, h)
    t3, s3, _ = ob.trace(rays, "box")
    rng = np.random.default_rng(3)
    ref = np.where(t3 < FLT_MAX, t3, 4.0)
    tmax = (ref * rng.uniform(0.5, 1.5, len(rays))).astype(np.float32)
    exact = rng.random(len(rays)) < 0.05
    tmax[exact] = ref[exact]                                     # tmax exactly at the hit: strict, so a miss
    r = pt.walk(rays8(rays, 0.0, tmax))
    want_hit = t3 < tmax
    np.testing.assert_array_equal(r["slot"] >= 0, want_hit)
    np.testing.assert_array_equal(bits(r["t"][want_hit]), bits(t3[want_hit]))
    np.testing.assert_array_equal(r["slot"][want_hit], s3[want_hit])
    assert 0.02 < want_hit.mean() and (~want_hit & (t3 < FLT_MAX)).sum() > 0


@pytest.mark.parametrize("which", ["sphere187", "sphere361", "soup"])
def test_box_equals_brute_force_on_random_intervals(oracle, scenes, tree, which):
    tri, cam, w, h = GOLDEN[which](scenes)
    ob = oracle.Bih(tri)
    pt = tree(ob)
    rays = oracle.camera_rays(cam, w, h)
    t3, _, _ = ob.trace(rays, "box")
    tmin, tmax = assorted_intervals(t3, seed=11)
    r8 = rays8(rays, tmin, tmax)
    a, b = pt.walk(r8), pt.brute(r8)
    np.testing.assert_array_equal(bits(a["t"]), bits(b["t"]))
    bad = a["prim"] != b["prim"]
    assert bad.sum() <= max(1, ID_MISMATCH_MAX * len(rays))            # tie tolerance (exact-t ties only)
    assert np.all(a["t"][bad] == b["t"][bad])
    assert (a["slot"] >= 0).mean() > 0.05


def test_peeling_visits_every_layer_front_to_back(oracle, scenes, tree):
    """random_soup: a query with tmin = the previous t, repeated until a miss, yields the distinct t of every triangle the ray
    crosses, increasing, the same sequence brute force peels."""
    tri = scenes.random_soup(20000, size=0.05)
    ob = oracle.Bih(tri)
    pt = tree(ob)
    rays = oracle.camera_rays(scenes.pinhole_camera(), 64, 36)
    seqs = {}
    for mode in ("box", "brute"):
        tmin = np.zeros(len(rays), np.float32)
        alive = np.ones(len(rays), bool)
        seq = [[] for _ in range(len(rays))]
        while alive.any():
            idx = np.nonzero(alive)[0]
            r = (pt.walk if mode == "box" else pt.brute)(rays8(rays[idx], tmin[idx], np.inf))
            hit = r["slot"] >= 0
            for i, t in zip(idx[hit], r["t"][hit]):
                assert t > tmin[i]
                seq[i].append(float(t))
            tmin[idx[hit]] = r["t"][hit]
            alive[idx[~hit]] = False
        seqs[mode] = seq
    assert seqs["box"] == seqs["brute"]
    depth = np.array([len(s) for s in seqs["box"]])
    assert depth.max() >= 5 and (depth >= 2).mean() > 0.2


@pytest.mark.parametrize("name", ["cornell", "sphere187", "atrium", "soup"])
def test_any_hit_hits_where_closest_hit_hits(oracle, scenes, tree, name):
    tri, cam, w, h = GOLDEN[name](scenes)
    ob = oracle.Bih(tri)
    pt = tree(ob)
    rays = oracle.camera_rays(cam, w, h)
    t3, _, _ = ob.trace(rays, "box")
    tmin, tmax = assorted_intervals(t3, seed=5)
    r8 = rays8(rays, tmin, tmax)
    c, a = pt.walk(r8), pt.walk(r8, "any")
    hit = a["slot"] >= 0
    np.testing.assert_array_equal(hit, c["slot"] >= 0)
    assert np.all(a["t"][hit] > np.maximum(tmin[hit], 0)) and np.all(a["t"][hit] < tmax[hit])
    assert np.all(a["t"][hit] >= c["t"][hit])
    assert a["counters"]["tris"] <= c["counters"]["tris"]


@pytest.mark.parametrize("name", ["dodecahedron", "cornell", "sphere187", "soup"])
def test_hit_record_is_consistent(oracle, scenes, tree, name):
    """u, v >= 0, u + v <= 1, o + t d ~ v0 + u e1 + v e2 (float64), ng = e1 x e2 facing the ray, miss = the miss record; t, u,
    v equal a numpy restatement of Moller-Trumbore on the reported triangle bit for bit."""
    tri, cam, w, h = GOLDEN[name](scenes)
    ob = oracle.Bih(tri)
    pt = tree(ob)
    rays = oracle.camera_rays(cam, w, h)
    t3, _, _ = ob.trace(rays, "box")
    tmin, tmax = assorted_intervals(t3, seed=9)
    r = pt.walk(rays8(rays, tmin, tmax))
    hit = r["slot"] >= 0
    assert hit.sum() > 100
    u, v, t, p = r["u"][hit], r["v"][hit], r["t"][hit], r["prim"][hit]
    assert np.all(u >= 0) and np.all(v >= 0) and np.all(u + v <= 1)
    T = tri.reshape(-1, 9).astype(np.float64)[p]
    o, d = rays[hit, :3].astype(np.float64), rays[hit, 3:].astype(np.float64)
    P = o + t[:, None].astype(np.float64) * d
    Q = T[:, 0:3] + u[:, None] * (T[:, 3:6] - T[:, 0:3]) + v[:, None] * (T[:, 6:9] - T[:, 0:3])
    scale = np.abs(T).max(axis=1) + np.abs(o).max(axis=1) + 1.0
    assert np.all(np.abs(P - Q).max(axis=1) <= 1e-5 * scale * (1 + t))
    ok, _, tn, un, vn = mt(tri, p, rays[hit])
    assert ok.all()
    np.testing.assert_array_equal(bits(t), bits(tn))
    np.testing.assert_array_equal(bits(u), bits(un))
    np.testing.assert_array_equal(bits(v), bits(vn))
    assert np.all((d * r["ng"][hit].astype(np.float64)).sum(1) < 0)
    miss = ~hit
    assert np.all(r["t"][miss] == FLT_MAX) and np.all(r["slot"][miss] == -1) and np.all(r["prim"][miss] == -1)
    assert not bits(r["u"][miss]).any() and not bits(r["v"][miss]).any() and not bits(r["ng"][miss]).any()


# ------------------------------------------------------------------------------------------------ GPU: the kernel

def gpu_intersect_host_and_device(renderer, r8, any_hit, outputs=OUTS):
    """The same query with numpy (host) buffers and with torch device buffers; returns both as numpy dicts."""
    import torch
    host = renderer.intersect(r8, any_hit=any_hit, outputs=outputs)
    dev = renderer.intersect(torch.from_numpy(r8).cuda(), any_hit=any_hit, outputs=outputs)
    return host, {k: x.cpu().numpy() for k, x in dev.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GOLDEN))
def test_parity_build_equals_restated_blob(renderer, oracle, scenes, tree, name):
    """The blob bihrt_bih_export writes after a parity build is orc_parity_blob's: header, every node's planes, child
    references and children boxes, every triangle record."""
    tri = GOLDEN[name](scenes)[0]
    renderer.load_models(tri).build()
    assert_blob_equals(blob_of(renderer), tree(oracle.Bih(tri)), name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GOLDEN))
def test_intersect_equals_range_oracle_bit_for_bit(renderer, oracle, scenes, tree, name):
    tri, cam, w, h = GOLDEN[name](scenes)
    ob = oracle.Bih(tri)
    pt = tree(ob)
    rays = oracle.camera_rays(cam, w, h)
    renderer.load_models(tri).build()
    t3, _, _ = ob.trace(rays, "box")
    tmin, tmax = assorted_intervals(t3, seed=17)
    r8 = rays8(rays, tmin, tmax)
    for any_hit in (False, True):
        want = pt.walk(r8, "any" if any_hit else "closest")
        host, dev = gpu_intersect_host_and_device(renderer, r8, any_hit)
        assert_records_equal(host, want, msg="host any=%s" % any_hit)
        assert_records_equal(dev, want, msg="device any=%s" % any_hit)
        hit = host["slot"] >= 0
        assert np.all((rays[hit, 3:].astype(np.float64) * host["ng"][hit]).sum(1) < 0)
        assert np.all(host["t"][~hit] == FLT_MAX) and np.all(host["prim"][~hit] == -1)
        assert not bits(host["u"][~hit]).any() and not bits(host["v"][~hit]).any() and not bits(host["ng"][~hit]).any()
    # subsets of the outputs (the rest NULL), host and device
    want = pt.walk(r8)
    for subset in (("t",), ("slot", "prim"), ("u", "v"), ("ng",), ("t", "ng", "prim")):
        host, dev = gpu_intersect_host_and_device(renderer, r8, False, subset)
        assert set(host) == set(subset) == set(dev)
        assert_records_equal(host, want, subset, "host %s" % (subset,))
        assert_records_equal(dev, want, subset, "device %s" % (subset,))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GOLDEN))
def test_full_interval_equals_trace(renderer, oracle, scenes, name):
    tri, cam, w, h = GOLDEN[name](scenes)
    rays = oracle.camera_rays(cam, w, h)
    renderer.load_models(tri).build()
    t, s, p = renderer.trace(rays)
    r = renderer.intersect(rays8(rays, 0.0, np.inf))
    np.testing.assert_array_equal(bits(r["t"]), bits(t))
    np.testing.assert_array_equal(r["slot"], s)
    np.testing.assert_array_equal(r["prim"], p)


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["sphere", "atrium"])
def test_secondary_lists_equal_trace_and_trace_any(renderer, scenes, scene):
    """Shadow and diffuse lists of bihrt_secondary_rays: (0, inf) equals bihrt_trace; ANY with tmax = 1 on every ray
    equals bihrt_trace_any(tmax = 1) in what hits, and every record it reports is a true hit of its triangle."""
    import torch
    from bihrt import interval_rays
    if scene == "sphere":
        tri, cam, w, h = scenes.displaced_sphere(96), scenes.pinhole_camera(aspect=320 / 180), 320, 180
    else:
        tri, cam, w, h = scenes.atrium(0.3), scenes.atrium_camera(320 / 180), 320, 180
    renderer.load_models(tri).build()
    for kind in ("shadow", "diffuse"):
        rays, _ = renderer.secondary_rays(cam, w, h, spp=2, kind=kind, light=(0.1, 0.8, -0.2), jitter=True)
        t, s, p = renderer.trace(rays)
        r = renderer.intersect(interval_rays(rays, 0.0, float("inf")))
        for k, x in (("t", t), ("slot", s), ("prim", p)):
            assert torch.equal(r[k], x), (kind, k)
        a = renderer.intersect(interval_rays(rays, 0.0, 1.0), any_hit=True)
        b = renderer.trace_any(rays, tmax=1.0)
        assert torch.equal(a["slot"] >= 0, b >= 0), kind
        hit = (a["slot"] >= 0).cpu().numpy()
        if kind == "shadow":
            assert hit.any()
        got = {k: x.cpu().numpy()[hit] for k, x in a.items()}
        ok, _, tn, un, vn = mt(tri, got["prim"], rays.cpu().numpy()[hit])
        assert ok.all()
        np.testing.assert_array_equal(bits(got["t"]), bits(tn))
        np.testing.assert_array_equal(bits(got["u"]), bits(un))
        np.testing.assert_array_equal(bits(got["v"]), bits(vn))
        assert np.all((got["t"] > 0) & (got["t"] < 1))


@pytest.mark.gpu
def test_per_sm_queue_launch_equals_trace(renderer, scenes):
    """2^24 + 1 rays: the launch takes the per-SM work queues."""
    import torch
    from bihrt import interval_rays
    tri = scenes.displaced_sphere(187)
    renderer.load_models(tri).build()
    g = torch.Generator(device="cuda").manual_seed(5)
    n = (1 << 24) + 1
    o = torch.rand((n, 3), device="cuda", generator=g) * 4 - 2
    target = torch.rand((n, 3), device="cuda", generator=g) - 0.5
    rays = torch.cat([o, target - o], 1).contiguous()
    t, s, p = renderer.trace(rays)
    r = renderer.intersect(interval_rays(rays, 0.0, float("inf")), outputs=("t", "slot", "prim", "ng"))
    assert torch.equal(r["t"], t) and torch.equal(r["slot"], s) and torch.equal(r["prim"], p)
    hit = s >= 0
    assert 0.1 < hit.float().mean().item() < 0.99
    assert bool(((rays[hit, 3:] * r["ng"][hit]).sum(1) < 0).all())


@pytest.mark.gpu
@pytest.mark.parametrize("cap", [1, 4, 16])
@pytest.mark.parametrize("name", ["cornell", "sphere187", "atrium", "soup"])
def test_quality_mode_equals_brute_force(renderer, oracle, scenes, tree, name, cap):
    tri, cam, w, h = GOLDEN[name](scenes)
    ob = oracle.Bih(tri)
    pt = tree(ob)
    rays = oracle.camera_rays(cam, w, h)
    renderer.set_option("morton_bits", 63)
    renderer.set_option("leaf_cap", cap)
    renderer.load_models(tri).build()
    t3, _, _ = ob.trace(rays, "brute")
    tmin, tmax = assorted_intervals(t3, seed=23)
    r8 = rays8(rays, tmin, tmax)
    want = pt.brute(r8)
    got = renderer.intersect(r8)
    np.testing.assert_array_equal(bits(got["t"]), bits(want["t"]))
    bad = got["prim"] != want["prim"]
    assert bad.sum() <= max(1, ID_MISMATCH_MAX * len(rays))            # tie tolerance (exact-t ties only)
    # slots index the quality tree's own triangle order, not the oracle's: only hit / miss compares
    np.testing.assert_array_equal(got["slot"] >= 0, want["slot"] >= 0)
    same = ~bad
    rec = ("t", "u", "v", "prim", "ng")
    assert_records_equal({k: got[k][same] for k in rec}, {k: want[k][same] for k in rec}, rec)
    a = renderer.intersect(r8, any_hit=True, outputs=("t", "slot"))
    np.testing.assert_array_equal(a["slot"] >= 0, want["slot"] >= 0)


@pytest.mark.gpu
def test_error_codes_and_stream_order(renderer, scenes, oracle):
    import torch
    import bihrt
    lib = bihrt.load_library()
    ctx = renderer._ctx
    rays = np.zeros((4, 8), np.float32)
    t = np.zeros(4, np.float32)
    hits = bihrt.Hits(t=t.ctypes.data)
    rp = C.c_void_p(rays.ctypes.data)
    assert lib.bihrt_intersect(ctx, rp, C.c_int64(4), C.c_uint32(0), C.byref(hits)) == -4       # no BIH built yet
    renderer.load_models(scenes.dodecahedron()).build()
    assert lib.bihrt_intersect(ctx, rp, C.c_int64(4), C.c_uint32(2), C.byref(hits)) == -1       # unknown flag bit
    assert lib.bihrt_intersect(ctx, None, C.c_int64(4), C.c_uint32(0), C.byref(hits)) == -1     # rays NULL, n > 0
    assert lib.bihrt_intersect(ctx, rp, C.c_int64(4), C.c_uint32(0), None) == -1                # out NULL
    assert lib.bihrt_intersect(ctx, rp, C.c_int64(-1), C.c_uint32(0), C.byref(hits)) == -1      # n < 0
    assert lib.bihrt_intersect(ctx, rp, C.c_int64((1 << 32) - (1 << 24)), C.c_uint32(0), C.byref(hits)) == -1
    d = torch.zeros(40, dtype=torch.float32, device="cuda")
    assert lib.bihrt_intersect(ctx, C.c_void_p(d.data_ptr() + 4), C.c_int64(4), C.c_uint32(0), C.byref(hits)) == -1  # misaligned
    assert lib.bihrt_intersect(ctx, None, C.c_int64(0), C.c_uint32(0), C.byref(hits)) == 0      # empty list
    # device outputs ordered with torch's current stream: the context runs on its own stream, rays are produced on torch's
    # stream right before the call (behind a long kernel), the outputs consumed right after
    tri = scenes.displaced_sphere(96)
    cam = scenes.pinhole_camera()
    rays6 = oracle.camera_rays(cam, 640, 360)
    want = renderer.load_models(tri).build().intersect(rays8(rays6, 0.5, 8.0))
    assert renderer.stream_handle() != torch.cuda.current_stream().cuda_stream
    base = torch.from_numpy(rays8(rays6, 0.5, 8.0)).cuda()
    for rep in range(3):
        torch.cuda._sleep(50_000_000)
        r8 = base * 1.0
        got = renderer.intersect(r8)
        s_sum = (got["slot"].long() + 1).sum()
        for k in OUTS:
            np.testing.assert_array_equal(bits(got[k].cpu().numpy()), bits(want[k]), err_msg=k)
        assert int(s_sum) == int((want["slot"].astype(np.int64) + 1).sum())
