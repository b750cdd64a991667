"""Double-sided ray queries: bihrt_intersect with BIHRT_INTERSECT_TWO_SIDED (csrc/trace.cu MODE 4).

The flag changes one thing: a triangle is a candidate when !(|det| < 1e-6) instead of !(det < 1e-6).
tests/walk_oracle.c restates it on the CPU: the one-sided query's walk and brute force with its two_sided flag set.  The CPU
tests tie the two-sided restatement to two-sided brute force, to the one-sided query (superset of hits, t never larger,
front-face records unchanged) and to an independent numpy Moller-Trumbore; the GPU tests hold the kernel to the restatement
bit for bit in all six outputs.

Tie tolerance: where two different walks are compared, primitive ids may differ on exact-t ties on at most ID_MISMATCH_MAX
of the rays (as in test_gpu_intersect.py); such comparisons are marked "tie tolerance".  Coplanar tolerance (quality-mode
trees only, include/bihrt.h): where two triangles of different leaves lie in one plane, their t differ only by rounding and
the walk may report the one an ulp further; checked as exactly that class, on at most ID_MISMATCH_MAX of the rays.  Every
other comparison is exact.
"""
import ctypes as C

import numpy as np
import pytest

from test_gpu_golden_scenes import SCENES as GOLDEN
from test_gpu_intersect import ID_MISMATCH_MAX
from walk_oracle import (FLT_MAX, OUTS, assert_records_equal, assorted_intervals, bits, degenerate_rays, mt, rays8,
                         tree)  # noqa: F401  (tree: fixture)

DET_EPS = np.array([0x358637be], np.uint32).view(np.float32)[0]
INSIDE_CAMERA = dict(origin=(0.03, -0.02, 0.05), half=0.9, aspect=1.0)      # inside the displaced sphere, looking +z


def check_against_one_sided(one, two, tri, rays6):
    """The properties the header states for the flag, on records of the same rays and intervals (numpy dicts with all six
    outputs): every one-sided hit is a two-sided hit with t <= the one-sided t; every two-sided hit is a true hit of its
    triangle (t, u, v bit for bit by mt_two_sided); dot(d, ng) < 0 exactly on front faces; and a front-face record equals
    the one-sided record.  Returns the front-face mask over the two-sided hits."""
    h1, h2 = one["slot"] >= 0, two["slot"] >= 0
    assert np.all(h2[h1]), "a one-sided hit is missing from the two-sided query"
    assert np.all(two["t"][h1] <= one["t"][h1])
    ok, det, t, u, v = mt(tri, two["prim"][h2], rays6[h2], two_sided=True)
    assert ok.all()
    np.testing.assert_array_equal(bits(two["t"][h2]), bits(t))
    np.testing.assert_array_equal(bits(two["u"][h2]), bits(u))
    np.testing.assert_array_equal(bits(two["v"][h2]), bits(v))
    front = det.astype(np.float64) >= 1e-6
    side = (rays6[h2, 3:].astype(np.float64) * two["ng"][h2].astype(np.float64)).sum(1)
    np.testing.assert_array_equal(side < 0, front)
    assert np.all(side != 0)
    idx = np.nonzero(h2)[0][front]
    assert np.all(h1[idx]), "a front-face two-sided hit is a one-sided miss"
    np.testing.assert_array_equal(bits(two["t"][idx]), bits(one["t"][idx]))
    tie = two["prim"][idx] != one["prim"][idx]
    assert tie.sum() <= max(1, ID_MISMATCH_MAX * len(rays6))           # tie tolerance (exact-t ties only)
    same = idx[~tie]
    assert_records_equal({k: two[k][same] for k in OUTS}, {k: one[k][same] for k in OUTS})
    return front


def assert_coplanar_near_ties(tri9, rays6, got, want, sel):
    """Coplanar tolerance: on the rays `sel` the GPU reports another triangle than brute force, at a t one ulp larger, and
    both triangles are true hits that lie in one plane (coincident surfaces, such as the bottom of a box resting on a floor)."""
    tg, tw = got["t"][sel], want["t"][sel]
    assert np.all(bits(tg).astype(np.int64) - bits(tw).astype(np.int64) == 1)
    ok, _, t, _, _ = mt(tri9, got["prim"][sel], rays6[sel], two_sided=True)
    assert ok.all()
    np.testing.assert_array_equal(bits(t), bits(tg))
    T = tri9.reshape(-1, 9).astype(np.float64)
    a, b = T[got["prim"][sel]].reshape(-1, 3, 3), T[want["prim"][sel]].reshape(-1, 3, 3)
    n = np.cross(b[:, 1] - b[:, 0], b[:, 2] - b[:, 0])
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    dist = np.abs(((a - b[:, :1]) * n[:, None, :]).sum(2)).max(1)
    assert np.all(dist <= 1e-6 * (1 + np.abs(b).max((1, 2))))


def inside_sphere(scenes, oracle, w, h):
    return scenes.displaced_sphere(187), oracle.camera_rays(scenes.pinhole_camera(**INSIDE_CAMERA), w, h)


def inside_box(scenes, oracle, w, h):
    """box(n=8) with outward faces, seen from a camera inside it (every hit is a back face)."""
    tri = scenes.box([-1.0, -0.8, -1.2], [1.1, 0.9, 1.3], n=8)
    cam = scenes.look_at_camera((0.13, 0.07, -0.21), (0.9, 0.31, 1.0), 0.8, 1.0)
    return tri, oracle.camera_rays(cam, w, h)


# ------------------------------------------------------------------------------------------------ CPU: the restatement

def test_det_threshold_is_symmetric():
    """|det| < 1e-6 in binary32 against 0x358637be (csrc/trace.cu DET_EPS) equals fabs((double)det) < 0.000001 (the two-sided
    restatement) on both sides of zero."""
    for sign in (0, 0x80000000):
        for b in range(0x358637be - 4, 0x358637be + 4):
            d = np.array([b | sign], np.uint32).view(np.float32)[0]
            assert (abs(float(d)) < 0.000001) == bool(np.abs(d) < DET_EPS)
    for d in np.float32([0.0, -0.0, -1.0, 1.0, -1e-7, -9.9e-7, -1e-6, -1.1e-6, 1e-6, 1.1e-6]):
        assert (abs(float(d)) < 0.000001) == bool(np.abs(d) < DET_EPS)


@pytest.mark.parametrize("which", ["sphere187", "sphere361", "soup", "inside_sphere"])
def test_two_sided_box_equals_brute_force(oracle, scenes, tree, which):
    if which == "inside_sphere":
        tri, rays = inside_sphere(scenes, oracle, 160, 160)
    else:
        tri, cam, w, h = GOLDEN[which](scenes)
        rays = oracle.camera_rays(cam, w, h)
    pt = tree(oracle.Bih(tri))
    tmin, tmax = assorted_intervals(pt.walk(rays8(rays), two_sided=True)["t"], seed=31)
    for r8 in (rays8(rays), rays8(rays, tmin, tmax)):
        a, b = pt.walk(r8, two_sided=True), pt.brute(r8, two_sided=True)
        np.testing.assert_array_equal(bits(a["t"]), bits(b["t"]))
        bad = a["prim"] != b["prim"]
        assert bad.sum() <= max(1, ID_MISMATCH_MAX * len(rays))        # tie tolerance (exact-t ties only)
        assert np.all(a["t"][bad] == b["t"][bad])
        assert (a["slot"] >= 0).mean() > 0.05


def scene_and_rays(name, oracle, scenes):
    if name == "degenerate":
        return degenerate_rays(scenes)
    tri, cam, w, h = GOLDEN[name](scenes)
    return tri, oracle.camera_rays(cam, w, h)


@pytest.mark.parametrize("name", list(GOLDEN) + ["degenerate"])
def test_two_sided_against_one_sided(oracle, scenes, tree, name):
    tri, rays = scene_and_rays(name, oracle, scenes)
    ob = oracle.Bih(tri)
    pt = tree(ob)
    t3, _, _ = ob.trace(rays, "box")
    tmin, tmax = assorted_intervals(t3, seed=13)
    for r8 in (rays8(rays), rays8(rays, tmin, tmax)):
        one, two = pt.walk(r8), pt.walk(r8, two_sided=True)
        check_against_one_sided(one, two, tri, rays)
        a = pt.walk(r8, "any", two_sided=True)
        hit = a["slot"] >= 0
        np.testing.assert_array_equal(hit, two["slot"] >= 0)
        assert np.all(a["t"][hit] >= two["t"][hit])
        ok, _, t, _, _ = mt(tri, a["prim"][hit], rays[hit], two_sided=True)
        assert ok.all()
        np.testing.assert_array_equal(bits(a["t"][hit]), bits(t))


def test_camera_inside_closed_mesh_sees_back_faces(oracle, scenes, tree):
    tri, rays = inside_sphere(scenes, oracle, 160, 160)
    pt = tree(oracle.Bih(tri))
    r8 = rays8(rays)
    one, two = pt.walk(r8), pt.walk(r8, two_sided=True)
    assert (one["slot"] >= 0).sum() == 0
    hit = two["slot"] >= 0
    assert hit.mean() > 0.995                    # Moller-Trumbore is not watertight: a ray through an edge may miss both
    assert np.all((rays[hit, 3:].astype(np.float64) * two["ng"][hit]).sum(1) > 0)


def test_peeling_visits_entry_and_exit_layers(oracle, scenes, tree):
    """A closed mesh seen from outside: two-sided peeling (tmin = the last t) yields front, back, front, back, ... at
    increasing t, the same sequence as brute force; one-sided peeling sees only the entries."""
    behind = (scenes.displaced_sphere(40).reshape(-1, 3) * 0.6 + np.float32([0.2, 0.1, 2.4])).reshape(-1, 9)
    tri = np.ascontiguousarray(np.concatenate([scenes.displaced_sphere(48), behind]), np.float32)
    pt = tree(oracle.Bih(tri))
    rays = oracle.camera_rays(scenes.pinhole_camera(origin=(0.1, 0.2, -2.5), aspect=1.0), 72, 72)
    seqs = {}
    for mode in ("box", "brute"):
        tmin = np.zeros(len(rays), np.float32)
        alive = np.ones(len(rays), bool)
        seq = [[] for _ in range(len(rays))]
        while alive.any():
            idx = np.nonzero(alive)[0]
            r = (pt.walk if mode == "box" else pt.brute)(rays8(rays[idx], tmin[idx], np.inf), two_sided=True)
            hit = r["slot"] >= 0
            side = (rays[idx[hit], 3:].astype(np.float64) * r["ng"][hit]).sum(1)
            for i, t, sd in zip(idx[hit], r["t"][hit], side):
                assert t > tmin[i]
                seq[i].append((float(t), "front" if sd < 0 else "back"))
            tmin[idx[hit]] = r["t"][hit]
            alive[idx[~hit]] = False
        seqs[mode] = seq
    assert seqs["box"] == seqs["brute"]
    depth = np.array([len(s) for s in seqs["box"]])
    alternating = np.array([all(f == ("front" if k % 2 == 0 else "back") for k, (_, f) in enumerate(s)) and len(s) % 2 == 0
                            for s in seqs["box"]])
    assert (depth >= 2).mean() > 0.2 and depth.max() >= 4
    assert alternating[depth > 0].mean() > 0.99                # a ray through a shared edge may skip one layer
    one = pt.walk(rays8(rays))
    entries = np.array([s[0][0] if s else FLT_MAX for s in seqs["box"]], np.float32)
    np.testing.assert_array_equal(bits(one["t"][alternating]), bits(entries[alternating]))


# ------------------------------------------------------------------------------------------------ GPU: the kernel

def gpu_intersect_host_and_device(renderer, r8, any_hit, outputs=OUTS):
    """The same two-sided query with numpy (host) buffers and with torch device buffers; returns both as numpy dicts."""
    import torch
    host = renderer.intersect(r8, any_hit=any_hit, two_sided=True, outputs=outputs)
    dev = renderer.intersect(torch.from_numpy(r8).cuda(), any_hit=any_hit, two_sided=True, outputs=outputs)
    return host, {k: x.cpu().numpy() for k, x in dev.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GOLDEN))
def test_two_sided_intersect_equals_restatement_bit_for_bit(renderer, oracle, scenes, tree, name):
    tri, cam, w, h = GOLDEN[name](scenes)
    ob = oracle.Bih(tri)
    pt = tree(ob)
    rays = oracle.camera_rays(cam, w, h)
    renderer.load_models(tri).build()
    t3, _, _ = ob.trace(rays, "box")
    tmin, tmax = assorted_intervals(t3, seed=19)
    r8 = rays8(rays, tmin, tmax)
    for any_hit in (False, True):
        want = pt.walk(r8, "any" if any_hit else "closest", two_sided=True)
        host, dev = gpu_intersect_host_and_device(renderer, r8, any_hit)
        assert_records_equal(host, want, msg="host any=%s" % any_hit)
        assert_records_equal(dev, want, msg="device any=%s" % any_hit)
    want = pt.walk(r8, two_sided=True)
    for subset in (("t",), ("slot", "prim"), ("u", "v"), ("ng",), ("t", "ng", "prim")):
        host, dev = gpu_intersect_host_and_device(renderer, r8, False, subset)
        assert set(host) == set(subset) == set(dev)
        assert_records_equal(host, want, subset, "host %s" % (subset,))
        assert_records_equal(dev, want, subset, "device %s" % (subset,))


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["inside_sphere", "inside_box"])
def test_camera_inside_equals_restatement(renderer, oracle, scenes, tree, which):
    """Inside the displaced sphere, and inside an axis-aligned box(n=8) with outward faces: the parity tree equals the
    restatement bit for bit (on the box that includes the reference's flat-geometry misses)."""
    tri, rays = (inside_sphere if which == "inside_sphere" else inside_box)(scenes, oracle, 320, 180)
    pt = tree(oracle.Bih(tri))
    renderer.load_models(tri).build()
    r8 = rays8(rays)
    for any_hit in (False, True):
        want = pt.walk(r8, "any" if any_hit else "closest", two_sided=True)
        host, dev = gpu_intersect_host_and_device(renderer, r8, any_hit)
        assert_records_equal(host, want, msg="host any=%s" % any_hit)
        assert_records_equal(dev, want, msg="device any=%s" % any_hit)
    hit = host["slot"] >= 0
    assert np.all((rays[hit, 3:].astype(np.float64) * host["ng"][hit]).sum(1) > 0)      # back faces only
    if which == "inside_sphere":
        assert hit.mean() > 0.995
    else:
        assert hit.mean() > 0.5
    assert (renderer.intersect(r8, outputs=("slot",))["slot"] >= 0).sum() == 0          # one-sided: nothing to see


@pytest.mark.gpu
@pytest.mark.parametrize("cap", [1, 4, 16])
@pytest.mark.parametrize("name", ["cornell", "sphere187", "atrium", "soup", "inside_box"])
def test_quality_mode_equals_two_sided_brute_force(renderer, oracle, scenes, tree, name, cap):
    if name == "inside_box":
        tri, rays = inside_box(scenes, oracle, 160, 160)
    else:
        tri, cam, w, h = GOLDEN[name](scenes)
        rays = oracle.camera_rays(cam, w, h)
    pt = tree(oracle.Bih(tri))
    renderer.set_option("morton_bits", 63)
    renderer.set_option("leaf_cap", cap)
    renderer.load_models(tri).build()
    tmin, tmax = assorted_intervals(pt.brute(rays8(rays), two_sided=True)["t"], seed=29)
    for r8 in (rays8(rays), rays8(rays, tmin, tmax)):
        want = pt.brute(r8, two_sided=True)
        got = renderer.intersect(r8, two_sided=True)
        near = bits(got["t"]) != bits(want["t"])
        assert near.sum() <= max(1, ID_MISMATCH_MAX * len(rays))       # coplanar tolerance
        assert_coplanar_near_ties(tri, rays, got, want, near)
        bad = (got["prim"] != want["prim"]) & ~near
        assert bad.sum() <= max(1, ID_MISMATCH_MAX * len(rays))        # tie tolerance (exact-t ties only)
        bad |= near
        # slots index the quality tree's own triangle order, not the oracle's: only hit / miss compares
        np.testing.assert_array_equal(got["slot"] >= 0, want["slot"] >= 0)
        same = ~bad
        rec = ("t", "u", "v", "prim", "ng")
        assert_records_equal({k: got[k][same] for k in rec}, {k: want[k][same] for k in rec}, rec)
        a = renderer.intersect(r8, any_hit=True, two_sided=True, outputs=("t", "slot"))
        np.testing.assert_array_equal(a["slot"] >= 0, want["slot"] >= 0)


@pytest.mark.gpu
def test_atrium_bounce_list_against_one_sided(renderer, scenes):
    """The atrium's diffuse bounce list on the GPU: two-sided records against one-sided ones (superset, t <=, front faces
    unchanged), and dot(d, ng) tells the side of every hit.  Many bounces leave through open or back-facing geometry."""
    tri, cam, w, h = scenes.atrium(0.3), scenes.atrium_camera(320 / 180), 320, 180
    renderer.load_models(tri).build()
    from bihrt import interval_rays
    rays, _ = renderer.secondary_rays(cam, w, h, spp=2, kind="diffuse", jitter=True)
    r8 = interval_rays(rays, 0.0, float("inf"))
    one = {k: x.cpu().numpy() for k, x in renderer.intersect(r8).items()}
    two = {k: x.cpu().numpy() for k, x in renderer.intersect(r8, two_sided=True).items()}
    front = check_against_one_sided(one, two, tri, rays.cpu().numpy())
    assert (~front).sum() > 100
    a = renderer.intersect(r8, any_hit=True, two_sided=True, outputs=("slot",))["slot"].cpu().numpy()
    np.testing.assert_array_equal(a >= 0, two["slot"] >= 0)


@pytest.mark.gpu
def test_per_sm_queue_launch(renderer, oracle, scenes, tree):
    """2^24 + 1 two-sided rays, many starting inside the sphere: the launch takes the per-SM work queues.  A sample of the
    rays equals the restatement bit for bit; all of them keep the properties against the one-sided query."""
    import torch
    from bihrt import interval_rays
    tri = scenes.displaced_sphere(187)
    pt = tree(oracle.Bih(tri))
    renderer.load_models(tri).build()
    g = torch.Generator(device="cuda").manual_seed(7)
    n = (1 << 24) + 1
    o = torch.rand((n, 3), device="cuda", generator=g) * 3 - 1.5
    target = torch.rand((n, 3), device="cuda", generator=g) - 0.5
    rays = torch.cat([o, target - o], 1).contiguous()
    r8 = interval_rays(rays, 0.0, float("inf"))
    one = {k: x.cpu().numpy() for k, x in renderer.intersect(r8).items()}
    two = {k: x.cpu().numpy() for k, x in renderer.intersect(r8, two_sided=True).items()}
    rays_np = rays.cpu().numpy()
    front = check_against_one_sided(one, two, tri, rays_np)
    assert (~front).sum() > n // 10
    pick = np.random.default_rng(3).choice(n, 200000, replace=False)
    want = pt.walk(rays8(rays_np[pick]), two_sided=True)
    assert_records_equal({k: two[k][pick] for k in OUTS}, want)


@pytest.mark.gpu
def test_error_codes(renderer, scenes):
    import bihrt
    lib = bihrt.load_library()
    ctx = renderer._ctx
    rays = np.zeros((4, 8), np.float32)
    rays[:, 6] = 1.0
    rays[:, 2] = -3.0
    rays[:, 7] = np.inf
    t = np.zeros(4, np.float32)
    hits = bihrt.Hits(t=t.ctypes.data)
    rp = C.c_void_p(rays.ctypes.data)
    for flags in (4, 5):
        assert lib.bihrt_intersect(ctx, rp, C.c_int64(4), C.c_uint32(flags), C.byref(hits)) == -4    # no BIH built yet
    renderer.load_models(scenes.dodecahedron()).build()
    for flags in (4, 5):
        assert lib.bihrt_intersect(ctx, rp, C.c_int64(4), C.c_uint32(flags), C.byref(hits)) == 0
        assert np.all(t < FLT_MAX)
    for flags in (2, 6, 8, 12, 0xFFFFFFF8, 0xFFFFFFFF):
        assert lib.bihrt_intersect(ctx, rp, C.c_int64(4), C.c_uint32(flags), C.byref(hits)) == -1, flags
    assert bihrt.INTERSECT_TWO_SIDED == 4
