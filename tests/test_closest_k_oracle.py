"""k-nearest-triangle queries (bihrt_closest_k) on the CPU: the restatement's walk (tests/closest_k_oracle.c, the kernel's list,
order, margin and pruning) equals brute force over every slot bit for bit in all nine outputs, on parity trees and on quality
trees at leaf caps 1, 4 and 16, for k in {1, 3, 8, 64}, with unbounded radii and radii at a point's j-th nearest distance, and
with and without the total.  At k = 1 the rows are bihrt_closest_point's records.  tests/test_gpu_closest_k.py holds the
kernel to the walk.
"""
import numpy as np
import pytest

from closest_k_oracle import CLOSEST_K_OUTS, K_MAX, closest_k  # noqa: F401  (closest_k: fixture)
from closest_oracle import CLOSEST_OUTS, closest  # noqa: F401  (closest: fixture)
from test_closest_oracle import CAPS, SCENE_NAMES, camera_for, identical, point_set, queries, radius_cases, scene_set
from walk_oracle import FLT_MAX, bits, tree  # noqa: F401  (tree: fixture)

KS = (1, 3, 8, 64)
RADIUS_COLUMN = 3               # the radius cases sit at each point's 4th nearest distance


def trees_of(tri, oracle, tree):
    """(label, Tree) for the parity tree and the quality trees at every cap"""
    yield "parity", tree(oracle.Bih(tri))
    for cap in CAPS:
        yield "q%d" % cap, tree(tri, cap)


def k_points(tri, pt, oracle, cam, seed=1):
    """point_set thinned to every other point, or fewer on large scenes (brute force and the walk with the total are O(n) per
    point), keeping its 12 points with NaN or infinite coordinates (the last ones)"""
    pts = point_set(tri, pt, oracle, cam, seed=seed)
    return np.concatenate([pts[:-12][::max(2, pt.n // 2500)], pts[-12:]])


def assert_k_equal(got, want, msg="", outs=CLOSEST_K_OUTS):
    for o in outs:
        if o in got and o in want:
            np.testing.assert_array_equal(bits(got[o]), bits(want[o]), err_msg="%s %s" % (msg, o))


def prefix(full, k):
    """The result at k from brute force at K_MAX with the total: the first k rows, count = min(total, k).  (The contract's
    rows are a prefix of the ordered candidates, so this is what every k must give.)"""
    r = {o: full[o][:, :k] for o in CLOSEST_OUTS}
    r["count"] = np.minimum(full["total"], k).astype(np.int32)
    r["total"] = full["total"]
    return r


def radius_queries(pts, full, seed):
    """Queries at the finite points with radius cases placed at each one's RADIUS_COLUMN-th nearest distance"""
    fin = np.isfinite(pts).all(1)
    rmax, kind = radius_cases(full["d2"][fin, RADIUS_COLUMN], np.random.default_rng(seed))
    return queries(pts[fin], rmax), kind


@pytest.mark.parametrize("name", SCENE_NAMES)
def test_walk_equals_brute_force(oracle, scenes, tree, closest_k, name):
    tri = scene_set(scenes)[name]
    for label, pt in trees_of(tri, oracle, tree):
        pts = k_points(tri, pt, oracle, camera_for(name, scenes))
        q = queries(pts)
        full = closest_k(pt, q, K_MAX, total=True, brute=True)
        qr, _ = radius_queries(pts, full, 4)
        full_r = closest_k(pt, qr, K_MAX, total=True, brute=True)
        for case, qq, ref in (("unbounded", q, full), ("radii", qr, full_r)):
            for k in KS:
                want = prefix(ref, k)
                for total in (False, True):
                    got = closest_k(pt, qq, k, total=total)
                    assert_k_equal(got, want, "%s %s %s k=%d total=%s" % (name, label, case, k, total))
                if case == "unbounded":          # brute force at k itself: the same prefix
                    assert_k_equal(closest_k(pt, qq, k, total=True, brute=True), want, "%s %s k=%d brute" % (name, label, k))
        # every finite point has candidates at an unbounded radius; the radius cases cut some of them off
        assert (full["count"] > 0).sum() == len(q) - 12
        assert (full_r["total"] < full["total"][np.isfinite(pts).all(1)]).any()


def test_brute_force_rows_are_the_ordered_candidates(oracle, scenes, tree, closest_k):
    """Brute force at k >= n lists every triangle: ascending (d2, slot), each slot once, count == total == n"""
    tri = scenes.dodecahedron()
    pt = tree(oracle.Bih(tri))
    assert pt.n <= K_MAX
    pts = np.random.default_rng(0).uniform(-2, 2, (500, 3)).astype(np.float32)
    r = closest_k(pt, queries(pts), K_MAX, total=True, brute=True)
    n = pt.n
    assert np.all(r["count"] == n) and np.all(r["total"] == n)
    key = r["d2"][:, :n].view(np.uint32).astype(np.uint64) << np.uint64(32) | r["slot"][:, :n].astype(np.uint64)
    assert np.all(np.diff(key.astype(np.int64), axis=1) > 0)
    np.testing.assert_array_equal(np.sort(r["slot"][:, :n], axis=1), np.tile(np.arange(n), (len(pts), 1)))


@pytest.mark.parametrize("name", ["cornell", "sphere", "needles", "identical", "coplanar"])
def test_k1_rows_are_closest_point_records(oracle, scenes, tree, closest, closest_k, name):
    tri = scene_set(scenes)[name]
    for label, pt in trees_of(tri, oracle, tree):
        pts = k_points(tri, pt, oracle, camera_for(name, scenes), seed=2)
        full = closest_k(pt, queries(pts), K_MAX, total=True, brute=True)
        qr, _ = radius_queries(pts, full, 5)
        for qq in (queries(pts), qr):
            a, b = closest_k(pt, qq, 1), closest(pt, qq)
            for o in CLOSEST_OUTS:
                np.testing.assert_array_equal(bits(a[o][:, 0]), bits(b[o]), err_msg="%s %s %s" % (name, label, o))
            np.testing.assert_array_equal(a["count"], (b["slot"] >= 0).astype(np.int32))


def test_ties_go_to_the_smaller_slots(tree, closest_k):
    tri = identical()
    pts = np.random.default_rng(2).uniform(-1, 1, (300, 3)).astype(np.float32)
    for cap in CAPS:
        pt = tree(tri, cap)
        for k in KS:
            for total in (False, True):
                r = closest_k(pt, queries(pts), k, total=total)
                np.testing.assert_array_equal(r["slot"], np.tile(np.arange(k, dtype=np.int32), (len(pts), 1)))
                assert np.all(r["count"] == k)
                assert np.all(r["d2"] == r["d2"][:, :1])
                if total:
                    assert np.all(r["total"] == 1000)


def test_k_larger_than_the_mesh(oracle, scenes, tree, closest_k):
    tri = scenes.dodecahedron()
    pts = np.random.default_rng(3).uniform(-2, 2, (400, 3)).astype(np.float32)
    for pt in (tree(oracle.Bih(tri)), tree(tri, 4)):
        n = pt.n
        for total in (False, True):
            r = closest_k(pt, queries(pts), 64, total=total)
            assert np.all(r["count"] == n)
            assert np.all(r["slot"][:, :n] >= 0)
            assert np.all(r["d2"][:, n:] == FLT_MAX) and np.all(r["slot"][:, n:] == -1) and np.all(r["prim"][:, n:] == -1)
            for o in ("u", "v", "q", "ng"):
                assert np.all(r[o][:, n:] == 0), o
            assert_k_equal(r, closest_k(pt, queries(pts), 64, total=total, brute=True), "dodecahedron total=%s" % total)


def test_k0_counts_only(oracle, scenes, tree, closest_k):
    tri = scenes.cornell_box()
    pt = tree(oracle.Bih(tri))
    rng = np.random.default_rng(4)
    pts = rng.uniform(-1.2, 1.2, (2000, 3)).astype(np.float32)
    q = queries(pts, rng.uniform(0, 0.5, 2000).astype(np.float32))
    want = closest_k(pt, q, K_MAX, total=True, brute=True)
    r = closest_k(pt, q, 0, total=True)
    assert all(r[o].shape[1] == 0 for o in CLOSEST_OUTS)
    assert np.all(r["count"] == 0)
    np.testing.assert_array_equal(r["total"], want["total"])
    assert (want["total"] > 1).any() and (want["total"] == 0).any()
    r = closest_k(pt, q, 0)                  # nothing is asked: no walk
    assert np.all(r["count"] == 0) and r["counters"] == {"nodes": 0, "tris": 0, "max_stack": 0}


def test_dead_queries_have_no_candidates(oracle, scenes, tree, closest_k):
    tri = scenes.cornell_box()
    pt = tree(oracle.Bih(tri))
    p = np.array([[np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf], [0.1, 0.2, 0.3], [0.1, 0.2, 0.3]], np.float32)
    q = queries(p, np.array([np.inf, np.inf, np.inf, np.nan, -1.0], np.float32))
    for k in (0, 3):
        for brute in (False, True):
            r = closest_k(pt, q, k, total=True, brute=brute)
            assert np.all(r["count"] == 0) and np.all(r["total"] == 0)
            assert np.all(r["slot"] == -1) and np.all(r["prim"] == -1) and np.all(r["d2"] == FLT_MAX)
            assert np.all(r["u"] == 0) and np.all(r["v"] == 0) and np.all(r["q"] == 0) and np.all(r["ng"] == 0)
            assert r["counters"] == {"nodes": 0, "tris": 0, "max_stack": 0}


def test_total_keeps_the_records_and_costs_more(oracle, scenes, tree, closest_k):
    tri = scenes.displaced_sphere(64)
    for pt in (tree(oracle.Bih(tri)), tree(tri, 4)):
        pts = k_points(tri, pt, oracle, scenes.pinhole_camera(aspect=1.0))
        q = queries(pts, 0.05)
        for k in (1, 8):
            a, b = closest_k(pt, q, k), closest_k(pt, q, k, total=True)
            assert_k_equal(a, b, "k=%d" % k, CLOSEST_OUTS + ("count",))
            assert a["counters"]["tris"] < b["counters"]["tris"]
            assert (b["total"] > k).any()
        # the k-walk prunes: far fewer distance evaluations than brute force
        assert closest_k(pt, queries(pts), 8)["counters"]["tris"] < 0.05 * len(pts) * pt.n


def test_without_margin_the_walk_loses_candidates(oracle, scenes, tree, closest_k):
    """The point sets of DESIGN.md section 8 catch a margin that is too small for the k-walk too"""
    lost = 0
    for name in ("coplanar", "cornell", "needles", "sphere"):
        tri = scene_set(scenes)[name]
        for label, pt in trees_of(tri, oracle, tree):
            q = queries(point_set(tri, pt, oracle, camera_for(name, scenes)))
            a, b = closest_k(pt, q, 8, margin_scale=0.0), closest_k(pt, q, 8, brute=True)
            lost += int((a["slot"] != b["slot"]).any(1).sum())
    assert lost > 0
