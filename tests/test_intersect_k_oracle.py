"""Multi-hit ray queries (bihrt_intersect_k) on the CPU: the restatement's walk (tests/intersect_k_oracle.c: walk_oracle.c's
walk with a list of the k nearest keys and the list's closed cut) against walk_oracle's closest-hit walk at k = 1, against brute
force over every slot on quality trees at leaf caps 1, 4 and 16 and on parity trees, and the contract's properties: ties,
prefixes, the peeling relation, counts and totals, k = 0, dead rays and the cost of the total.
tests/test_gpu_intersect_k.py holds the kernel to the walk.
"""
import numpy as np
import pytest

from intersect_k_oracle import K_MAX, K_OUTS, intersect_k  # noqa: F401  (intersect_k: fixture)
from test_closest_oracle import CAPS, coplanar_grid, identical
from test_gpu_golden_scenes import SCENES as GOLDEN
from walk_oracle import FLT_MAX, OUTS, assorted_intervals, bits, degenerate_rays, mt, rays8, tree  # noqa: F401  (tree: fixture)

KS = (1, 3, 8, 64)


def assert_k_equal(got, want, msg="", outs=K_OUTS):
    for o in outs:
        if o in got and o in want:
            np.testing.assert_array_equal(bits(got[o]), bits(want[o]), err_msg="%s %s" % (msg, o))


def keys(r):
    """(N,k) uint64 keys t_bits << 32 | slot of the rows (misses: FLT_MAX << 32 | 2^32 - 1)"""
    return r["t"].view(np.uint32).astype(np.uint64) << np.uint64(32) | r["slot"].view(np.uint32).astype(np.uint64)


def prefix(full, k):
    """The result at k from a result at K_MAX with the total: the first k rows, count = min(total, k)."""
    r = {o: full[o][:, :k] for o in OUTS}
    r["count"] = np.minimum(full["total"], k).astype(np.int32)
    r["total"] = full["total"]
    return r


def k_scenes(scenes):
    """name -> (triangles, camera rays (N,6)) at resolutions brute force over every slot can afford"""
    from oracle import oracle as O
    out = {}
    for name, w, h in (("cornell", 48, 48), ("sphere187", 64, 36), ("atrium", 64, 36), ("soup", 32, 18)):
        tri, cam, _, _ = GOLDEN[name](scenes)
        out[name] = (tri, O.camera_rays(cam, w, h))
    tri = scenes.random_soup(20000, size=0.05)
    out["layers"] = (tri, O.camera_rays(scenes.pinhole_camera(), 48, 27))
    rng = np.random.default_rng(5)
    one = identical(1).reshape(3, 3).astype(np.float64)        # rays towards points around the triangle, from its front side
    ng = np.cross(one[1] - one[0], one[2] - one[0])
    uv = rng.uniform(-0.2, 0.8, (600, 2))
    p = one[0] + uv[:, :1] * (one[1] - one[0]) + uv[:, 1:] * (one[2] - one[0])
    o = p + 3 * ng / np.linalg.norm(ng) + rng.normal(scale=0.3, size=(600, 3))
    out["identical"] = (identical(), np.concatenate([o, p - o], 1).astype(np.float32))
    grid = coplanar_grid(scenes)
    v = grid.reshape(-1, 3)
    lo, hi = v.min(0), v.max(0)
    o = rng.uniform(lo - 0.2 * (hi - lo) - 1, hi + 0.2 * (hi - lo) + 1, (1500, 3))
    d = rng.uniform(lo, hi, (1500, 3)) - o
    out["coplanar"] = (grid, np.concatenate([o, d], 1).astype(np.float32))
    return out


def intervals(rays, pt, seed):
    """rays8 with assorted_intervals around each ray's closest hit"""
    t0 = pt.walk(rays8(rays))["t"]
    tmin, tmax = assorted_intervals(t0, seed)
    return rays8(rays, tmin, tmax)


# ------------------------------------------------------------------------------------------------ anchor: walk_oracle's walk

@pytest.mark.parametrize("two_sided", [False, True])
@pytest.mark.parametrize("name", list(GOLDEN) + ["degenerate"])
def test_k1_is_the_closest_hit_walk(oracle, scenes, tree, intersect_k, name, two_sided):
    """k = 1 without the total: t bit for bit the closest-hit walk's; the slot too, except on exact-t ties, where the k-walk
    has the smaller slot and both triangles are hit at that t."""
    if name == "degenerate":
        tri, rays = degenerate_rays(scenes)
    else:
        tri, cam, w, h = GOLDEN[name](scenes)
        rays = oracle.camera_rays(cam, w, h)
    pt = tree(oracle.Bih(tri))
    r8 = intervals(rays, pt, 31)
    for case, rr in (("full", rays8(rays)), ("intervals", r8)):
        a = pt.walk(rr, two_sided=two_sided)
        b = intersect_k(pt, rr, 1, two_sided=two_sided)
        np.testing.assert_array_equal(bits(b["t"][:, 0]), bits(a["t"]), err_msg="%s %s" % (name, case))
        np.testing.assert_array_equal(b["count"], (a["slot"] >= 0).astype(np.int32))
        tie = b["slot"][:, 0] != a["slot"]
        assert np.all(b["slot"][tie, 0] < a["slot"][tie]), name
        for s in (b["slot"][tie, 0], a["slot"][tie]):
            ok, _, t, _, _ = mt(tri, pt.tris[s, 9], rays[tie], two_sided)
            assert ok.all() and np.array_equal(bits(t), bits(a["t"][tie])), name
        same = ~tie
        for o in ("u", "v", "prim", "ng"):
            np.testing.assert_array_equal(bits(b[o][same, 0]), bits(a[o][same]), err_msg="%s %s %s" % (name, case, o))


# ------------------------------------------------------------------------------------------------ brute force

@pytest.mark.parametrize("two_sided", [False, True])
@pytest.mark.parametrize("name", ["cornell", "sphere187", "atrium", "soup", "layers", "identical", "coplanar"])
def test_quality_walk_equals_brute_force(oracle, scenes, tree, intersect_k, name, two_sided):
    tri, rays = k_scenes(scenes)[name]
    for cap in CAPS:
        pt = tree(tri, cap)
        r8 = intervals(rays, pt, 7)
        for rr in (rays8(rays), r8):
            full = intersect_k(pt, rr, K_MAX, total=True, two_sided=two_sided, brute=True)
            for k in KS:
                want = prefix(full, k)
                for total in (False, True):
                    got = intersect_k(pt, rr, k, total=total, two_sided=two_sided)
                    assert_k_equal(got, want, "%s q%d k=%d total=%s" % (name, cap, k, total))
        assert (full["total"] > 0).any()


@pytest.mark.parametrize("name", ["cornell", "sphere187", "atrium", "soup", "layers"])
def test_parity_rows_are_ordered_candidates(oracle, scenes, tree, intersect_k, name):
    """Every row is an accepted triangle of brute force, rows ascend by (t, slot), and the walk's rows at K_MAX with the total
    are the candidates it reaches: a subset of brute force's, in its order -- all of them on the sphere and the soup, where no
    geometry lies in the parity tree's split planes; on the Cornell box and the atrium the missing ones are the flat-geometry
    class (DESIGN.md section 2)."""
    tri, rays = k_scenes(scenes)[name]
    pt = tree(oracle.Bih(tri))
    rr = intervals(rays, pt, 3)
    for two_sided in (False, True):
        full = intersect_k(pt, rr, K_MAX, total=True, two_sided=two_sided, brute=True)
        got = intersect_k(pt, rr, K_MAX, total=True, two_sided=two_sided)
        kg, kb = keys(got), keys(full)
        both = np.arange(1, K_MAX)[None, :] < got["count"][:, None]        # rows j - 1 and j are written
        assert np.all((kg[:, 1:] > kg[:, :-1])[both])
        lost = 0
        for i in range(len(rr)):
            g, b = kg[i, :got["count"][i]], set(kb[i, :full["count"][i]].tolist())
            assert set(g.tolist()) <= b, (name, i)
            lost += len(b) - len(g)
        assert np.all(got["total"] <= full["total"])
        if name in ("sphere187", "soup", "layers"):
            assert lost == 0
            assert_k_equal(got, full, name)
        for k in KS:
            assert_k_equal(intersect_k(pt, rr, k, two_sided=two_sided), prefix(got, k), "%s k=%d" % (name, k),
                           OUTS + ("count",))


# ------------------------------------------------------------------------------------------------ contract properties

def test_ties_are_consecutive_rows_in_slot_order(oracle, tree, intersect_k, scenes):
    """1000 identical triangles: every row of a ray through them has the same t and the rows' slots ascend from 0 -- peeling
    sees one of them."""
    tri, rays = k_scenes(scenes)["identical"]
    for pt in (tree(oracle.Bih(tri)), tree(tri, 4)):
        for k in KS:
            for total in (False, True):
                r = intersect_k(pt, rays8(rays), k, total=total)
                hit = r["count"] > 0
                assert hit.mean() > 0.3
                assert np.all(r["count"][hit] == k)
                np.testing.assert_array_equal(r["slot"][hit], np.tile(np.arange(k, dtype=np.int32), (hit.sum(), 1)))
                assert np.all(r["t"][hit] == r["t"][hit, :1])
                if total:
                    assert np.all(r["total"][hit] == 1000)
        peel = pt.walk(rays8(rays, r["t"][:, 0], np.inf))
        assert np.all(peel["slot"][hit] == -1)              # the next peel skips the 999 others


@pytest.mark.parametrize("two_sided", [False, True])
def test_peeling_yields_the_distinct_t_of_the_rows(oracle, scenes, tree, intersect_k, two_sided):
    """tests/test_gpu_intersect.py's peeling construction: where total <= K_MAX the distinct t of the rows are the peeled
    sequence, on the parity tree and on a quality tree."""
    tri = scenes.random_soup(20000, size=0.05)
    rays = oracle.camera_rays(scenes.pinhole_camera(), 64, 36)
    for pt in (tree(oracle.Bih(tri)), tree(tri, 4)):
        r = intersect_k(pt, rays8(rays), K_MAX, total=True, two_sided=two_sided)
        tmin = np.zeros(len(rays), np.float32)
        alive = np.ones(len(rays), bool)
        seq = [[] for _ in range(len(rays))]
        while alive.any():
            idx = np.nonzero(alive)[0]
            p = pt.walk(rays8(rays[idx], tmin[idx], np.inf), two_sided=two_sided)
            hit = p["slot"] >= 0
            for i, t in zip(idx[hit], p["t"][hit]):
                seq[i].append(float(t))
            tmin[idx[hit]] = p["t"][hit]
            alive[idx[~hit]] = False
        ok = r["total"] <= K_MAX
        assert ok.mean() > 0.9 and (r["total"] >= 5).any()
        for i in np.nonzero(ok)[0]:
            rows = r["t"][i, :r["count"][i]].tolist()
            assert sorted(set(rows)) == seq[i], i


@pytest.mark.parametrize("name", ["cornell", "atrium", "layers"])
def test_prefix_count_and_total(oracle, scenes, tree, intersect_k, name):
    """The rows at k are the first k rows at K_MAX; count = min(k, total); pruned and total-mode rows are equal, and the
    total costs more triangle tests."""
    tri, rays = k_scenes(scenes)[name]
    for pt in (tree(oracle.Bih(tri)), tree(tri, 4)):
        for two_sided in (False, True):
            rr = intervals(rays, pt, 13)
            full = intersect_k(pt, rr, K_MAX, total=True, two_sided=two_sided)
            for k in KS:
                a = intersect_k(pt, rr, k, two_sided=two_sided)
                b = intersect_k(pt, rr, k, total=True, two_sided=two_sided)
                assert_k_equal(b, prefix(full, k), "%s k=%d total" % (name, k))
                assert_k_equal(a, b, "%s k=%d pruned" % (name, k), OUTS + ("count",))
                np.testing.assert_array_equal(b["count"], np.minimum(b["total"], k))
                assert a["counters"]["tris"] <= b["counters"]["tris"]
                if k == 1:
                    assert a["counters"]["tris"] < b["counters"]["tris"]


def test_k0_counts_crossings_only(oracle, scenes, tree, intersect_k):
    """k = 0 with the total counts the accepted triangles (two-sided on a closed mesh: odd inside, even outside); without it
    nothing is walked."""
    tri = scenes.displaced_sphere(48)
    rng = np.random.default_rng(4)
    o = rng.uniform(-1.5, 1.5, (3000, 3)).astype(np.float32)
    d = rng.normal(size=(3000, 3)).astype(np.float32)
    rays = np.concatenate([o, d], 1)
    for pt in (tree(oracle.Bih(tri)), tree(tri, 4)):
        want = intersect_k(pt, rays8(rays), K_MAX, total=True, two_sided=True, brute=True)
        r = intersect_k(pt, rays8(rays), 0, total=True, two_sided=True)
        assert all(r[o_].shape[1] == 0 for o_ in OUTS)
        assert np.all(r["count"] == 0)
        np.testing.assert_array_equal(r["total"], want["total"])
        inside = np.linalg.norm(o, axis=1) < 0.5
        assert np.all(r["total"][inside] % 2 == 1)
        assert (r["total"] == 0).any() and (r["total"] >= 2).any()
        r = intersect_k(pt, rays8(rays), 0)
        assert np.all(r["count"] == 0) and r["counters"] == {"nodes": 0, "tris": 0, "max_stack": 0}


def test_dead_rays_have_no_candidates(oracle, scenes, tree, intersect_k):
    tri = scenes.cornell_box()
    pt = tree(oracle.Bih(tri))
    rays = np.tile(np.array([[0, 0, -3, 0, 0, 1]], np.float32), (5, 1))
    tmin = np.array([np.nan, 0.0, 2.0, 1.0, 0.0], np.float32)
    tmax = np.array([np.inf, np.nan, 2.0, 0.5, -1.0], np.float32)
    for k in (0, 3):
        for brute in (False, True):
            r = intersect_k(pt, rays8(rays, tmin, tmax), k, total=True, brute=brute)
            assert np.all(r["count"] == 0) and np.all(r["total"] == 0)
            assert np.all(r["slot"] == -1) and np.all(r["prim"] == -1) and np.all(r["t"] == FLT_MAX)
            assert np.all(r["u"] == 0) and np.all(r["v"] == 0) and np.all(r["ng"] == 0)
            assert r["counters"] == {"nodes": 0, "tris": 0, "max_stack": 0}
    assert (intersect_k(pt, rays8(rays[:1]), 3, total=True)["total"] > 0).all()
