"""Closest-point queries (bihrt_closest_point) on the CPU: the restatement's walk (tests/closest_oracle.c, the kernel's
order, margin and pruning) equals its brute force over every slot bit for bit in all seven outputs, on parity trees and on
quality trees at leaf caps 1, 4 and 16; an independent float64 computation from the input vertices confirms what the records
say; and the search radius means what include/bihrt.h says.  tests/test_gpu_closest.py holds the kernel to the walk.

The point sets and scenes here are shared with the GPU tests.
"""
import numpy as np
import pytest

from closest_oracle import CLOSEST_OUTS, closest  # noqa: F401  (closest: fixture)
from walk_oracle import FLT_MAX, bits, tree  # noqa: F401  (tree: fixture)

CAPS = (1, 4, 16)


# ------------------------------------------------------------------------------------------------ scenes

def needles_and_points(rng, n=400, exact=False):
    """Zero-area triangles: needles (three collinear vertices, one of them repeated or between the others) and point-triangles
    (three equal vertices), scattered in the unit cube, plus a few ordinary triangles so that the tree has shape.  exact: only
    needles with a repeated vertex, whose area is zero in binary32 too (a vertex between the others is collinear only up to
    rounding)."""
    a = rng.uniform(-1, 1, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32) * np.float32(0.05)
    k = rng.choice([0, 1, 3], n) if exact else rng.integers(0, 4, n)
    b = (a + d).astype(np.float32)
    c = np.select([k[:, None] == 0, k[:, None] == 1, k[:, None] == 2], [a, b, (a + np.float32(0.5) * d).astype(np.float32)],
                  (a + np.float32(2.0) * d).astype(np.float32))
    b[k == 3] = a[k == 3]
    pts = rng.integers(0, n, n // 8)
    b[pts] = a[pts]
    c[pts] = a[pts]
    tri = np.concatenate([a, b, c], 1)
    ordinary = np.concatenate([a[:40], a[:40] + rng.uniform(-0.05, 0.05, (40, 3)), a[:40] + rng.uniform(-0.05, 0.05, (40, 3))], 1)
    return np.concatenate([tri, ordinary]).astype(np.float32)


def identical(n=1000):
    """n copies of one triangle: every query ties across all of them, and the smallest slot must win."""
    return np.tile(np.array([[0.1, -0.2, 0.3, 0.7, 0.1, -0.1, -0.2, 0.6, 0.2]], np.float32), (n, 1))


def coplanar_grid(scenes):
    """Axis-aligned coplanar triangles, a floor of 32x32 quads in y = 0 plus a wall in x = 0.5: many leaves whose boxes are flat
    and share their planes."""
    floor = scenes.quad_grid((-1.0, 0.0, -1.0), (2.0, 0.0, 0.0), (0.0, 0.0, 2.0), 32, 32)
    wall = scenes.quad_grid((0.5, -1.0, -1.0), (0.0, 2.0, 0.0), (0.0, 0.0, 2.0), 8, 8)
    return np.concatenate([floor, wall]).astype(np.float32)


def scene_set(scenes):
    rng = np.random.default_rng(5)
    return {
        "dodecahedron": scenes.dodecahedron(),
        "cornell": scenes.cornell_box(),
        "sphere": scenes.displaced_sphere(64),
        "atrium": scenes.atrium(0.15),
        "soup": scenes.random_soup(5000, size=0.05),
        "needles": needles_and_points(rng),
        "needles_exact": needles_and_points(rng, exact=True),
        "identical": identical(),
        "coplanar": coplanar_grid(scenes),
    }


SCENE_NAMES = ("dodecahedron", "cornell", "sphere", "atrium", "soup", "needles", "needles_exact", "identical", "coplanar")


# ------------------------------------------------------------------------------------------------ points

def _lohi(tri):
    v = tri.reshape(-1, 3)
    return v.min(0), v.max(0)


def _normals(tri):
    t = tri.reshape(-1, 9).astype(np.float64)
    ng = np.cross(t[:, 3:6] - t[:, 0:3], t[:, 6:9] - t[:, 0:3])
    ln = np.linalg.norm(ng, axis=1, keepdims=True)
    return np.where(ln > 0, ng / np.where(ln > 0, ln, 1), 0.0)


def surface_points(tri, rng, k):
    """Vertices, edge midpoints and points inside triangles (what rays hit): k of each kind, exactly on the surface in
    binary32 where the coordinates allow it."""
    t = tri.reshape(-1, 9).astype(np.float32)
    i = rng.integers(0, len(t), (3, k))
    j = rng.integers(0, 3, k)
    vert = t[i[0]].reshape(-1, 3, 3)[np.arange(k), j]
    a, b = t[i[1]].reshape(-1, 3, 3)[np.arange(k), j], t[i[1]].reshape(-1, 3, 3)[np.arange(k), (j + 1) % 3]
    mid = ((a + b) * np.float32(0.5)).astype(np.float32)
    w = rng.dirichlet((1, 1, 1), k).astype(np.float32)
    inner = np.einsum("kj,kjc->kc", w, t[i[2]].reshape(-1, 3, 3)).astype(np.float32)
    return np.concatenate([vert, mid, inner]), np.concatenate([i[0], i[1], i[2]])


def hit_points(tri, cam, oracle, pt, w=48, h=27):
    """The closest hits of the camera's pixel-centre primary rays (the restatement's walk), with the hit triangle."""
    rays = oracle.camera_rays(cam, w, h)
    r = pt.walk(rays)
    hit = r["slot"] >= 0
    p = (rays[hit, 0:3] + r["t"][hit, None] * rays[hit, 3:6]).astype(np.float32)
    return p, r["prim"][hit]


def box_plane_points(pt, rng, k):
    """Points with one coordinate exactly on a plane of a child box of the tree (the other two from the same box, widened)."""
    nodes = pt.nodes[pt.reach] if len(pt.nodes) else pt.nodes
    if len(nodes) == 0:
        return np.zeros((0, 3), np.float32)
    boxes = nodes[:, 4:16].view(np.float32).reshape(-1, 6)
    b = boxes[rng.integers(0, len(boxes), k)]
    lo, hi = b[:, 0:3], b[:, 3:6]
    ext = np.maximum(hi - lo, 1e-3)
    p = rng.uniform(lo - 0.5 * ext, hi + 0.5 * ext).astype(np.float32)
    ax = rng.integers(0, 3, k)
    side = rng.integers(0, 2, k)
    p[np.arange(k), ax] = np.where(side == 0, lo[np.arange(k), ax], hi[np.arange(k), ax])
    return p


def point_set(tri, pt, oracle, cam, seed=1, k=300):
    """Every point set of the tests for one scene, as (N,3) float32: uniform in 1.5x the scene box; exactly on the surface
    (vertices, edge midpoints, inner points, ray hit points); the hit points moved +-1e-6 and +-1e-3 along the normal; points
    with a coordinate on a child-box plane; points 1e2..1e4 scene sizes away; points with NaN or infinite coordinates."""
    rng = np.random.default_rng(seed)
    lo, hi = _lohi(tri)
    c, ext = (lo + hi) * 0.5, np.maximum(hi - lo, 1e-3)
    uni = rng.uniform(c - 0.75 * ext, c + 0.75 * ext, (k, 3))
    surf, _ = surface_points(tri, rng, k // 3)
    hp, hprim = hit_points(tri, cam, oracle, pt)
    nrm = _normals(tri)
    moved = [hp + s * e * nrm[hprim] for e in (1e-6, 1e-3) for s in (-1.0, 1.0)]
    planes = box_plane_points(pt, rng, k)
    far_dir = rng.normal(size=(k // 3, 3))
    far_dir /= np.linalg.norm(far_dir, axis=1, keepdims=True)
    far = c + far_dir * (10.0 ** rng.uniform(2, 4, (k // 3, 1))) * ext.max()
    bad = rng.uniform(lo, hi, (12, 3))
    for i, val in enumerate((np.nan, np.inf, -np.inf)):
        bad[4 * i:4 * i + 4, np.arange(4) % 3] = val
    return np.concatenate([uni, surf, hp] + moved + [planes, far, bad]).astype(np.float32)


def queries(points, rmax=np.inf):
    from bihrt import point_queries
    return point_queries(np.asarray(points, np.float32), rmax)


def camera_for(name, scenes):
    return {"cornell": scenes.cornell_camera(), "atrium": scenes.atrium_camera()}.get(name, scenes.pinhole_camera(aspect=1.0))


def trees_of(name, tri, oracle, tree):
    """(label, Tree) for the parity tree and the quality trees at every cap"""
    yield "parity", tree(oracle.Bih(tri))
    for cap in CAPS:
        yield "q%d" % cap, tree(tri, cap)


def assert_closest_equal(got, want, msg=""):
    for k in CLOSEST_OUTS:
        np.testing.assert_array_equal(bits(got[k]), bits(want[k]), err_msg="%s %s" % (msg, k))


# ------------------------------------------------------------------------------------------------ float64 reference

def exact_distance(tri, p, pairs=False):
    """Distance (float64) from points p (N,3) to triangles tri (M,9) from the input vertices: the point's projection on the
    plane where it falls inside (normal equations for its barycentrics), otherwise the nearest of the three edge segments
    (clamped projections).  Returns (N, M), or with pairs=True (N,) for point i against triangle i."""
    t = tri.reshape(-1, 9).astype(np.float64)
    a, b, c = t[:, 0:3], t[:, 3:6], t[:, 6:9]
    p = np.asarray(p, np.float64)
    if not pairs:
        p = p[:, None, :]

    def seg(s0, s1):
        e = s1 - s0
        ee = (e * e).sum(-1)
        tt = np.clip(((p - s0) * e).sum(-1) / np.where(ee > 0, ee, 1.0), 0.0, 1.0)
        return np.linalg.norm(p - (s0 + tt[..., None] * e), axis=-1)
    dist = np.minimum(np.minimum(seg(a, b), seg(a, c)), seg(b, c))
    e1, e2 = b - a, c - a
    g11, g12, g22 = (e1 * e1).sum(-1), (e1 * e2).sum(-1), (e2 * e2).sum(-1)
    det = g11 * g22 - g12 * g12
    ok = det > 1e-30 * np.maximum(g11 * g22, 1e-300)
    r = p - a
    r1, r2 = (r * e1).sum(-1), (r * e2).sum(-1)
    sd = np.where(ok, det, 1.0)
    s, tt = (g22 * r1 - g12 * r2) / sd, (g11 * r2 - g12 * r1) / sd
    inside = ok & (s >= 0) & (tt >= 0) & (s + tt <= 1)
    proj = np.linalg.norm(r - s[..., None] * e1 - tt[..., None] * e2, axis=-1)
    return np.where(inside, np.minimum(proj, dist), dist)


# ------------------------------------------------------------------------------------------------ tests

@pytest.mark.parametrize("name", SCENE_NAMES)
def test_walk_equals_brute_force(oracle, scenes, tree, closest, name):
    tri = scene_set(scenes)[name]
    for label, pt in trees_of(name, tri, oracle, tree):
        q = queries(point_set(tri, pt, oracle, camera_for(name, scenes)))
        a, b = closest(pt, q), closest(pt, q, brute=True)
        assert_closest_equal(a, b, "%s %s" % (name, label))
        assert (a["slot"] >= 0).sum() == len(q) - 12                   # every finite point finds a triangle
        if name != "identical":                                         # (there every box ties with the best: all are walked)
            assert a["counters"]["tris"] < b["counters"]["tris"]


def test_walk_prunes_far_less_than_brute_force(oracle, scenes, tree, closest):
    tri = scenes.displaced_sphere(64)
    pt = tree(oracle.Bih(tri))
    q = queries(point_set(tri, pt, oracle, scenes.pinhole_camera(aspect=1.0)))
    a = closest(pt, q)
    assert a["counters"]["tris"] < 0.05 * len(q) * pt.n
    assert 0 < a["counters"]["max_stack"] <= 31


def test_without_margin_the_walk_loses_candidates(oracle, scenes, tree, closest):
    """The point sets catch a margin that is too small: with none at all the walk misses the brute-force result somewhere."""
    lost = 0
    for name in ("coplanar", "cornell", "needles", "sphere"):
        tri = scene_set(scenes)[name]
        for label, pt in trees_of(name, tri, oracle, tree):
            q = queries(point_set(tri, pt, oracle, camera_for(name, scenes)))
            a, b = closest(pt, q, margin_scale=0.0), closest(pt, q, brute=True)
            lost += int((a["slot"] != b["slot"]).sum())
    assert lost > 0


@pytest.mark.parametrize("name", ["cornell", "sphere", "soup", "needles_exact", "coplanar"])
def test_records_against_float64(oracle, scenes, tree, closest, name):
    tri = scene_set(scenes)[name]
    pt = tree(tri, 4)
    pts = point_set(tri, pt, oracle, camera_for(name, scenes), k=150)[::2]
    pts = pts[np.isfinite(pts).all(1)]
    r = closest(pt, queries(pts))
    assert (r["slot"] >= 0).all()
    lo, hi = _lohi(tri)
    mag = np.maximum(np.abs(pts).max(1), max(np.abs(lo).max(), np.abs(hi).max()))
    tol = 1e-5 * mag
    dist = exact_distance(tri, pts)
    dmin = dist.min(1)
    idx = np.arange(len(pts))
    assert np.all(np.abs(np.sqrt(r["d2"].astype(np.float64)) - dmin) <= tol)
    assert np.all(dist[idx, r["prim"]] - dmin <= tol)
    assert np.all(r["u"] >= 0) and np.all(r["v"] >= 0) and np.all(r["u"].astype(np.float64) + r["v"] <= 1 + 1e-6)
    on = exact_distance(tri.reshape(-1, 9)[r["prim"]], r["q"], pairs=True)
    assert np.all(on <= tol)
    # q is the reported point: d2 is |p - q|^2 within rounding
    dq = np.linalg.norm(pts.astype(np.float64) - r["q"], axis=1)
    assert np.all(np.abs(dq - np.sqrt(r["d2"].astype(np.float64))) <= tol)
    # ng is e1 x e2 of the reported triangle
    t = tri.reshape(-1, 9)[r["prim"]].astype(np.float64)
    ng = np.cross(t[:, 3:6] - t[:, 0:3], t[:, 6:9] - t[:, 0:3])
    assert np.allclose(r["ng"], ng, rtol=1e-5, atol=1e-6 * mag.max() ** 2)


def radius_cases(d2_unbounded, rng):
    """Per-point rmax drawn from {inf, FLT_MAX, 0, negative, NaN, just below the nearest distance, the smallest binary32 whose
    square rounds to at least the nearest d2}.  Returns rmax and the kind of each."""
    n = len(d2_unbounded)
    kind = rng.integers(0, 7, n)
    hit = np.empty(n, np.float32)
    f = np.float32
    for i, d2 in enumerate(d2_unbounded):
        r = f(np.sqrt(np.float64(d2)))
        while f(r * r) < d2:
            r = np.nextafter(r, f(np.inf))
        while r > 0 and f(np.nextafter(r, f(0)) * np.nextafter(r, f(0))) >= d2:
            r = np.nextafter(r, f(0))
        hit[i] = r
    below = np.nextafter(hit, np.float32(0))
    rmax = np.select([kind == 0, kind == 1, kind == 2, kind == 3, kind == 4, kind == 5],
                     [np.full(n, np.inf), np.full(n, FLT_MAX), np.zeros(n), -rng.uniform(0, 1, n), np.full(n, np.nan), below],
                     hit).astype(np.float32)
    return rmax, kind


@pytest.mark.parametrize("name", ["cornell", "sphere", "identical", "coplanar"])
def test_radius(oracle, scenes, tree, closest, name):
    tri = scene_set(scenes)[name]
    for label, pt in trees_of(name, tri, oracle, tree):
        pts = point_set(tri, pt, oracle, camera_for(name, scenes), seed=3)
        pts = pts[np.isfinite(pts).all(1)]
        full = closest(pt, queries(pts), brute=True)
        rmax, kind = radius_cases(full["d2"], np.random.default_rng(9))
        q = queries(pts, rmax)
        a, b = closest(pt, q), closest(pt, q, brute=True)
        assert_closest_equal(a, b, "%s %s" % (name, label))
        unbounded = (kind <= 1) | (kind == 6)
        zero_hit = ((kind == 2) | (kind == 5)) & (full["d2"] == 0)       # (no radius lies below a distance of 0)
        want_hit = unbounded | zero_hit
        np.testing.assert_array_equal(a["slot"] >= 0, want_hit, err_msg=label)
        for k in CLOSEST_OUTS:
            np.testing.assert_array_equal(bits(a[k][want_hit]), bits(full[k][want_hit]), err_msg="%s %s" % (label, k))
        miss = ~want_hit
        assert np.all(a["d2"][miss] == FLT_MAX) and np.all(a["prim"][miss] == -1)
        assert np.all(a["u"][miss] == 0) and np.all(a["v"][miss] == 0)
        assert np.all(a["q"][miss] == 0) and np.all(a["ng"][miss] == 0)
        assert (kind == 5).sum() > 0 and (kind == 6).sum() > 0


def test_identical_triangles_report_the_smallest_slot(tree, closest):
    tri = identical()
    for cap in CAPS:
        pt = tree(tri, cap)
        rng = np.random.default_rng(2)
        r = closest(pt, queries(rng.uniform(-1, 1, (500, 3))))
        assert np.all(r["slot"] == 0)


def test_nonfinite_points_and_bad_radii_miss_without_a_walk(oracle, scenes, tree, closest):
    tri = scenes.cornell_box()
    pt = tree(oracle.Bih(tri))
    p = np.array([[np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf], [0.1, 0.2, 0.3], [0.1, 0.2, 0.3]], np.float32)
    r = closest(pt, queries(p, np.array([np.inf, np.inf, np.inf, np.nan, -1.0], np.float32)))
    np.testing.assert_array_equal(r["slot"], -1)
    assert np.all(r["d2"] == FLT_MAX)
    assert r["counters"] == {"nodes": 0, "tris": 0, "max_stack": 0}
