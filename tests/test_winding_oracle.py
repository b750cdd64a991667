"""Winding-number queries (bihrt_winding_number) on the CPU: the restatement's walk (tests/winding_oracle.c: the far-field
table, the kernel's walk order and accumulation) in exact mode equals its brute force over every slot bit for bit on parity
trees and on quality trees at leaf caps 1, 4 and 16; against an independent float64 solid-angle sum over the input triangles
it classifies closed meshes exactly and stays within the stated error per beta; the table is checked against per-subtree
float64 moments; special points never give NaN.  tests/test_gpu_winding.py holds the kernel to the walk.

Tolerances: the largest errors the restatement shows on these scenes (DESIGN.md section 9), doubled.
  exact mode (beta = inf) against float64: 2e-6 for points at least 1e-3 of the scene diagonal off the surface (largest seen
    9.1e-7).  Each triangle's term carries the binary32 rounding of det = a.(b x c), about 2^-24 |a||b||c|, so the error
    grows with the number of triangles and near the surface, not with beta;
  beta 2 / 3 / 4 against float64: 3e-2 / 6e-3 / 1.5e-3 (largest seen 1.5e-2 / 3.0e-3 / 5.8e-4, all on the atrium): the
    truncation of the order-2 expansion.
"""
from types import SimpleNamespace

import numpy as np
import pytest

from closest_oracle import closest  # noqa: F401  (fixture)
from test_closest_oracle import (CAPS, SCENE_NAMES, camera_for, point_set, queries, scene_set, surface_points,
                                 trees_of)
from walk_oracle import bits, tree  # noqa: F401  (fixture)
from winding_oracle import WREC, winding  # noqa: F401  (fixture)

EXACT_TOL = 2e-6
BETA_TOL = {2.0: 3e-2, 3.0: 6e-3, 4.0: 1.5e-3}


# ------------------------------------------------------------------------------------------------ scenes and points

def overlapping_spheres(scenes):
    """Two closed spheres of 8 k triangles, overlapping: w = 2 where both contain the point."""
    s = scenes.displaced_sphere(64).reshape(-1, 3, 3)
    return np.concatenate([s, s + np.float32([0.8, 0.1, 0.0])]).reshape(-1, 9).astype(np.float32)


def closed_scenes(scenes):
    return {
        "dodecahedron": scenes.dodecahedron(),
        "sphere_70k": scenes.displaced_sphere(scenes.SPHERE_NSEG["70k"]),
        "sphere_260k": scenes.displaced_sphere(scenes.SPHERE_NSEG["260k"]),
        "box_n4": scenes.box([-1, -0.5, -0.7], [1, 0.5, 0.7], n=4),
        "box_n4_inward": scenes.box([-1, -0.5, -0.7], [1, 0.5, 0.7], inward=True, n=4),
        "overlapping_spheres": overlapping_spheres(scenes),
    }


def _lohi(tri):
    v = tri.reshape(-1, 3)
    return v.min(0).astype(np.float64), v.max(0).astype(np.float64)


def sample_points(tri, rng, k=400):
    """Uniform in 1.2x the scene box, and points near the surface (inner points of triangles moved along the normal by
    1e-3 .. 3e-2 of the scene diagonal, both sides)."""
    lo, hi = _lohi(tri)
    c, ext = (lo + hi) * 0.5, hi - lo
    uni = rng.uniform(c - 0.6 * ext, c + 0.6 * ext, (k, 3))
    t = tri.reshape(-1, 3, 3)[rng.integers(0, len(tri), k)].astype(np.float64)
    w = rng.dirichlet((1, 1, 1), k)
    nrm = np.cross(t[:, 1] - t[:, 0], t[:, 2] - t[:, 0])
    nrm /= np.maximum(np.linalg.norm(nrm, axis=1, keepdims=True), 1e-300)
    off = np.linalg.norm(ext) * 10 ** rng.uniform(-3, -1.5, k) * rng.choice([-1.0, 1.0], k)
    near = np.einsum("kj,kjc->kc", w, t) + off[:, None] * nrm
    return np.concatenate([uni, near]).astype(np.float32)


def off_surface(tri, pts, pt, closest, frac):  # noqa: F811
    """Mask of the points whose distance to the surface is at least frac x the scene-box diagonal."""
    lo, hi = _lohi(tri)
    d2 = closest(pt, queries(pts))["d2"].astype(np.float64)
    return np.sqrt(d2) >= frac * np.linalg.norm(hi - lo)


def assert_bits(a, b, msg=""):
    np.testing.assert_array_equal(bits(a), bits(b), err_msg=msg)


# ------------------------------------------------------------------------------------------------ tests

@pytest.mark.parametrize("name", SCENE_NAMES)
def test_exact_walk_equals_brute_force(oracle, scenes, tree, winding, name):
    tri = scene_set(scenes)[name]
    for label, pt in trees_of(name, tri, oracle, tree):
        q = queries(point_set(tri, pt, oracle, camera_for(name, scenes)))
        a, ca = winding(pt, q, np.inf)
        b, _ = winding(pt, q, brute=True)
        assert_bits(a, b, "%s %s" % (name, label))
        assert ca["far"] == 0 and ca["exact"] == pt.n * (len(q) - 12)          # every leaf of every finite point, no expansion
        assert not np.isnan(a).any()
        np.testing.assert_array_equal(a[-12:], 0.0)                             # point_set ends with 12 non-finite points


@pytest.mark.parametrize("name", ["dodecahedron", "cornell", "sphere", "soup", "coplanar"])
def test_exact_mode_against_float64(oracle, scenes, tree, closest, winding, name):  # noqa: F811
    tri = scene_set(scenes)[name]
    pt = tree(oracle.Bih(tri))
    pts = sample_points(tri, np.random.default_rng(1))
    keep = off_surface(tri, pts, pt, closest, 1e-3)
    w, _ = winding(pt, queries(pts[keep]), np.inf)
    err = np.abs(w - winding.f64(tri, pts[keep]))
    assert err.max() <= EXACT_TOL, err.max()


@pytest.mark.parametrize("name", ["dodecahedron", "sphere_70k", "sphere_260k", "box_n4", "box_n4_inward", "overlapping_spheres"])
def test_closed_meshes_classify_exactly(oracle, scenes, tree, closest, winding, name):  # noqa: F811
    tri = closed_scenes(scenes)[name]
    rng = np.random.default_rng(3)
    pts = sample_points(tri, rng, k=300)
    want = {"box_n4_inward": {-1, 0}, "overlapping_spheres": {0, 1, 2}}.get(name, {0, 1})
    for label, pt in (("parity", tree(oracle.Bih(tri))), ("q4", tree(tri, 4))):
        keep = off_surface(tri, pts, pt, closest, 1e-4)
        p = pts[keep]
        w64 = winding.f64(tri, p)
        truth = np.round(w64)
        assert np.abs(w64 - truth).max() < 1e-6                                 # float64 is an integer off the surface
        assert set(truth.astype(int)) == want, set(truth.astype(int))
        for beta in (2.0, 3.0, np.inf):
            w, _ = winding(pt, queries(p), beta)
            np.testing.assert_array_equal(np.round(w), truth, err_msg="%s %s beta %s" % (name, label, beta))


@pytest.mark.parametrize("name", ["atrium", "cornell", "soup", "coplanar"])
def test_open_scenes_against_float64(oracle, scenes, tree, closest, winding, name):  # noqa: F811
    tri = scene_set(scenes)[name]
    pts = sample_points(tri, np.random.default_rng(4), k=300)
    w64 = None
    for label, pt in (("parity", tree(oracle.Bih(tri))), ("q4", tree(tri, 4))):
        keep = off_surface(tri, pts, pt, closest, 1e-3)
        w64 = winding.f64(tri, pts[keep]) if w64 is None else w64
        for beta, tol in BETA_TOL.items():
            w, c = winding(pt, queries(pts[keep]), beta)
            err = np.abs(w - w64).max()
            assert err <= tol, (name, label, beta, err)
            assert c["far"] > 0


def subtree_slots(pt, ref):
    """Slots of the subtree under child reference ref, in slot order."""
    out, stack = [], [int(ref)]
    while stack:
        r = stack.pop()
        if r & 0x80000000:
            s = (r & 0x7FFFFFFF) >> 2
            while True:
                out.append(s)
                if pt.tris[s, 10] & 1:
                    break
                s += 1
        else:
            nw = pt.nodes[r >> 2]
            stack += [int(nw[3]), int(nw[2])]
    return np.array(sorted(out))


def moments64(pt, slots, c):
    """float64 N, M, Q (Q as i x (00 01 02 11 12 22)) of the record triangles of `slots` about c"""
    rec = pt.tris[slots].view(np.float32)[:, :9].astype(np.float64)
    v0, e1, e2 = rec[:, 0:3], rec[:, 3:6], rec[:, 6:9]
    h = 0.5 * np.cross(e1, e2)
    s = np.stack([v0 - c, v0 + e1 - c, v0 + e2 - c], 1)
    S = s.sum(1)
    E = (np.einsum("tvj,tvk->tjk", s, s) + np.einsum("tj,tk->tjk", S, S)) / 12.0
    N = h.sum(0)
    M = np.einsum("ti,tj->ij", h, S / 3.0)
    Q = np.einsum("ti,tjk->ijk", h, E)
    jj, kk = [0, 0, 0, 1, 1, 2], [0, 1, 2, 1, 2, 2]
    scale = np.abs(h).sum() * np.abs(s).max() ** np.arange(3)
    return np.concatenate([N, M.ravel(), Q[:, jj, kk].ravel()]), scale


@pytest.mark.parametrize("cap", (None,) + CAPS)
def test_table_against_float64_moments(oracle, scenes, tree, winding, cap):
    tri = np.concatenate([scenes.displaced_sphere(16), scenes.random_soup(300, size=0.1)]).astype(np.float32)
    pt = tree(oracle.Bih(tri)) if cap is None else tree(tri, cap)
    tab = winding.table(pt)
    checked = 0
    for x in np.nonzero(pt.reach)[0]:
        nw = pt.nodes[x]
        boxes = nw[4:16].view(np.float32).reshape(2, 6)
        for side in range(2):
            c = ((boxes[side, 0:3] + boxes[side, 3:6]) * np.float32(0.5)).astype(np.float64)
            want, scale = moments64(pt, subtree_slots(pt, nw[2 + side]), c)
            got = tab[x, side, :30].astype(np.float64)
            tol = 1e-5 * np.concatenate([np.full(3, scale[0]), np.full(9, scale[1]), np.full(18, scale[2])])
            assert np.all(np.abs(got - want) <= tol), (cap, x, side, np.abs(got - want) / tol)
            assert np.all(tab[x, side, 30:] == 0)
            checked += 1
    assert checked == 2 * (pt.nu - 1)


def test_special_points_and_degenerate_triangles_give_no_nan(oracle, scenes, tree, winding):
    sphere = scenes.displaced_sphere(48)
    poles = sphere.reshape(-1, 3)[np.argsort(np.abs(sphere.reshape(-1, 3)[:, 1]))[-8:]]   # the collapsed poles
    for name, tri in (("needles", scene_set(scenes)["needles"]), ("identical", scene_set(scenes)["identical"]),
                      ("sphere", sphere), ("coplanar", scene_set(scenes)["coplanar"])):
        rng = np.random.default_rng(7)
        surf, _ = surface_points(tri, rng, 200)                 # vertices, edge midpoints, inner points
        pts = np.concatenate([surf, poles, tri.reshape(-1, 3)[:50]]).astype(np.float32)
        for label, pt in trees_of(name, tri, oracle, tree):
            for beta in (1.5, 2.0, np.inf):
                w, _ = winding(pt, queries(pts), beta)
                assert not np.isnan(w).any() and np.isfinite(w).all(), (name, label, beta)
            b, _ = winding(pt, queries(pts), brute=True)
            assert not np.isnan(b).any()


def test_nonfinite_points_empty_scene_single_leaf(oracle, scenes, tree, winding):
    tri = scenes.cornell_box()
    pt = tree(oracle.Bih(tri))
    p = np.array([[np.nan, 0, 0], [0, np.inf, 0], [0, 0, -np.inf], [0.1, 0.2, 0.3]], np.float32)
    w, c = winding(pt, queries(p), 2.0)
    np.testing.assert_array_equal(w[:3], 0.0)
    assert w[3] != 0
    _, c3 = winding(pt, queries(p[3:]), 2.0)
    assert c == c3                                               # the non-finite points did no work
    empty = SimpleNamespace(hdr=np.zeros(16, np.uint32), nodes=np.zeros((0, 16), np.uint32), tris=np.zeros((0, 12), np.uint32))
    w, c = winding(empty, queries(p), 2.0)
    np.testing.assert_array_equal(w, 0.0)
    assert c == {"nodes": 0, "far": 0, "exact": 0}
    for one, cap in ((scenes.dodecahedron()[:1], None), (scenes.dodecahedron()[:12], 16)):
        pt1 = tree(oracle.Bih(one)) if cap is None else tree(one, cap)
        assert pt1.nu == 1
        q = queries(np.random.default_rng(2).uniform(-1.5, 1.5, (500, 3)))
        a, ca = winding(pt1, q, 2.0)
        assert_bits(a, winding(pt1, q, brute=True)[0])
        assert ca["far"] == 0 and ca["exact"] == len(one) * 500


def test_python_layer_validates_beta():
    import bihrt
    q = queries(np.zeros((4, 3), np.float32))
    for beta in (1.0, 0.5, -2.0, np.nan, -np.inf):
        with pytest.raises(ValueError):
            bihrt.Renderer.winding_number(object(), q, beta=beta)        # refused before the library is called


@pytest.mark.parametrize("cap", (None, 4))
def test_power_of_two_scaling_is_exact(oracle, scenes, tree, winding, cap):
    """Every operation of the table, the far test and both kinds of terms scales exactly with the coordinates: a mesh and
    points scaled by 2^16 or 2^-16 give the same w bit for bit at every beta."""
    tri = np.concatenate([scenes.dodecahedron(), scenes.displaced_sphere(24) * np.float32(0.6)]).astype(np.float32)
    pts = sample_points(tri, np.random.default_rng(5), k=500)
    base = tree(oracle.Bih(tri)) if cap is None else tree(tri, cap)
    for s in (np.float32(2.0 ** 16), np.float32(2.0 ** -16)):
        pt = tree(oracle.Bih(tri * s)) if cap is None else tree(tri * s, cap)
        np.testing.assert_array_equal(pt.tris[:, 9], base.tris[:, 9])          # the same slot order
        np.testing.assert_array_equal(pt.nodes[:, 2:4], base.nodes[:, 2:4])    # and the same tree
        for beta in (1.5, 2.0, 4.0, np.inf):
            assert_bits(winding(pt, queries(pts * s), beta)[0], winding(base, queries(pts), beta)[0], "%s %s" % (s, beta))
