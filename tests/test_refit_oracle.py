"""bihrt_refit restated on the CPU, and what its trees give the ray, closest-point and winding walks.

A refit (csrc/build.cu, bihrt_refit_launch) keeps the Morton order, the leaves and the topology of the last full build and
recomputes what depends on vertex positions: the scene box, the triangle records, the children boxes and the clip planes.
refit_bih restates it from the oracle's own pieces: the build's arrays, `orc_prep` of the moved triangles for the triangle
boxes and the scene box (seeded with the first vertex, as the build's), and `orc_clip_planes` over the build's topology.
The result has an oracle.Bih's fields, so the reference view comparison, walk_oracle's blob restatement and walks, and the
closest-point and winding walks all take it as they take a full build; tests/test_gpu_refit.py pins the kernel to it.

The deformations cross the tree: a phase change of the sphere, a random permutation of the triangles' positions, a scale
and translation that moves the scene outside its old box, a mirror (front faces become back faces), clamps to a floor,
flattening onto a plane of each axis, a collapse to one point, and a small jitter of a scene made of axis-aligned walls.
"""
import copy
import ctypes as C

import numpy as np
import pytest

from closest_oracle import closest  # noqa: F401  (fixture)
from test_closest_oracle import assert_closest_equal, queries
from test_winding_oracle import assert_bits, sample_points
from walk_oracle import FLT_MAX, tree  # noqa: F401  (fixture)
from winding_oracle import winding  # noqa: F401  (fixture)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def refit_bih(ob, moved):
    """The tree bihrt_refit makes from `ob` (the oracle.Bih of the last full build) after the vertices became `moved`
    ((n, 9) float32): the build's order, leaves and topology (its Morton codes included, now stale), tri9 = moved, the
    triangle boxes and scene box of `moved`, and the clip planes recomputed over the build's topology."""
    from oracle import oracle as O
    lib = O.lib()
    moved = np.ascontiguousarray(moved, np.float32).reshape(-1, 9)
    assert len(moved) == ob.n
    n, nu, m = ob.n, ob.nu, max(ob.n, 1)
    r = copy.copy(ob)
    r.tri9 = moved
    r.lo, r.hi, r.cnorm = (np.zeros((m, 3), np.float32) for _ in range(3))
    r.scene_lo, r.scene_hi = np.zeros(3, np.float32), np.zeros(3, np.float32)
    centre = np.zeros((m, 3), np.float32)
    lib.orc_prep(_p(moved), C.c_int64(n), _p(r.lo), _p(r.hi), _p(centre), _p(r.cnorm), _p(r.scene_lo), _p(r.scene_hi))
    clip = np.empty((max(nu - 1, 1), 2), np.float32)
    clip[:] = (-FLT_MAX, FLT_MAX)
    topo = [np.ascontiguousarray(x) for x in (ob.tris_idx, ob.leaf_parents, ob.cnt, ob.first, ob.axis, ob.children, ob.parent)]
    lib.orc_clip_planes(C.c_int64(nu), _p(r.lo), _p(r.hi), *[_p(x) for x in topo], _p(clip))
    r.clip = clip[:max(nu - 1, 0)]
    return r


# ------------------------------------------------------------------------------------------------ deformations

FLOORS = (-0.3, 0.0, 0.5)
CROSSING = ("phase0.15", "phase0.7", "shuffle", "scale_translate", "mirror_x")
FLATTENING = tuple("floor%g" % c for c in FLOORS) + ("flat_x", "flat_y", "flat_z", "point")
DEFORMATIONS = CROSSING + FLATTENING


def deform(tri, how, seed=0, phased=None):
    """`tri` moved by `how`: one of DEFORMATIONS, or "jitter" (every vertex by up to 1e-3 on every axis).  The phase
    changes take the moved mesh from `phased(phase)` (a displaced sphere of tri's size); without it they move every vertex
    along a smooth field instead."""
    rng = np.random.default_rng(seed)
    v = np.array(tri, np.float32).reshape(-1, 3, 3)
    if how.startswith("phase"):
        ph = float(how[5:])
        if phased is not None:
            return np.ascontiguousarray(phased(ph), np.float32).reshape(-1, 9)
        v = v + np.float32(0.1) * np.sin(np.float32(6.0) * v[..., [1, 2, 0]] + np.float32(2 * np.pi * ph)).astype(np.float32)
    elif how == "shuffle":
        v = v[rng.permutation(len(v))]
    elif how == "scale_translate":
        v = v * np.float32(300.0) + np.float32(1000.0)
    elif how == "mirror_x":
        v[..., 0] = -v[..., 0]
    elif how.startswith("floor"):
        v[..., 1] = np.maximum(v[..., 1], np.float32(float(how[5:])))
    elif how.startswith("flat_"):
        v[..., "xyz".index(how[5])] = np.float32(0.25)
    elif how == "point":
        v[:] = np.array([0.1, 0.2, 0.3], np.float32)
    elif how == "jitter":
        v = v + rng.uniform(-1e-3, 1e-3, v.shape).astype(np.float32)
    else:
        raise ValueError(how)
    return np.ascontiguousarray(v.astype(np.float32).reshape(-1, 9))


def random_rays(tri, n=20000, seed=1):
    """Rays from a sphere of twice the scene box's diagonal around its centre, aimed at points of the box enlarged by 10 %
    (plus a few along the axes): every part of the scene, from every side."""
    rng = np.random.default_rng(seed)
    v = np.asarray(tri, np.float64).reshape(-1, 3)
    lo, hi = v.min(0), v.max(0)
    c, ext = (lo + hi) / 2, np.maximum(hi - lo, 1e-3 * max(np.abs(hi - lo).max(), 1e-3))
    dirs = rng.normal(size=(n, 3))
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    o = c + dirs * np.linalg.norm(ext) * 2
    target = rng.uniform(c - 0.55 * ext, c + 0.55 * ext, (n, 3))
    d = target - o
    along = np.flatnonzero(rng.random(n) < 0.05)                  # along one axis, towards the target
    axis = rng.integers(0, 3, len(along))
    step = d[along, axis]
    d[along] = 0.0
    d[along, axis] = np.where(step < 0, -1.0, 1.0)
    return np.concatenate([o, d], 1).astype(np.float32)


def sphere(scenes, phase=0.0):
    return scenes.displaced_sphere(96, phase=phase)


def moved_sphere(scenes, how):
    return deform(sphere(scenes), how, phased=lambda ph: sphere(scenes, ph))


# ------------------------------------------------------------------------------------------------ tests

def assert_bih_equal(r, ob, what=""):
    from conftest import assert_view_equals_oracle
    view = {"n": r.n, "nu": r.nu, "morton_codes": r.codes, "tris_indexes": r.tris_idx, "unique_morton_codes": r.umc,
            "duplicates_cnts": r.cnt, "first_idxs": r.first, "children": r.children, "is_leaf": r.is_leaf, "axis": r.axis,
            "parent": r.parent, "leaf_parents": r.leaf_parents, "clip_planes": r.clip, "scene_lo": r.scene_lo,
            "scene_hi": r.scene_hi}
    try:
        assert_view_equals_oracle(view, ob)
    except AssertionError as e:
        raise AssertionError("%s: %s" % (what, e))


def small_scenes(scenes):
    one = np.array([[0, 0, 0, 1, 0, 0, 0, 1, 0]], np.float32)
    return {"one": one, "two": scenes.random_soup(2, size=0.1, seed=2), "three": scenes.random_soup(3, size=0.1, seed=3),
            "seven_identical": np.tile(one, (7, 1)), "sphere": sphere(scenes), "cornell": scenes.cornell_box(),
            "atrium": scenes.atrium(0.2), "soup": scenes.random_soup(4097, size=0.05, seed=5)}


def test_refit_of_unmoved_vertices_is_the_build(oracle, scenes):
    """On scenes of 1, 2, 3 and 7 identical triangles and larger ones: the restated refit of the build's own vertices gives
    back the build, clip planes and scene box included."""
    for name, tri in small_scenes(scenes).items():
        ob = oracle.Bih(tri)
        assert_bih_equal(refit_bih(ob, tri), ob, name)


def test_scene_box_and_planes_follow_the_moved_vertices(oracle, scenes):
    """The scene box is the moved vertices' box; every clip plane is the extent of the side of its node it bounds: clip0 is
    the largest coordinate on the node's axis over the left subtree's triangles, clip1 the smallest over the right one's."""
    ob = oracle.Bih(sphere(scenes))
    for how in DEFORMATIONS:
        b = moved_sphere(scenes, how)
        r = refit_bih(ob, b)
        v = b.reshape(-1, 3)
        np.testing.assert_array_equal(r.scene_lo, v.min(0), err_msg=how)
        np.testing.assert_array_equal(r.scene_hi, v.max(0), err_msg=how)
        tv = b.reshape(-1, 3, 3)
        slot_lo, slot_hi = tv.min(1)[r.tris_idx], tv.max(1)[r.tris_idx]          # per slot
        leaf_end = np.append(r.first[1:], r.n)

        def leaves(node, side):                                                   # leaf range [a, b] under a child
            c = r.children[node, side]
            if r.is_leaf[node, side]:
                return c, c
            return leaves(c, 0)[0], leaves(c, 1)[1]
        for i in range(r.nu - 1):
            ax = r.axis[i]
            la, lb = leaves(i, 0)
            ra, rb = leaves(i, 1)
            assert r.clip[i, 0] == slot_hi[r.first[la]:leaf_end[lb], ax].max(), (how, i)
            assert r.clip[i, 1] == slot_lo[r.first[ra]:leaf_end[rb], ax].min(), (how, i)


def test_chain_of_refits_returns_to_the_build(oracle, scenes):
    """A refit to b, then to c, then back to a equals the build of a: the restatement depends on the build's topology and
    the current vertices only."""
    a = sphere(scenes)
    ob = oracle.Bih(a)
    r = ob
    for how in ("phase0.7", "scale_translate", "floor0"):
        r = refit_bih(r, moved_sphere(scenes, how))
        assert_bih_equal(r, refit_bih(ob, moved_sphere(scenes, how)), how)
    assert_bih_equal(refit_bih(r, a), ob, "back to a")


def walks(oracle, tree, r, rays):  # noqa: F811
    """The reference walk ("ref"), the shipped walk ("box"), the blob walk (Tree.walk) and brute force on refit tree r."""
    out = {m: r.trace(rays, m, want_counters=True) for m in ("ref", "box")}
    out["brute"] = r.trace(rays, "brute")
    out["tree"] = tree(r).walk(rays)
    return out


def assert_blob_walk_is_box(w, what):
    t, s, p, c = w["box"]
    np.testing.assert_array_equal(w["tree"]["t"], t, err_msg=what)
    np.testing.assert_array_equal(w["tree"]["slot"], s, err_msg=what)
    np.testing.assert_array_equal(w["tree"]["prim"], p, err_msg=what)
    assert w["tree"]["counters"] == c, what


@pytest.mark.parametrize("how", CROSSING)
def test_walks_equal_brute_force_on_deformations_that_cross_the_tree(oracle, scenes, tree, how):  # noqa: F811
    """The sphere refit after motions that make its children overlap, leave its old box or flip its faces: the reference
    walk, the shipped walk and the blob walk equal brute force over the moved triangles, by primitive and t."""
    r = refit_bih(oracle.Bih(sphere(scenes)), moved_sphere(scenes, how))
    rays = random_rays(r.tri9)
    w = walks(oracle, tree, r, rays)
    assert_blob_walk_is_box(w, how)
    tb, _, pb = w["brute"]
    for m in ("ref", "box"):
        np.testing.assert_array_equal(w[m][2], pb, err_msg="%s %s" % (how, m))
        np.testing.assert_array_equal(w[m][0], tb, err_msg="%s %s" % (how, m))
    assert (pb >= 0).mean() > 0.05


@pytest.mark.parametrize("how", FLATTENING + ("jitter",))
def test_flattening_deformations_lose_hits_but_report_only_true_ones(oracle, scenes, tree, how):  # noqa: F811
    """Deformations that flatten geometry onto axis-aligned planes the old topology splits across, and the atrium (whose
    walls are axis-aligned planes already) with every vertex jittered by up to 1e-3.  A node whose two sides now meet in
    one plane gets clip0 = clip1, the far side's ray interval shrinks to a single point, and the reference's strict plane
    test, which the parity walk keeps, drops it.  A ray then misses, or walks on to a farther triangle behind the one it
    lost.  So: the walks hit only where brute force hits, every hit they report is a true Moller-Trumbore hit of that
    primitive at that t, and no t is nearer than brute force's.  A full build of the moved mesh finds brute force's t on
    every ray (it never splits triangles that coincide on an axis along that axis).

    Measured on the sphere with the 20 000 random_rays of this file (brute-force hits -> the walk's hits, of which farther
    than brute force's): floor -0.3: 13209 -> 12606 (0), floor 0: 12589 -> 10267 (51), floor 0.5: 11099 -> 8305 (276),
    flat x: 12076 -> 324 (68), flat y: 12054 -> 5165 (37), flat z: 11997 -> 8292 (88), one point: 0 -> 0; the jittered
    atrium loses nothing (17869).  These losses are recorded, not asserted: a walk or refit that keeps every hit passes."""
    from walk_oracle import bits, mt
    if how == "jitter":
        a = scenes.atrium(0.2)
        b = deform(a, "jitter", seed=4)
    else:
        a, b = sphere(scenes), moved_sphere(scenes, how)
    r = refit_bih(oracle.Bih(a), b)
    rays = random_rays(b)
    w = walks(oracle, tree, r, rays)
    assert_blob_walk_is_box(w, how)
    tb, sb, pb = w["brute"]
    for m in ("ref", "box"):
        t, s, p = w[m][:3]
        what = "%s %s" % (how, m)
        hit = s >= 0
        assert not (hit & (sb < 0)).any(), what
        assert (t[hit] >= tb[hit]).all(), what
        ok, _, tm, _, _ = mt(b, p[hit], rays[hit])
        assert ok.all(), what
        np.testing.assert_array_equal(bits(tm), bits(t[hit]), err_msg=what)
        np.testing.assert_array_equal(t[~hit], FLT_MAX, err_msg=what)
    np.testing.assert_array_equal(oracle.Bih(b).trace(rays, "ref")[0], tb, err_msg=how)     # (ties on the floor: t, not prim)


@pytest.mark.parametrize("how", DEFORMATIONS)
def test_closest_point_and_exact_winding_equal_brute_force(oracle, scenes, tree, closest, winding, how):  # noqa: F811
    """Closest-point and winding queries prune with the children boxes, not with the strict plane test: on every refit tree,
    flattened ones included, the closest-point walk and the exact winding walk (beta = inf) equal brute force bit for bit."""
    b = moved_sphere(scenes, how)
    rt = tree(refit_bih(oracle.Bih(sphere(scenes)), b))
    rng = np.random.default_rng(7)
    q = queries(sample_points(b, rng, 1500))
    got = closest(rt, q)
    assert_closest_equal(got, closest(rt, q, brute=True), how)
    assert (got["slot"] >= 0).all()
    assert_bits(winding(rt, q, np.inf)[0], winding(rt, q, brute=True)[0], how)
