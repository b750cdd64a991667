"""Quality-mode trees (morton_bits 63, leaf_cap) and every trace entry point on them, held bit for bit to a CPU restatement.

tests/walk_oracle.c restates the quality build from the definition of the tree (63-bit Morton keys, stable order,
radix tree over key + slot position, subtrees of at most leaf_cap triangles as leaves, exact children boxes) and the walk
the kernel takes on it (traverse_box without the reference's strict test, long stack) with three exits: closest hit,
first accepted triangle, first accepting leaf.  The CPU tests tie the walk to brute force and check the restated tree's
structure; the GPU tests compare the exported blob with the restated one and every trace entry point's hits and counters
with the walk, exactly.  The occlusion tests pin bihrt_trace_any's blocker on both tree kinds.
"""
import itertools
import math

import numpy as np
import pytest

from test_gpu_octant_walk import check_frame
from walk_oracle import (FLT_MAX, assert_blob_equals, assorted_intervals, bits, blob_of, rays8,
                         tree)  # noqa: F401  (tree: fixture)

CAPS = (1, 4, 16, 64)


# ------------------------------------------------------------------------------------------------ scenes

def deep_comb(levels=21, dup=4096):
    """A scene whose quality tree is deeper than any parity tree can be, and whose walk needs more than the parity stack.

    A comb along the Morton key: tooth k of axis x (y, z) is a pair of identical triangles whose centre lies 1.5 * 2^k
    cells of the 21-bit grid out along that axis, so its key's highest bit is bit k of that axis, above every key of the
    teeth below it.  The keys form a comb of 3 * `levels` key levels, and each tooth (two triangles, leaf_cap 1) is a node
    of its own.  `dup` identical triangles at the comb's deepest point add log2(dup) position levels below it.  All
    triangles face -x, and a ray along +x near y = z = 0.1 cell crosses every tooth's box and the box of the rest of the
    comb below it, so it stacks one tooth per key level, then one subtree per position level, on its way to its hit."""
    c = 1.0                                   # one cell of the grid: the scene spans about [0, 2^21] on every axis (so that the
    w = 0.25 * c                              # triangles' det clears Moller-Trumbore's absolute 1e-6)

    def facing(x, y0, z0, y1, z1, y2, z2):    # a triangle in the plane x = const, facing -x
        return [x, y0, z0, x, y2, z2, x, y1, z1]

    tri = []
    for k in range(levels):
        big = 3.0 * (1 << k) * c
        tri += [facing(1.5 * (1 << k) * c, -w, -w, 3 * w, -w, -w, 3 * w)] * 2      # x tooth: centre x = 1.5 * 2^k cells
        tri += [facing(2.0 * w, 0.0, -w, big, 0.0, 0.0, w)] * 2                     # y tooth: y spans [0, 3 * 2^k] cells
        tri += [facing(3.0 * w, -w, 0.0, 0.0, big, w, 0.0)] * 2                     # z tooth
    tri += [facing(w, -w, -w, 3 * w, -w, -w, 3 * w)] * dup                           # the comb's deepest point
    top = float(1 << 21)
    tri += [facing(top, top, top, top - c, top, top, top - c)]                       # pins the scene box's hi corner
    return np.array(tri, np.float32)


def deep_comb_rays(n=4096, seed=5):
    """Rays along +x from left of the comb, at y, z of 0.05 .. 0.2 cells, tilted by less than 1e-6 towards +y and +z."""
    rng = np.random.default_rng(seed)
    c = 1.0
    o = np.stack([np.full(n, -4 * c), rng.uniform(0.05, 0.2, n) * c, rng.uniform(0.05, 0.2, n) * c], 1)
    d = np.stack([np.ones(n), rng.uniform(1e-8, 1e-6, n), rng.uniform(1e-8, 1e-6, n)], 1)
    return np.concatenate([o, d], 1).astype(np.float32)


def mirrored(tri, rays, signs):
    """The scene and rays reflected on the axes where signs is -1 (vertex order swapped for an odd number of reflections, so
    that the triangles still face the rays)."""
    s = np.array(signs, np.float32)
    t = (tri.reshape(-1, 3, 3) * s).astype(np.float32)
    if np.prod(signs) < 0:
        t = t[:, [0, 2, 1]]
    r = np.concatenate([rays[:, 0:3] * s, rays[:, 3:6] * s], 1).astype(np.float32)
    return np.ascontiguousarray(t.reshape(-1, 9)), r


def comb_camera(signs):
    """A pinhole camera whose rays are deep_comb_rays' kind (along +x, tilted by 1e-7 .. 1.1e-6 towards +y and +z at
    y = z = 0.125 cells), reflected like `mirrored`."""
    s = np.array(signs, np.float32)
    o = np.array([-4.0, 0.125, 0.125], np.float32)
    llc = np.array([-3.0, 0.125 + 1e-7, 0.125 + 1e-7], np.float32)
    return np.concatenate([o * s, llc * s, np.array([0, 1e-6, 0], np.float32) * s, np.array([0, 0, 1e-6], np.float32) * s])


def quality(renderer, cap):
    renderer.set_option("morton_bits", 63)
    renderer.set_option("leaf_cap", cap)
    return renderer


# ------------------------------------------------------------------------------------------------ CPU: the restatement

def check_structure(qt):
    """Every slot is in exactly one leaf, a leaf holds at most cap slots and ends at the only flagged slot of its range, nu
    counts the leaves, every plane and box is the exact bound of its subtree's vertices, the depth is at most the key levels
    plus the position levels (63 + ceil(log2 n))."""
    n, cap = qt.n, qt.cap
    v = qt.tri9.reshape(n, 3, 3)[qt.tris[:, 9].astype(np.int64)]       # vertices by slot
    np.testing.assert_array_equal(np.sort(qt.tris[:, 9]), np.arange(n))
    np.testing.assert_array_equal(qt.tris[:, 11], np.arange(n))
    slo, shi = v.min(axis=1), v.max(axis=1)
    last = np.flatnonzero(qt.tris[:, 10])
    leaves = []                                                          # (first, last) slot of each leaf reached

    def sub(ref, depth):                                                 # -> first slot, last slot, box lo, box hi, depth
        if ref & 0x80000000:
            a = (ref & 0x7FFFFFFF) >> 2
            b = int(last[np.searchsorted(last, a)])
            leaves.append((a, b))
            return a, b, slo[a:b + 1].min(0), shi[a:b + 1].max(0), depth
        nd = qt.nodes[ref >> 2]
        ax = ref & 3
        la, lb, llo, lhi, ld = sub(int(nd[2]), depth + 1)
        ra, rb, rlo, rhi, rd = sub(int(nd[3]), depth + 1)
        assert lb + 1 == ra
        box = nd[4:16].view(np.float32)
        np.testing.assert_array_equal(box, np.concatenate([llo, lhi, rlo, rhi]))
        assert nd[0:1].view(np.float32)[0] == lhi[ax] and nd[1:2].view(np.float32)[0] == rlo[ax]
        return la, rb, np.minimum(llo, rlo), np.maximum(lhi, rhi), max(ld, rd)

    if n <= cap:
        assert qt.nu == 1 and qt.depth == 0 and list(last) == [n - 1]
        return
    a, b, lo, hi, depth = sub(int(qt.hdr[9]), 0)
    assert (a, b) == (0, n - 1) and depth == qt.depth
    np.testing.assert_array_equal(qt.hdr[2:5].view(np.float32), lo)
    np.testing.assert_array_equal(qt.hdr[5:8].view(np.float32), hi)
    leaves.sort()
    assert len(leaves) == qt.nu == len(last)
    assert [x[1] for x in leaves] == list(last) and leaves[0][0] == 0
    assert all(p[1] + 1 == q[0] for p, q in zip(leaves, leaves[1:]))
    assert max(x[1] - x[0] + 1 for x in leaves) <= cap
    assert qt.depth <= 63 + math.ceil(math.log2(n))


CPU_SCENES = {
    "dodecahedron": lambda S: (S.dodecahedron(), S.pinhole_camera(aspect=1.0), 96, 96),
    "cornell": lambda S: (S.cornell_box(), S.cornell_camera(), 96, 96),
    "sphere187": lambda S: (S.displaced_sphere(187), S.pinhole_camera(), 96, 54),
    "sphere361": lambda S: (S.displaced_sphere(361), S.pinhole_camera(), 64, 36),
    "atrium": lambda S: (S.atrium(0.3), S.atrium_camera(), 96, 54),
    "soup": lambda S: (S.random_soup(50000), S.pinhole_camera(), 96, 54),
}


@pytest.mark.parametrize("name", list(CPU_SCENES))
def test_walk_equals_brute_force_and_tree_is_well_formed(oracle, scenes, tree, name):
    """On the golden scenes at caps 1, 4, 16 and 64: the closest walk's t equals brute force bit for bit and it hits exactly
    where brute force hits; 'first' hits exactly there too with no more work; the any-walk hits exactly where the closest t
    is below tmax; the restated tree is well formed."""
    tri, cam, w, h = CPU_SCENES[name](scenes)
    rays = oracle.camera_rays(cam, w, h, spp=2, jitter=True)
    t0, s0, _ = oracle.Bih(tri).trace(rays, "brute")
    assert 0.05 < (s0 >= 0).mean()
    for cap in CAPS:
        qt = tree(tri, cap)
        check_structure(qt)
        res = qt.walk(rays)
        t, s, p, c = res["t"], res["slot"], res["prim"], res["counters"]
        np.testing.assert_array_equal(t, t0, err_msg="cap %d" % cap)
        np.testing.assert_array_equal(s >= 0, s0 >= 0)
        np.testing.assert_array_equal(p[s >= 0], qt.tris[s[s >= 0], 9].astype(np.int32))
        f = qt.walk(rays, "first")
        tf, sf, cf = f["t"], f["slot"], f["counters"]
        np.testing.assert_array_equal(sf >= 0, s >= 0)
        assert np.all(tf[sf >= 0] >= t[sf >= 0])
        assert cf["nodes"] <= c["nodes"] and cf["tris"] <= c["tris"] and cf["max_stack"] <= c["max_stack"]
        for tmax in (np.float32(np.median(t0[s0 >= 0])), np.float32(np.inf)):
            a = qt.walk(rays, "any", tmax=tmax, ht_max=np.inf)
            ta, sa, ca = a["t"], a["slot"], a["counters"]
            np.testing.assert_array_equal(sa >= 0, (s >= 0) & (t < tmax))
            hit = sa >= 0
            assert np.all(ta[hit] < tmax) and np.all(ta[hit] >= t[hit]) and ca["tris"] <= c["tris"]


@pytest.mark.parametrize("cap", [1, 2, 4, 16, 64])
def test_restated_tree_is_well_formed_on_edge_cases(scenes, tree, cap):
    """Sizes around the cap, tied keys (position levels), a flat axis and -0 coordinates."""
    for tri in build_cases(scenes, cap, small=True):
        check_structure(tree(tri, cap))


def test_deep_comb_needs_the_long_stack(oracle, tree):
    """The deep scene's tree is deeper than a parity tree (31 levels) and its rays stack more than the parity stack holds
    (32 items), in every reflection of the scene; they all hit, at brute force's t."""
    for signs in itertools.product((1, -1), repeat=3):
        tri, rays = mirrored(deep_comb(), deep_comb_rays(1024), signs)
        qt = tree(tri, 1)
        check_structure(qt)
        assert qt.depth > 64
        res = qt.walk(rays)
        assert res["counters"]["max_stack"] > 32 and (res["slot"] >= 0).all(), signs
        np.testing.assert_array_equal(res["t"], oracle.Bih(tri).trace(rays, "brute")[0])
        cf = qt.walk(oracle.camera_rays(comb_camera(signs), 16, 8, spp=4, jitter=True), "first")["counters"]
        assert cf["max_stack"] > 32, signs


def build_cases(scenes, cap, small=False):
    """Scenes for the build comparison: n = 1 .. cap + 1, 2049 and 10^5 triangles of soup, heavy duplicates (tied keys: the
    split falls in the position bits), a scene flat on one axis and -0.0 coordinates."""
    base = scenes.displaced_sphere(40)
    for n in range(1, cap + 2):
        yield np.ascontiguousarray(base[:: max(1, len(base) // n)][:n])
    yield scenes.random_soup(2049)
    if not small:
        yield scenes.random_soup(100000)
    yield np.ascontiguousarray(np.repeat(base[:37], 53, axis=0))
    flat = base.copy().reshape(-1, 3, 3)
    flat[:, :, 1] = np.float32(0.25)
    yield np.ascontiguousarray(flat.reshape(-1, 9))
    negz = base.copy()
    negz[np.abs(negz) < np.float32(0.3)] = np.float32(-0.0)
    negz[::7, 0::3] = np.float32(0.0)
    yield negz


# ------------------------------------------------------------------------------------------------ GPU: the build

@pytest.mark.gpu
@pytest.mark.parametrize("cap", [1, 2, 4, 16, 64])
def test_quality_build_equals_restatement(renderer, scenes, tree, cap):
    for i, tri in enumerate(build_cases(scenes, cap)):
        quality(renderer, cap).load_models(tri).build()
        assert_blob_equals(blob_of(renderer), tree(tri, cap), "case %d (n %d)" % (i, len(tri)))


@pytest.mark.gpu
def test_quality_build_of_one_million_triangles_and_after_a_parity_build(renderer, scenes, tree):
    """The 1 M-triangle sphere; then a smaller scene built in parity mode and in quality mode on the same context, so the
    quality blob's node slots hold the parity tree's stale records."""
    tri = scenes.displaced_sphere(scenes.SPHERE_NSEG["1m"])
    quality(renderer, 4).load_models(tri).build()
    assert_blob_equals(blob_of(renderer), tree(tri, 4), "1 M")
    tri = scenes.displaced_sphere(187)
    renderer.set_option("morton_bits", 30)
    renderer.load_models(tri).build()
    quality(renderer, 16).build()
    qt = tree(tri, 16)
    assert_blob_equals(blob_of(renderer), qt, "after parity")
    assert not qt.reach.all()


# ------------------------------------------------------------------------------------------------ GPU: ray lists

LIST_CASES = {
    "cornell": lambda S: (S.cornell_box(), S.cornell_camera(), 128, 128),
    "sphere187": lambda S: (S.displaced_sphere(187), S.pinhole_camera(), 160, 90),
    "atrium": lambda S: (S.atrium(0.2), S.atrium_camera(), 160, 90),
    "soup": lambda S: (S.random_soup(20000), S.pinhole_camera(), 160, 90),
}


def secondary_like(rays, t, seed):
    """Rays from the hit points (or far along the missing rays) in random directions: incoherent lists."""
    rng = np.random.default_rng(seed)
    tt = np.where(t < FLT_MAX, t, np.float32(2.0))[:, None] * np.float32(0.999)
    o = rays[:, :3] + rays[:, 3:] * tt
    d = rng.normal(size=o.shape)
    return np.concatenate([o, d], 1).astype(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("cap", [1, 4, 16])
@pytest.mark.parametrize("name", list(LIST_CASES))
def test_counted_trace_equals_walk(renderer, scenes, oracle, tree, name, cap):
    """trace(counted=True) on a quality tree: t, slot and prim equal the closest walk's bit for bit (no tie allowance),
    nodes, triangle tests and the deepest stack exactly; the uncounted kernel gives the same outputs."""
    tri, cam, w, h = LIST_CASES[name](scenes)
    qt = tree(tri, cap)
    quality(renderer, cap).load_models(tri).build()
    prim_rays = oracle.camera_rays(cam, w, h)
    for rays in (prim_rays, secondary_like(prim_rays, qt.walk(prim_rays)["t"], 3)):
        res = qt.walk(rays)
        t0, s0, p0, c0 = res["t"], res["slot"], res["prim"], res["counters"]
        t, s, p, cnt = renderer.trace(rays, counted=True)
        np.testing.assert_array_equal(bits(t), bits(t0))
        np.testing.assert_array_equal(s, s0)
        np.testing.assert_array_equal(p, p0)
        assert (cnt["nodes"], cnt["tris"], cnt["max_stack"]) == (c0["nodes"], c0["tris"], c0["max_stack"])
        t2, s2, p2 = renderer.trace(rays)
        np.testing.assert_array_equal(bits(t2), bits(t0))
        np.testing.assert_array_equal(s2, s0)
        np.testing.assert_array_equal(p2, p0)


# ------------------------------------------------------------------------------------------------ GPU: framebuffers

@pytest.mark.gpu
@pytest.mark.parametrize("signs", list(itertools.product((1, -1), repeat=3)))
def test_quality_diagonal_views(renderer, scenes, oracle, tree, signs):
    """test_gpu_octant_walk's diagonal views on a quality tree: every octant copy of the node phase with Q set."""
    tri = scenes.displaced_sphere(187)
    qt = tree(tri, 4)
    quality(renderer, 4).load_models(tri).build()
    s = np.array(signs, np.float64)
    cam = scenes.look_at_camera(2.2 * s + np.array([0.05, 0.03, 0.0]), (0.0, 0.0, 0.0), 0.3, 1.5)
    for spp, jitter in ((1, False), (4, True), (16, True)):
        rays, s0 = check_frame(renderer, oracle, qt, cam, 120, 80, spp, jitter)
        assert (np.sign(rays[:, 3:]) == -s).all(axis=1).mean() > 0.95
        assert 0.2 < (s0 >= 0).mean() < 0.9


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(97, 65), (160, 90), (75, 41)])
def test_quality_sign_changes_inside_warps(renderer, scenes, oracle, tree, w, h):
    tri = scenes.displaced_sphere(187)
    qt = tree(tri, 1)
    quality(renderer, 1).load_models(tri).build()
    cam = scenes.pinhole_camera(aspect=w / h)
    for spp in (1, 4, 16):
        for jitter in (False, True):
            check_frame(renderer, oracle, qt, cam, w, h, spp, jitter, groups=(-1, 1, 2))


@pytest.mark.gpu
def test_quality_zero_direction_component_in_a_uniform_warp(renderer, scenes, oracle, tree):
    tri = scenes.displaced_sphere(187)
    qt = tree(tri, 16)
    quality(renderer, 16).load_models(tri).build()
    cam = scenes.pinhole_camera(origin=(0.0, 0.2, -3.0), half=0.5, aspect=1.0)
    for spp in (1, 16):
        rays, s0 = check_frame(renderer, oracle, qt, cam, 97, 64, spp, False, groups=(-1, 1))
        zero = rays[:, 3] == 0
        assert zero.sum() == 64 * spp and (s0[zero] >= 0).any()


@pytest.mark.gpu
@pytest.mark.parametrize("view", ["atrium_camera", "diagonal_down", "diagonal_up_back"])
def test_quality_camera_inside_the_atrium(renderer, scenes, oracle, tree, view):
    tri = scenes.atrium(0.2)
    qt = tree(tri, 4)
    quality(renderer, 4).load_models(tri).build()
    cam = {"atrium_camera": lambda: scenes.atrium_camera(160 / 90),
           "diagonal_down": lambda: scenes.look_at_camera((-1.2, 0.3, 0.4), (0.0, -0.5, -0.4), 0.6, 160 / 90),
           "diagonal_up_back": lambda: scenes.look_at_camera((1.0, -0.4, 0.3), (-0.2, 0.4, 1.2), 0.6, 160 / 90)}[view]()
    for spp, jitter in ((1, False), (4, True), (16, False)):
        _, s0 = check_frame(renderer, oracle, qt, cam, 160, 90, spp, jitter, groups=(-1, 1))
        assert (s0 >= 0).mean() > 0.5


@pytest.mark.gpu
@pytest.mark.parametrize("cap", [1, 16])
def test_quality_render_hits_and_sharded_renders(renderer, scenes, oracle, tree, cap):
    """render_hits (MODE 2) equals the closest walk bit for bit; render_samples summed over rank splits and
    render_interleaved summed over its indices, resolved, equal render."""
    import torch
    from bihrt import multi
    tri, cam, w, h = (scenes.atrium(0.2), scenes.atrium_camera(160 / 90), 160, 90)
    qt = tree(tri, cap)
    quality(renderer, cap).load_models(tri).build()
    for spp, jitter in ((1, False), (4, True)):
        rays = oracle.camera_rays(cam, w, h, spp=spp, jitter=jitter, seed=1984)
        res = qt.walk(rays)
        t0, s0, p0 = res["t"], res["slot"], res["prim"]
        t, s, p = renderer.render_hits(cam, w, h, spp=spp, jitter=jitter)
        np.testing.assert_array_equal(bits(t), bits(t0))
        np.testing.assert_array_equal(s, s0)
        np.testing.assert_array_equal(p, p0)
    spp = 4
    exp = renderer.render(cam, w, h, spp=spp, jitter=True).framebuffer().copy()
    rays = oracle.camera_rays(cam, w, h, spp=spp, jitter=True, seed=1984)
    np.testing.assert_array_equal(exp.ravel(), oracle.pack_framebuffer(qt.walk(rays)["slot"], w, h, spp))
    for parts in ((2, "samples"), (4, "interleaved")):
        counts = torch.zeros((h, w), dtype=torch.int32, device="cuda")
        for k in range(parts[0]):
            if parts[1] == "samples":
                s_a, s_b = multi.sample_range(spp, k, parts[0])
                renderer.render_samples(cam, w, h, spp, s_a, s_b, jitter=True)
            else:
                renderer.render_interleaved(cam, w, h, spp, k, parts[0], jitter=True)
            renderer.sync()
            counts += multi.framebuffer_tensor(renderer)
            torch.cuda.synchronize()
        multi.framebuffer_tensor(renderer).copy_(counts)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(renderer.framebuffer_resolve(spp).framebuffer(), exp, err_msg=parts[1])


# ------------------------------------------------------------------------------------------------ GPU: occlusion

OCCLUSION_TMAX = (0.25, 1.0, 3.0, 1e30, np.inf)


def occlusion_rays(oracle, scenes):
    tri, cam, w, h = LIST_CASES["atrium"](scenes)
    prim = oracle.camera_rays(cam, w, h)
    t0, _, _ = oracle.Bih(tri).trace(prim, "box")
    return tri, np.concatenate([prim, secondary_like(prim, t0, 9)])


def check_trace_any(renderer, rays, want_slot):
    """trace_any's blocker equals want_slot(tmax) exactly, for host and device buffers and with and without the ray sort;
    for finite tmax it equals intersect(any_hit=True) on (0, tmax)."""
    import torch
    from bihrt import interval_rays
    dev = torch.from_numpy(rays).cuda()
    try:
        for sort in (0, 1):
            renderer.set_option("trace_sort_rays", sort)
            for tmax in OCCLUSION_TMAX:
                want = want_slot(np.float32(tmax))
                np.testing.assert_array_equal(renderer.trace_any(rays, tmax=tmax), want, err_msg="host tmax %g sort %d" % (tmax, sort))
                got = renderer.trace_any(dev, tmax=tmax)
                torch.cuda.synchronize()
                np.testing.assert_array_equal(got.cpu().numpy(), want, err_msg="device tmax %g sort %d" % (tmax, sort))
                if np.isfinite(tmax):
                    r = renderer.intersect(interval_rays(rays, 0.0, tmax), any_hit=True, outputs=("slot",))
                    np.testing.assert_array_equal(r["slot"], want)
                assert 0 < (want >= 0).mean() < 1 or tmax >= 3
    finally:
        renderer.set_option("trace_sort_rays", 0)
    import bihrt
    for bad in (0.0, -1.0, float("nan")):
        with pytest.raises(bihrt.BihrtError) as e:
            renderer.trace_any(rays[:8], tmax=bad)
        assert e.value.code == -1


@pytest.mark.gpu
def test_trace_any_blocker_on_parity_tree(renderer, scenes, oracle, tree):
    """On the reference's tree the blocker is the any-walk's slot over (0, tmax), with h.t starting at min(tmax, FLT_MAX)."""
    tri, rays = occlusion_rays(oracle, scenes)
    pt = tree(oracle.Bih(tri))
    renderer.load_models(tri).build()
    check_trace_any(renderer, rays, lambda tmax: pt.walk(rays, "any", tmax=tmax)["slot"])


@pytest.mark.gpu
@pytest.mark.parametrize("cap", [1, 4])
def test_trace_any_blocker_on_quality_tree(renderer, scenes, oracle, tree, cap):
    """On a quality tree the blocker is the any-walk's slot, with h.t starting at tmax as passed."""
    tri, rays = occlusion_rays(oracle, scenes)
    qt = tree(tri, cap)
    quality(renderer, cap).load_models(tri).build()
    check_trace_any(renderer, rays, lambda tmax: qt.walk(rays, "any", tmax=tmax, ht_max=np.inf)["slot"])


# ------------------------------------------------------------------------------------------------ GPU: ray queries

@pytest.mark.gpu
@pytest.mark.parametrize("cap", [1, 4, 16])
@pytest.mark.parametrize("name", ["cornell", "sphere187", "atrium", "soup"])
def test_quality_intersect_equals_walk(renderer, scenes, oracle, tree, name, cap):
    """intersect on a quality tree, closest and ANY, one- and two-sided, on random intervals: slot and t equal the walk's."""
    tri, cam, w, h = LIST_CASES[name](scenes)
    qt = tree(tri, cap)
    quality(renderer, cap).load_models(tri).build()
    rays = oracle.camera_rays(cam, w, h)
    tmin, tmax = assorted_intervals(qt.walk(rays)["t"], seed=31)
    r8 = rays8(rays, tmin, tmax)
    for any_hit, two_sided in itertools.product((False, True), repeat=2):
        res = qt.walk(r8, "any" if any_hit else "closest", two_sided=two_sided)
        t0, s0, p0 = res["t"], res["slot"], res["prim"]
        got = renderer.intersect(r8, any_hit=any_hit, two_sided=two_sided, outputs=("t", "slot", "prim"))
        what = "any %s two-sided %s" % (any_hit, two_sided)
        np.testing.assert_array_equal(bits(got["t"]), bits(t0), err_msg=what)
        np.testing.assert_array_equal(got["slot"], s0, err_msg=what)
        np.testing.assert_array_equal(got["prim"], p0, err_msg=what)
        assert (s0 >= 0).any(), what


# ------------------------------------------------------------------------------------------------ GPU: a deep tree

@pytest.mark.gpu
def test_deep_tree_counters_and_hits(renderer, oracle, tree):
    """A tree deeper than any parity tree, walked with more than the parity stack: counters and hits of trace (MODE 0),
    of the framebuffer kernel in every octant copy (MODE 1) and hits of intersect (MODE 3) equal the restatement."""
    from bihrt import interval_rays
    for signs in itertools.product((1, -1), repeat=3):
        tri, rays = mirrored(deep_comb(), deep_comb_rays(), signs)
        qt = tree(tri, 1)
        quality(renderer, 1).load_models(tri).build()
        assert_blob_equals(blob_of(renderer), qt, str(signs))
        res = qt.walk(rays)
        t0, s0, p0, c0 = res["t"], res["slot"], res["prim"], res["counters"]
        assert c0["max_stack"] > 32
        t, s, p, cnt = renderer.trace(rays, counted=True)
        np.testing.assert_array_equal(bits(t), bits(t0))
        np.testing.assert_array_equal(s, s0)
        np.testing.assert_array_equal(p, p0)
        assert (cnt["nodes"], cnt["tris"], cnt["max_stack"]) == (c0["nodes"], c0["tris"], c0["max_stack"]), signs
        for any_hit in (False, True):
            r8 = interval_rays(rays, 0.0, np.inf)
            a = qt.walk(r8, "any" if any_hit else "closest")
            ta, sa = a["t"], a["slot"]
            got = renderer.intersect(r8, any_hit=any_hit, outputs=("t", "slot"))
            np.testing.assert_array_equal(bits(got["t"]), bits(ta))
            np.testing.assert_array_equal(got["slot"], sa)
        cam = comb_camera(signs)
        for spp in (4, 16):
            crays, _ = check_frame(renderer, oracle, qt, cam, 24, 16, spp, True, groups=(-1, 1))
            assert qt.walk(crays, "first")["counters"]["max_stack"] > 32
            assert (np.sign(crays[:, 3:]) == np.array(signs)).all()
