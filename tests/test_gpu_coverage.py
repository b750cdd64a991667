"""Framebuffer renders are coverage queries: a sample ends at the first triangle it accepts.

A pixel's colour (and the hit counts of the sharded renders) depends only on WHETHER each sample hits, so the framebuffer
kernel (csrc/trace.cu, MODE 1, COVER) stops a sample's walk at its first accepted triangle instead of
searching on for the closest one.  tests/walk_oracle.c restates that walk on the CPU (exit "first" of its walk on the
parity tree: the oracle's "box" traversal with that one exit).  The CPU tests check that "first" hits exactly where "ref"
and "box" hit and never does more work than "box"; the GPU tests pin render_counted's counters to "first" exactly, and
every framebuffer path to the image of the closest-hit oracle.
"""
import numpy as np
import pytest

from test_gpu_golden_scenes import SCENES as GOLDEN
from walk_oracle import degenerate_rays, tree  # noqa: F401  (tree: fixture)


def assert_first_covers_like_ref(tree, ob, rays):
    """'first' hits exactly where 'ref' and 'box' hit, with no more nodes or triangle tests than 'box'; returns the counters."""
    t0, s0, _ = ob.trace(rays, "ref")
    t3, s3, _, c3 = ob.trace(rays, "box", want_counters=True)
    f = tree(ob).walk(rays, "first")
    tf, sf, pf, cf = f["t"], f["slot"], f["prim"], f["counters"]
    np.testing.assert_array_equal(sf >= 0, s0 >= 0)
    np.testing.assert_array_equal(sf >= 0, s3 >= 0)
    hit = sf >= 0
    assert np.all(tf[hit] > 0) and np.all(tf[~hit] == np.finfo(np.float32).max) and np.all(pf[~hit] == -1)
    assert np.all(tf[hit] >= t3[hit])                  # the first accepted triangle is never closer than the closest one
    assert cf["nodes"] <= c3["nodes"] and cf["tris"] <= c3["tris"] and cf["max_stack"] <= c3["max_stack"]
    return s0, cf, c3


# ------------------------------------------------------------------------------------------------ CPU: the restatement

@pytest.mark.parametrize("name", list(GOLDEN))
def test_first_hit_equals_reference_on_golden_scenes(oracle, scenes, tree, name):
    tri, cam, w, h = GOLDEN[name](scenes)
    ob = oracle.Bih(tri)
    for spp, jitter in ((1, False), (2, True)):
        rays = oracle.camera_rays(cam, w, h, spp=spp, jitter=jitter, seed=1984)
        s0, cf, c3 = assert_first_covers_like_ref(tree, ob, rays)
        if 0.02 < (s0 >= 0).mean():
            assert cf["tris"] < c3["tris"]                 # the exit does remove work wherever rays hit


def test_first_hit_equals_reference_on_degenerate_rays(oracle, scenes, tree):
    """Zero direction components, origins on grid planes and on the scene box, diagonal directions (the rays of
    test_oracle_semantics' box-mode regression test), and origins far from the scene."""
    rng = np.random.default_rng(7)
    tri, rays = degenerate_rays(scenes, rng)
    ob = oracle.Bih(tri)
    s0, _, _ = assert_first_covers_like_ref(tree, ob, rays)
    assert (s0 >= 0).sum() > 1000
    tri = scenes.displaced_sphere(48)
    ob = oracle.Bih(tri)
    for dist in (1e2, 1e4):
        target = rng.uniform(-0.6, 0.6, (4000, 3))
        dirs = rng.normal(size=(4000, 3)); dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
        rays = np.concatenate([(target - dirs * dist).astype(np.float32), dirs.astype(np.float32)], 1).astype(np.float32)
        assert_first_covers_like_ref(tree, ob, rays)


def test_first_hit_keeps_the_reference_misses_on_flat_geometry(oracle, scenes, tree):
    """On axis-aligned walls the reference's strict test skips leaves brute force would test (it hits a farther wall);
    the coverage walk takes the same decisions up to its first hit, so it hits exactly where the reference does."""
    for tri, cam, w, h in ((scenes.cornell_box(), scenes.cornell_camera(), 256, 256),
                           (scenes.atrium(0.05), scenes.atrium_camera(), 240, 135)):
        ob = oracle.Bih(tri)
        for spp, jitter in ((1, False), (2, True)):
            rays = oracle.camera_rays(cam, w, h, spp=spp, jitter=jitter)
            s0, _, _ = assert_first_covers_like_ref(tree, ob, rays)
            if len(tri) < 100:
                _, s2, _ = ob.trace(rays, "brute")
                assert (s0 != s2).sum() > 0                  # the strict test decides on these rays


# ------------------------------------------------------------------------------------------------ GPU: the kernel

COUNTED_CASES = {
    "sphere187": lambda S: (S.displaced_sphere(187), S.pinhole_camera(aspect=160 / 90), 160, 90),
    "cornell": lambda S: (S.cornell_box(), S.cornell_camera(), 96, 96),
    "atrium": lambda S: (S.atrium(0.2), S.atrium_camera(160 / 90), 160, 90),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(COUNTED_CASES))
def test_render_counters_equal_first_hit_oracle(renderer, scenes, oracle, tree, name):
    """render_counted (the instrumented framebuffer kernel) visits exactly the nodes and triangles of mode 'first'."""
    tri, cam, w, h = COUNTED_CASES[name](scenes)
    pt = tree(oracle.Bih(tri))
    renderer.load_models(tri).build()
    for spp in (1, 3, 4, 16):
        for jitter in (False, True):
            rays = oracle.camera_rays(cam, w, h, spp=spp, jitter=jitter, seed=1984)
            cf = pt.walk(rays, "first")["counters"]
            cnt = renderer.render_counted(cam, w, h, spp=spp, seed=1984, jitter=jitter)
            assert cnt["rays"] == len(rays)
            assert (cnt["nodes"], cnt["tris"], cnt["max_stack"]) == (cf["nodes"], cf["tris"], cf["max_stack"]), (spp, jitter)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sphere187", "cornell", "atrium"])
def test_framebuffers_equal_closest_hit_image(renderer, scenes, oracle, name):
    """Every framebuffer path -- lane groupings, tile shards, sample shards and unit interleave (hit counts:
    BIHRT_RENDER_COUNTS, then resolve) -- gives the image of the closest-hit oracle bit for bit."""
    import torch
    from bihrt import multi
    tri, cam, w, h = COUNTED_CASES[name](scenes)
    ob = oracle.Bih(tri)
    renderer.load_models(tri).build()
    for spp in (1, 3, 4, 16):
        for jitter in (False, True):
            rays = oracle.camera_rays(cam, w, h, spp=spp, jitter=jitter, seed=1984)
            _, s0, _ = ob.trace(rays, "ref")
            exp = oracle.pack_framebuffer(s0, w, h, spp).reshape(h, w)
            for groups in (-1, 1, 2):
                renderer.set_option("trace_lane_groups", groups)
                fb = renderer.render(cam, w, h, spp=spp, seed=1984, jitter=jitter).framebuffer()
                np.testing.assert_array_equal(fb, exp, err_msg="spp %d jitter %s groups %d" % (spp, jitter, groups))
            renderer.set_option("trace_lane_groups", -1)
    # shards and hit counts, jittered 4 spp
    spp = 4
    rays = oracle.camera_rays(cam, w, h, spp=spp, jitter=True, seed=1984)
    _, s0, _ = ob.trace(rays, "ref")
    exp = oracle.pack_framebuffer(s0, w, h, spp).reshape(h, w)
    acc = np.zeros_like(exp)
    for k in range(3):
        acc += renderer.render(cam, w, h, spp=spp, jitter=True, shard=(k, 3)).framebuffer()
    np.testing.assert_array_equal(acc, exp)
    hits_per_pixel = (s0 >= 0).reshape(h, w, spp).sum(axis=2).astype(np.int32)
    counts = torch.zeros((h, w), dtype=torch.int32, device="cuda")
    for k in range(2):
        s_a, s_b = multi.sample_range(spp, k, 2)
        renderer.render_samples(cam, w, h, spp, s_a, s_b, jitter=True)
        renderer.sync()
        counts += multi.framebuffer_tensor(renderer)
        torch.cuda.synchronize()
    np.testing.assert_array_equal(counts.cpu().numpy(), hits_per_pixel)
    counts.zero_()
    for k in range(4):
        renderer.render_interleaved(cam, w, h, spp, k, 4, jitter=True)
        renderer.sync()
        counts += multi.framebuffer_tensor(renderer)
        torch.cuda.synchronize()
    np.testing.assert_array_equal(counts.cpu().numpy(), hits_per_pixel)
    multi.framebuffer_tensor(renderer).copy_(counts)
    torch.cuda.synchronize()
    np.testing.assert_array_equal(renderer.framebuffer_resolve(spp).framebuffer(), exp)
