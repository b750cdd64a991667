"""Framebuffer renders are coverage queries: a sample ends at the first triangle it accepts.

A pixel's colour (and the hit counts of the sharded renders) depends only on WHETHER each sample hits, so the framebuffer
kernel (csrc/trace.cu, MODE 1, COVER) stops a sample's walk at its first accepted triangle instead of
searching on for the closest one.  tests/coverage_oracle.c restates that walk on the CPU (mode "first": the oracle's
"box" traversal with that one exit).  The CPU tests check that "first" hits exactly where "ref" and "box" hit and never
does more work than "box"; the GPU tests pin render_counted's counters to "first" exactly, and every framebuffer path to
the image of the closest-hit oracle.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_gpu_golden_scenes import SCENES as GOLDEN

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.join(os.path.dirname(HERE), "oracle")


@pytest.fixture(scope="session")
def trace_first(tmp_path_factory):
    """Builds tests/coverage_oracle.c (the oracle's source plus mode "first") into a temporary directory; returns
    trace_first(bih, rays) -> t, slot, prim, counters, with the arguments and results of oracle.Bih.trace."""
    out = str(tmp_path_factory.mktemp("coverage_oracle") / "libcoverage_oracle.so")
    cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
    subprocess.check_call([cc, "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-fvisibility=hidden", "-std=c11",
                           "-shared", "-I" + ORACLE_DIR, "-o", out, os.path.join(HERE, "coverage_oracle.c"), "-lm"])
    lib = C.CDLL(out)

    def _p(a):
        return a.ctypes.data_as(C.c_void_p)

    def run(ob, rays6):
        rays6 = np.ascontiguousarray(rays6, dtype=np.float32).reshape(-1, 6)
        nr = rays6.shape[0]
        t, slot, prim = np.empty(nr, np.float32), np.empty(nr, np.int32), np.empty(nr, np.int32)
        cnt = np.zeros(3, np.uint64)
        keep = [np.ascontiguousarray(x) for x in (ob.tris_idx, ob.cnt, ob.first, ob.clip, ob.axis, ob.is_leaf, ob.children)]
        lib.orc_trace_first(_p(ob.tri9), C.c_int64(ob.n), C.c_int64(ob.nu), *[_p(k) for k in keep], _p(ob.scene_lo),
                            _p(ob.scene_hi), _p(rays6), C.c_int64(nr), _p(t), _p(slot), _p(prim), _p(cnt), C.c_int(0))
        return t, slot, prim, {"nodes": int(cnt[0]), "tris": int(cnt[1]), "max_stack": int(cnt[2])}
    return run


def assert_first_covers_like_ref(trace_first, ob, rays):
    """'first' hits exactly where 'ref' and 'box' hit, with no more nodes or triangle tests than 'box'; returns the counters."""
    t0, s0, _ = ob.trace(rays, "ref")
    t3, s3, _, c3 = ob.trace(rays, "box", want_counters=True)
    tf, sf, pf, cf = trace_first(ob, rays)
    np.testing.assert_array_equal(sf >= 0, s0 >= 0)
    np.testing.assert_array_equal(sf >= 0, s3 >= 0)
    hit = sf >= 0
    assert np.all(tf[hit] > 0) and np.all(tf[~hit] == np.finfo(np.float32).max) and np.all(pf[~hit] == -1)
    assert np.all(tf[hit] >= t3[hit])                  # the first accepted triangle is never closer than the closest one
    assert cf["nodes"] <= c3["nodes"] and cf["tris"] <= c3["tris"] and cf["max_stack"] <= c3["max_stack"]
    return s0, cf, c3


# ------------------------------------------------------------------------------------------------ CPU: the restatement

@pytest.mark.parametrize("name", list(GOLDEN))
def test_first_hit_equals_reference_on_golden_scenes(oracle, scenes, trace_first, name):
    tri, cam, w, h = GOLDEN[name](scenes)
    ob = oracle.Bih(tri)
    for spp, jitter in ((1, False), (2, True)):
        rays = oracle.camera_rays(cam, w, h, spp=spp, jitter=jitter, seed=1984)
        s0, cf, c3 = assert_first_covers_like_ref(trace_first, ob, rays)
        if 0.02 < (s0 >= 0).mean():
            assert cf["tris"] < c3["tris"]                 # the exit does remove work wherever rays hit


def test_first_hit_equals_reference_on_degenerate_rays(oracle, scenes, trace_first):
    """Zero direction components, origins on grid planes and on the scene box, diagonal directions (the rays of
    test_oracle_semantics' box-mode regression test), and origins far from the scene."""
    tri = np.concatenate([scenes.cornell_box(), scenes.displaced_sphere(24) * 0.3])
    ob = oracle.Bih(tri)
    rng = np.random.default_rng(7)
    n = 20000
    o = rng.uniform(-1.2, 1.2, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    which = rng.integers(0, 7, n)
    d[which == 0, 0] = 0.0
    d[which == 1, 1] = 0.0
    d[which == 2, 2] = 0.0
    d[which == 3, :2] = 0.0
    o[which == 4] = np.round(o[which == 4] * 4) / 4
    d[which == 5] = np.sign(d[which == 5])
    o[which == 6, 0] = -1.0
    d[(which == 3) & (d[:, 2] == 0), 2] = 1.0
    rays = np.concatenate([o, d], 1).astype(np.float32)
    s0, _, _ = assert_first_covers_like_ref(trace_first, ob, rays)
    assert (s0 >= 0).sum() > 1000
    tri = scenes.displaced_sphere(48)
    ob = oracle.Bih(tri)
    for dist in (1e2, 1e4):
        target = rng.uniform(-0.6, 0.6, (4000, 3))
        dirs = rng.normal(size=(4000, 3)); dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
        rays = np.concatenate([(target - dirs * dist).astype(np.float32), dirs.astype(np.float32)], 1).astype(np.float32)
        assert_first_covers_like_ref(trace_first, ob, rays)


def test_first_hit_keeps_the_reference_misses_on_flat_geometry(oracle, scenes, trace_first):
    """On axis-aligned walls the reference's strict test skips leaves brute force would test (it hits a farther wall);
    the coverage walk takes the same decisions up to its first hit, so it hits exactly where the reference does."""
    for tri, cam, w, h in ((scenes.cornell_box(), scenes.cornell_camera(), 256, 256),
                           (scenes.atrium(0.05), scenes.atrium_camera(), 240, 135)):
        ob = oracle.Bih(tri)
        for spp, jitter in ((1, False), (2, True)):
            rays = oracle.camera_rays(cam, w, h, spp=spp, jitter=jitter)
            s0, _, _ = assert_first_covers_like_ref(trace_first, ob, rays)
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
def test_render_counters_equal_first_hit_oracle(renderer, scenes, oracle, trace_first, name):
    """render_counted (the instrumented framebuffer kernel) visits exactly the nodes and triangles of mode 'first'."""
    tri, cam, w, h = COUNTED_CASES[name](scenes)
    ob = oracle.Bih(tri)
    renderer.load_models(tri).build()
    for spp in (1, 3, 4, 16):
        for jitter in (False, True):
            rays = oracle.camera_rays(cam, w, h, spp=spp, jitter=jitter, seed=1984)
            _, _, _, cf = trace_first(ob, rays)
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
