"""GPU traversal + intersection vs the oracle, through the C ABI.

Tolerances (BASELINE.json north_star): hit slot / primitive ids bit-exact except on documented ties,
at most 1e-4 of the rays; hit distance within 1e-5 relative.  Against the oracle's restatement of the shipped
traversal (mode "box": pruned traversal + children boxes, the same logical algorithm in the same IEEE arithmetic) the kernel
is expected to be bit-identical, node and triangle counters included."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ID_MISMATCH_MAX = 1e-4
T_REL_TOL = 1e-5


def compare(t_gpu, s_gpu, p_gpu, t_ref, s_ref, p_ref):
    n = len(s_ref)
    bad = s_gpu != s_ref
    assert bad.sum() <= ID_MISMATCH_MAX * n, "%d of %d slot ids differ" % (bad.sum(), n)
    ok = ~bad
    np.testing.assert_array_equal(p_gpu[ok], p_ref[ok])
    hit = ok & (s_ref >= 0)
    np.testing.assert_allclose(t_gpu[hit], t_ref[hit], rtol=T_REL_TOL, atol=0)
    assert np.all(t_gpu[ok & (s_ref < 0)] == np.finfo(np.float32).max)


CASES = {
    "dodecahedron": lambda S: (S.dodecahedron(), S.pinhole_camera(aspect=1.0), 128, 128),
    "cornell": lambda S: (S.cornell_box(), S.cornell_camera(), 512, 512),                 # BASELINE config 1
    "sphere187": lambda S: (S.displaced_sphere(187), S.pinhole_camera(), 1920, 1080),     # BASELINE config 2
    "atrium": lambda S: (S.atrium(), S.atrium_camera(), 960, 540),                        # BASELINE config 3
    "soup": lambda S: (S.random_soup(100000), S.pinhole_camera(), 640, 360),
    "single_cell": lambda S: (np.tile(np.array([[0, 0, 0, 1, 0, 0, 0, 1, 0]], np.float32), (3, 1)),
                              S.look_at_camera((0.3, 0.3, 2), (0.3, 0.3, 0), 0.5, 1.0), 64, 64),
}


@pytest.mark.parametrize("name", list(CASES))
def test_trace_matches_reference_semantics(renderer, scenes, oracle, name):
    tri, cam, w, h = CASES[name](scenes)
    ob = oracle.Bih(tri)
    rays = oracle.camera_rays(cam, w, h)
    renderer.load_models(tri).build()
    t, s, p, cnt = renderer.trace(rays, counted=True)
    t0, s0, p0 = ob.trace(rays, "ref")
    compare(t, s, p, t0, s0, p0)
    # same logical algorithm on the CPU (pruned traversal + children boxes): bit-identical, counters included
    t1, s1, p1, c1 = ob.trace(rays, "box", want_counters=True)
    np.testing.assert_array_equal(s, s1)
    np.testing.assert_array_equal(t, t1)
    assert cnt["nodes"] == c1["nodes"] and cnt["tris"] == c1["tris"] and cnt["max_stack"] == c1["max_stack"]
    # uninstrumented kernel gives the same answer
    t2, s2, p2 = renderer.trace(rays)
    np.testing.assert_array_equal(s, s2)
    np.testing.assert_array_equal(t, t2)
    np.testing.assert_array_equal(p, p2)


def test_incoherent_secondary_rays(renderer, scenes, oracle):
    """BASELINE config 3: shadow rays to a point light and a diffuse bounce from the primary hits."""
    tri = scenes.atrium()
    ob = oracle.Bih(tri)
    cam = scenes.atrium_camera()
    rays = oracle.camera_rays(cam, 480, 270)
    renderer.load_models(tri).build()
    t, s, p = renderer.trace(rays)
    hit = s >= 0
    P = rays[hit, :3] + t[hit, None] * rays[hit, 3:]
    v = tri[p[hit]].reshape(-1, 3, 3)
    nrm = np.cross(v[:, 1] - v[:, 0], v[:, 2] - v[:, 0])
    nrm /= np.maximum(np.linalg.norm(nrm, axis=1, keepdims=True), 1e-20)
    P = (P + 1e-3 * nrm).astype(np.float32)
    light = np.array([0.0, 0.8, 0.0], np.float32)
    shadow = np.concatenate([P, (light - P)], axis=1).astype(np.float32)
    rng = np.random.default_rng(1984)
    d = rng.normal(size=P.shape)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    d = np.where((d * nrm).sum(1, keepdims=True) < 0, -d, d)
    bounce = np.concatenate([P, d], axis=1).astype(np.float32)
    for batch in (shadow, bounce):
        tg, sg, pg = renderer.trace(batch)
        t0, s0, p0 = ob.trace(batch, "ref")
        compare(tg, sg, pg, t0, s0, p0)


def test_one_million_triangles_primary(renderer, scenes, oracle):
    """BASELINE config 5 scene (1 002 528 triangles), 960x540 sample of the 1080p frame vs the oracle."""
    tri = scenes.displaced_sphere(708)
    ob = oracle.Bih(tri)
    rays = oracle.camera_rays(scenes.pinhole_camera(), 960, 540)
    renderer.load_models(tri).build()
    t, s, p = renderer.trace(rays)
    t0, s0, p0 = ob.trace(rays, "ref")
    compare(t, s, p, t0, s0, p0)
    assert 0.2 < (s >= 0).mean() < 0.4


def test_device_buffers_and_mixed_outputs(renderer, scenes, oracle):
    import torch
    tri = scenes.displaced_sphere(64)
    rays = oracle.camera_rays(scenes.pinhole_camera(), 320, 180)
    renderer.load_models(tri).build()
    t, s, p = renderer.trace(rays)
    dr = torch.from_numpy(rays).cuda()
    td, sd, pd = renderer.trace(dr)
    renderer.sync()
    np.testing.assert_array_equal(td.cpu().numpy(), t)
    np.testing.assert_array_equal(sd.cpu().numpy(), s)
    np.testing.assert_array_equal(pd.cpu().numpy(), p)
    # ragged ray counts
    for n in (1, 31, 33, 1000):
        tn, sn, pn = renderer.trace(rays[:n])
        np.testing.assert_array_equal(sn, s[:n])
    tn, sn, pn = renderer.trace(rays[:0])
    assert len(sn) == 0


def test_render_hits_framebuffer_and_shards(renderer, scenes, oracle):
    tri = scenes.displaced_sphere(96)
    cam = scenes.pinhole_camera(aspect=200 / 120)
    w, h, spp = 200, 120, 4
    ob = oracle.Bih(tri)
    renderer.load_models(tri).build()
    for jitter in (False, True):
        rays = oracle.camera_rays(cam, w, h, spp=spp, jitter=jitter, seed=1984)
        t0, s0, p0 = ob.trace(rays, "ref")
        t, s, p = renderer.render_hits(cam, w, h, spp=spp, seed=1984, jitter=jitter)
        compare(t, s, p, t0, s0, p0)                      # in-kernel ray generation == oracle's rays
        fb = renderer.render(cam, w, h, spp=spp, seed=1984, jitter=jitter).framebuffer()
        exp = oracle.pack_framebuffer(s, w, h, spp).reshape(h, w)
        np.testing.assert_array_equal(fb, exp)
    # tile shards: disjoint, zero elsewhere, union == full image  (multi-GPU partition)
    full = renderer.render(cam, w, h, spp=spp, jitter=True).framebuffer().copy()
    acc = np.zeros_like(full)
    for k in range(3):
        part = renderer.render(cam, w, h, spp=spp, jitter=True, shard=(k, 3)).framebuffer()
        assert np.all((acc == 0) | (part == 0))
        acc += part
    np.testing.assert_array_equal(acc, full)
    # sample shards: per-pixel hit counts of disjoint sample ranges; sum + resolve == full image
    from bihrt import multi
    import torch
    counts = torch.zeros((h, w), dtype=torch.int32, device="cuda")
    for k in range(3):
        s0, s1 = multi.sample_range(spp, k, 3)
        renderer.render_samples(cam, w, h, spp, s0, s1, jitter=True)
        renderer.sync()                                   # the library runs on its own stream here
        counts += multi.framebuffer_tensor(renderer)
        torch.cuda.synchronize()
    assert int(counts.max()) <= spp
    multi.framebuffer_tensor(renderer).copy_(counts)
    torch.cuda.synchronize()
    np.testing.assert_array_equal(renderer.framebuffer_resolve(spp).framebuffer(), full)
    # unit interleave: every rank walks every tile, owns every count-th 32-ray unit; disjoint pixels
    for count in (2, 4, 8):
        counts.zero_()
        owned = torch.zeros((h, w), dtype=torch.int32, device="cuda")
        for k in range(count):
            renderer.render_interleaved(cam, w, h, spp, k, count, jitter=True)
            renderer.sync()
            part = multi.framebuffer_tensor(renderer)
            counts += part
            owned += (part > 0).int()
            torch.cuda.synchronize()
        assert int(owned.max()) <= 1
        multi.framebuffer_tensor(renderer).copy_(counts)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(renderer.framebuffer_resolve(spp).framebuffer(), full)


def test_bih_blob_roundtrip(scenes, oracle):
    """Replication path of the multi-GPU design: export -> (broadcast) -> import on another context."""
    import torch
    import bihrt
    tri = scenes.displaced_sphere(80)
    rays = oracle.camera_rays(scenes.pinhole_camera(), 256, 144)
    a, b = bihrt.Renderer(0), bihrt.Renderer(0)
    a.load_models(tri).build()
    nbytes = a.bih_blob_bytes()
    blob = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    a.bih_export(blob, nbytes)
    a.sync()
    b.bih_import(blob, nbytes)
    ta, sa, pa = a.trace(rays)
    tb, sb, pb = b.trace(rays)
    np.testing.assert_array_equal(sa, sb)
    np.testing.assert_array_equal(ta, tb)
    np.testing.assert_array_equal(pa, pb)
    a.close(); b.close()


@pytest.mark.parametrize("opts", [{"trace_sm_queues": 1}, {"trace_sm_queues": 0}, {"trace_blocks_per_sm": 3}],
                         ids=["sm_queues_1", "sm_queues_0", "blocks_per_sm_3"])
def test_scheduling_variants_do_not_change_results(renderer, scenes, oracle, opts):
    """Scheduling options (per-SM work queues, occupancy) reorder work across warps but never a ray's own
    sequence of leaf tests: hits must stay bit-identical."""
    for tri, cam, w, h in ((scenes.atrium(0.2), scenes.atrium_camera(), 320, 180),
                           (scenes.displaced_sphere(187), scenes.pinhole_camera(), 480, 270)):
        ob = oracle.Bih(tri)
        rays = oracle.camera_rays(cam, w, h, spp=2, jitter=True)
        t1, s1, p1, c1 = ob.trace(rays, "box", want_counters=True)
        renderer.load_models(tri).build()
        for k, v in opts.items():
            renderer.set_option(k, v)
        t, s, p, cnt = renderer.trace(rays, counted=True)
        np.testing.assert_array_equal(s, s1)
        np.testing.assert_array_equal(t, t1)
        np.testing.assert_array_equal(p, p1)
        assert cnt["tris"] == c1["tris"] and cnt["nodes"] == c1["nodes"]
        tt, ss, pp = renderer.render_hits(cam, w, h, spp=2, jitter=True)
        np.testing.assert_array_equal(ss, s1)
        np.testing.assert_array_equal(tt, t1)


@pytest.mark.parametrize("spp", [1, 4, 3])
def test_cost_ordered_tiles_do_not_change_the_frame(scenes, oracle, spp):
    """The second and later launches of a frame geometry trace the tiles in the cost order the previous launch
    measured (expensive tiles first).  Pixels, per-sample hits and the framebuffer must not depend on that order."""
    import bihrt
    tri = scenes.displaced_sphere(160)
    cam = scenes.pinhole_camera(aspect=331 / 197)
    w, h = 331, 197                                   # ragged edge tiles
    ob = oracle.Bih(tri)
    rays = oracle.camera_rays(cam, w, h, spp=spp, jitter=True)
    t0, s0, _ = ob.trace(rays, "ref")
    fb0 = oracle.pack_framebuffer(s0, w, h, spp)
    r = bihrt.Renderer(0)
    r.load_models(tri).build()
    for order in (2, 1, 0):                           # always / small launches / never
        r.set_option("trace_tile_order", order)
        for rep in range(3):                          # launch 0 has no history, 1 and 2 follow the measured costs
            fb = r.render(cam, w, h, spp=spp, jitter=True).framebuffer()
            np.testing.assert_array_equal(fb.ravel(), fb0)
            tt, ss, _ = r.render_hits(cam, w, h, spp=spp, jitter=True)
            np.testing.assert_array_equal(ss, s0)
            np.testing.assert_array_equal(tt, t0)
            # ray lists are dealt in cost-ordered chunks of 1024 rays (the last one padded): same contract
            tl, sl, pl = r.trace(rays)
            np.testing.assert_array_equal(sl, s0)
            np.testing.assert_array_equal(tl, t0)
            np.testing.assert_array_equal(pl >= 0, s0 >= 0)
            np.testing.assert_array_equal(r.trace_any(rays, tmax=2.5) >= 0, (s0 >= 0) & (t0 < 2.5))
    r.close()


def test_axis_parallel_and_degenerate_rays(renderer, scenes, oracle):
    """Rays with zero direction components (1/0 = inf, 0*inf = NaN plane distances), origins inside the scene,
    on the scene box, and pointing away: the kernel must follow the oracle's IEEE behaviour exactly."""
    tri = np.concatenate([scenes.cornell_box(), scenes.displaced_sphere(24) * 0.3])
    ob = oracle.Bih(tri)
    renderer.load_models(tri).build()
    rng = np.random.default_rng(7)
    n = 20000
    o = rng.uniform(-1.2, 1.2, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    which = rng.integers(0, 7, n)
    d[which == 0, 0] = 0.0                       # parallel to the yz plane
    d[which == 1, 1] = 0.0
    d[which == 2, 2] = 0.0
    d[which == 3, :2] = 0.0                      # axis-parallel
    o[which == 4] = np.round(o[which == 4] * 4) / 4      # origins on grid planes (walls at +-1, box faces)
    d[which == 5] = np.sign(d[which == 5])       # diagonal directions
    o[which == 6, 0] = -1.0                      # exactly on the scene box
    d[(which == 3) & (d[:, 2] == 0), 2] = 1.0
    rays = np.concatenate([o, d], 1).astype(np.float32)
    t, s, p = renderer.trace(rays)
    t0, s0, p0 = ob.trace(rays, "ref")
    bad = s != s0
    assert bad.sum() <= ID_MISMATCH_MAX * n, "%d of %d ids differ" % (bad.sum(), n)
    np.testing.assert_array_equal(t[~bad], t0[~bad])
    t1, s1, _ = ob.trace(rays, "box")
    np.testing.assert_array_equal(s, s1)         # the same logical algorithm, NaN handling included
    np.testing.assert_array_equal(t, t1)


def test_ten_million_triangles(renderer, scenes, oracle):
    """BASELINE config 4 size (9 999 392 triangles): build compared with the oracle bit for bit (sorted codes,
    permutation, leaves, every node) and a ray sample compared with the oracle's literal traversal."""
    from conftest import assert_view_equals_oracle
    tri = scenes.displaced_sphere(2236)
    assert len(tri) == 9999392
    renderer.load_models(tri).build()
    v = renderer.reference_view()
    codes = v["morton_codes"]
    assert np.all(codes[1:] >= codes[:-1])
    assert np.array_equal(np.sort(v["tris_indexes"]), np.arange(len(tri), dtype=np.uint32))
    ob = oracle.Bih(tri)
    assert_view_equals_oracle(v, ob)
    rays = oracle.camera_rays(scenes.pinhole_camera(), 384, 216)
    t, s, p = renderer.trace(rays)
    t0, s0, p0 = ob.trace(rays, "ref")
    compare(t, s, p, t0, s0, p0)


@pytest.mark.parametrize("spp", [1, 3, 6, 12, 32, 40])
def test_sample_counts_and_lane_groups(renderer, scenes, oracle, spp):
    """Any sample count: the samples of a pixel are split over 2^k lanes (k = largest power of two dividing
    spp, at most 32 lanes) -- the image and the per-sample hits must not depend on the grouping."""
    tri = scenes.displaced_sphere(64)
    cam = scenes.pinhole_camera(aspect=96 / 64)
    w, h = 96, 64
    ob = oracle.Bih(tri)
    renderer.load_models(tri).build()
    rays = oracle.camera_rays(cam, w, h, spp=spp, jitter=True, seed=7)
    t0, s0, p0 = ob.trace(rays, "ref")
    exp = oracle.pack_framebuffer(s0, w, h, spp).reshape(h, w)
    for groups in (-1, 1, 2):
        renderer.set_option("trace_lane_groups", groups)
        fb = renderer.render(cam, w, h, spp=spp, seed=7, jitter=True).framebuffer()
        np.testing.assert_array_equal(fb, exp)
        t, s, p = renderer.render_hits(cam, w, h, spp=spp, seed=7, jitter=True)
        np.testing.assert_array_equal(s, s0)
        np.testing.assert_array_equal(t, t0)
