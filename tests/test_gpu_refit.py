"""bihrt_refit on the GPU, held bit for bit to its CPU restatement (tests/test_refit_oracle.py, refit_bih) and every query on
a refit tree held to the restated tree's walks.

Each case builds mesh a (parity), moves its vertices to b (bihrt_scene_update_vertices) and refits.  Then the reference
view (order, topology and the build's now stale Morton codes, clip planes, scene box), the exported blob (header, planes,
children boxes, records), bihrt_trace with and without counters, bihrt_trace_any, bihrt_intersect (closest and any, one-
and two-sided, on assorted intervals), the camera kernels, bihrt_closest_point and bihrt_winding_number all equal the
restatement of the refit of a's build to b.  The sizes straddle the heap levels of heap_levels_launch: no k_heap_up
(n <= 256), one launch, chained levels (n > 65536).
"""
import itertools

import numpy as np
import pytest

from closest_oracle import closest  # noqa: F401  (fixture)
from conftest import assert_view_equals_oracle
from test_closest_oracle import assert_closest_equal, queries
from test_gpu_octant_walk import check_frame
from test_refit_oracle import DEFORMATIONS, deform, moved_sphere, random_rays, refit_bih, sphere
from test_winding_oracle import assert_bits, sample_points
from walk_oracle import OUTS, assert_blob_equals, assorted_intervals, bits, blob_of, rays8, tree  # noqa: F401  (tree: fixture)
from winding_oracle import winding  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu

W, H = 331, 197
STATE, INVALID = -4, -1


def refit(renderer, a, b):
    renderer.set_option("morton_bits", 30)
    renderer.load_models(a).build()
    renderer.update_vertices(b)
    renderer.refit()
    return renderer


def camera(tri):
    v = np.asarray(tri, np.float64).reshape(-1, 3)
    lo, hi = v.min(0), v.max(0)
    c, diag = (lo + hi) / 2, max(np.linalg.norm(hi - lo), 1e-3)
    return c, diag


def frame_camera(scenes, tri):
    """A view of the whole scene from above, in front and to the side."""
    c, diag = camera(tri)
    return scenes.look_at_camera(c + diag * np.array([0.7, 0.5, -1.3]), c, 0.35, W / H)


def check_rays(renderer, rt, rays, what):
    """trace (with and without counters), trace_any at three tmax and intersect's four kinds equal the walks of rt."""
    res = rt.walk(rays)
    t, s, p, cnt = renderer.trace(rays, counted=True)
    assert_bits(t, res["t"], what + " counted t")
    np.testing.assert_array_equal(s, res["slot"], err_msg=what)
    np.testing.assert_array_equal(p, res["prim"], err_msg=what)
    c0 = res["counters"]
    assert (cnt["nodes"], cnt["tris"], cnt["max_stack"]) == (c0["nodes"], c0["tris"], c0["max_stack"]), what
    t, s, p = renderer.trace(rays)
    assert_bits(t, res["t"], what + " t")
    np.testing.assert_array_equal(s, res["slot"], err_msg=what)
    np.testing.assert_array_equal(p, res["prim"], err_msg=what)
    for tmax in (0.25, 1.0, 3.0):
        np.testing.assert_array_equal(renderer.trace_any(rays, tmax=tmax), rt.walk(rays, "any", tmax=np.float32(tmax))["slot"],
                                      err_msg="%s trace_any %g" % (what, tmax))
    tmin, tmax = assorted_intervals(res["t"], seed=31)
    r8 = rays8(rays, tmin, tmax)
    for any_hit, two_sided in itertools.product((False, True), repeat=2):
        want = rt.walk(r8, "any" if any_hit else "closest", two_sided=two_sided)
        got = renderer.intersect(r8, any_hit=any_hit, two_sided=two_sided)
        for k in OUTS:
            np.testing.assert_array_equal(bits(got[k]), bits(want[k]), err_msg="%s intersect any %s two-sided %s %s" %
                                          (what, any_hit, two_sided, k))
    return res


def check_frames(renderer, oracle, scenes, rt, what):
    """render / render_counted (check_frame), render_hits, and render_samples and render_interleaved summed and resolved,
    on a ragged frame at 1 and 4 spp."""
    import torch
    from bihrt import multi
    cam = frame_camera(scenes, rt.tri9)
    for spp, jitter in ((1, False), (4, True)):
        rays, s0 = check_frame(renderer, oracle, rt, cam, W, H, spp, jitter)
        first = rt.walk(rays, "first")["slot"]
        fb = renderer.render(cam, W, H, spp=spp, seed=1984, jitter=jitter).framebuffer()
        np.testing.assert_array_equal(fb.ravel(), oracle.pack_framebuffer(first, W, H, spp), err_msg=what)
        res = rt.walk(rays)
        t, s, p = renderer.render_hits(cam, W, H, spp=spp, jitter=jitter)
        assert_bits(t, res["t"], what + " render_hits")
        np.testing.assert_array_equal(s, res["slot"], err_msg=what)
        np.testing.assert_array_equal(p, res["prim"], err_msg=what)
    spp = 4
    exp = renderer.render(cam, W, H, spp=spp, jitter=True).framebuffer().copy()
    for parts, kind in ((2, "samples"), (4, "interleaved")):
        counts = torch.zeros((H, W), dtype=torch.int32, device="cuda")
        for k in range(parts):
            if kind == "samples":
                renderer.render_samples(cam, W, H, spp, *multi.sample_range(spp, k, parts), jitter=True)
            else:
                renderer.render_interleaved(cam, W, H, spp, k, parts, jitter=True)
            renderer.sync()
            counts += multi.framebuffer_tensor(renderer)
            torch.cuda.synchronize()
        multi.framebuffer_tensor(renderer).copy_(counts)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(renderer.framebuffer_resolve(spp).framebuffer(), exp, err_msg="%s %s" % (what, kind))


def check_points(renderer, rt, closest, winding, nq, what):  # noqa: F811
    """closest_point equals the walk and brute force; winding_number at beta = inf equals the exact sum over every slot, at
    beta = 2 the winding walk."""
    q = queries(sample_points(rt.tri9, np.random.default_rng(5), nq // 2))
    got = renderer.closest_point(q)
    assert_closest_equal(got, closest(rt, q), what + " closest walk")
    assert_closest_equal(got, closest(rt, q, brute=True), what + " closest brute force")
    assert_bits(renderer.winding_number(q, np.inf), winding(rt, q, brute=True)[0], what + " winding inf")
    assert_bits(renderer.winding_number(q, 2.0), winding(rt, q, 2.0)[0], what + " winding 2")


def check_refit(renderer, oracle, scenes, tree, closest, winding, r, what, frames=True):  # noqa: F811
    """Everything on the renderer's refit tree against the restated refit tree r."""
    assert_view_equals_oracle(renderer.reference_view(), r)
    rt = tree(r)
    assert_blob_equals(blob_of(renderer), rt, what)
    check_rays(renderer, rt, random_rays(r.tri9, 16384, seed=3), what)
    if frames:
        check_frames(renderer, oracle, scenes, rt, what)
    check_points(renderer, rt, closest, winding, 2000 if r.n <= 70000 else 200, what)
    return rt


# ------------------------------------------------------------------------------------------------ deformations and sizes

@pytest.mark.parametrize("how", DEFORMATIONS)
def test_refit_of_the_sphere_equals_restatement(renderer, oracle, scenes, tree, closest, winding, how):  # noqa: F811
    a, b = sphere(scenes), moved_sphere(scenes, how)
    refit(renderer, a, b)
    check_refit(renderer, oracle, scenes, tree, closest, winding, refit_bih(oracle.Bih(a), b), how)


def test_refit_of_the_jittered_atrium_equals_restatement(renderer, oracle, scenes, tree, closest, winding):  # noqa: F811
    a = scenes.atrium(0.2)
    b = deform(a, "jitter", seed=4)
    refit(renderer, a, b)
    check_refit(renderer, oracle, scenes, tree, closest, winding, refit_bih(oracle.Bih(a), b), "atrium jitter")


SIZES = (1, 2, 3, 7, 255, 256, 257, 65536, 65537)


def sized(scenes, n, phase):
    """n triangles of the displaced sphere at `phase`; n = 7: seven identical triangles (one leaf), which the motion
    separates."""
    if n == 7:
        one = np.tile(np.array([[0, 0, 0, 1, 0, 0, 0, 1, 0]], np.float32), (7, 1))
        return one if phase == 0 else deform(one, "jitter", seed=7)
    return np.ascontiguousarray(scenes.displaced_sphere(182, phase=phase)[:n])


@pytest.mark.parametrize("n", SIZES)
def test_refit_at_heap_level_boundaries(renderer, oracle, scenes, tree, closest, winding, n):  # noqa: F811
    """Sizes around the heap levels (and nu = 1): a phase change, and a floor clamp of the same build."""
    a = sized(scenes, n, 0.0)
    ob = oracle.Bih(a)
    assert ob.nu == 1 or n != 7
    for how in ("phase0.7", "floor0"):
        b = sized(scenes, n, 0.7) if how == "phase0.7" else deform(a, how)
        refit(renderer, a, b)
        check_refit(renderer, oracle, scenes, tree, closest, winding, refit_bih(ob, b), "n %d %s" % (n, how), frames=n >= 255)


def test_refit_of_one_million_triangles(renderer, oracle, scenes, tree, closest, winding):  # noqa: F811
    nseg = scenes.SPHERE_NSEG["1m"]
    a, b = scenes.displaced_sphere(nseg), scenes.displaced_sphere(nseg, phase=0.7)
    refit(renderer, a, b)
    check_refit(renderer, oracle, scenes, tree, closest, winding, refit_bih(oracle.Bih(a), b), "1m")


# ------------------------------------------------------------------------------------------------ chains and replicas

def test_chain_of_refits_uses_the_build_topology(renderer, oracle, scenes, tree):  # noqa: F811
    """refit to b, then c, then back to a: each equals the restatement from the build's topology, and the last one
    reproduces the build's blob byte for byte."""
    a = sphere(scenes)
    ob = oracle.Bih(a)
    renderer.load_models(a).build()
    words = blob_of(renderer).copy()
    for how in ("phase0.7", "scale_translate", None):
        b = a if how is None else moved_sphere(scenes, how)
        renderer.update_vertices(b)
        renderer.refit()
        r = refit_bih(ob, b)
        assert_view_equals_oracle(renderer.reference_view(), r)
        rt = tree(r)
        assert_blob_equals(blob_of(renderer), rt, str(how))
        check_rays(renderer, rt, random_rays(b, 4096, seed=2), str(how))
    np.testing.assert_array_equal(blob_of(renderer), words)


def test_replicas_of_a_refit_tree(renderer, oracle, scenes, tree, closest, winding):  # noqa: F811
    """A refit tree exported and imported into a second context, and copied into a third: the replicas answer every query as
    the refitting context does, and refuse a refit of their own."""
    import torch
    import bihrt
    a, b = sphere(scenes), moved_sphere(scenes, "floor0")
    refit(renderer, a, b)
    rays = random_rays(b, 8192, seed=6)
    r8 = rays8(rays, 0.0, np.inf)
    q = queries(sample_points(b, np.random.default_rng(6), 1000))
    cam = frame_camera(scenes, b)

    def answers(r):
        out = list(r.trace(rays)) + [r.trace_any(rays, tmax=1.0)]
        out += [r.intersect(r8, any_hit=k, two_sided=True)[o] for k in (False, True) for o in OUTS]
        out += [r.closest_point(q)[o] for o in ("d2", "slot", "q")] + [r.winding_number(q, 2.0)]
        out += [r.render(cam, W, H, spp=4, jitter=True).framebuffer().copy()]
        return [bits(np.asarray(x)) for x in out]
    want = answers(renderer)
    nbytes = renderer.bih_blob_bytes()
    blob = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    renderer.bih_export(blob, nbytes)
    renderer.sync()
    r2, r3 = bihrt.Renderer(0), bihrt.Renderer(0)
    try:
        r2.bih_import(blob, nbytes)
        assert r3._lib.bihrt_bih_copy(r3._ctx, renderer._ctx) == 0
        for r, what in ((r2, "imported"), (r3, "copied")):
            for i, (g, w) in enumerate(zip(answers(r), want)):
                np.testing.assert_array_equal(g, w, err_msg="%s output %d" % (what, i))
            with pytest.raises(bihrt.BihrtError) as e:
                r.refit()
            assert e.value.code == STATE, what
    finally:
        r2.close()
        r3.close()


# ------------------------------------------------------------------------------------------------ state rules

def test_refit_state_rules(renderer, scenes):
    """refit is refused before any build, after loading another mesh of the same n, after a quality build and with
    morton_bits 63; update_vertices keeps n; every query between update_vertices and the next refit or build is refused."""
    import bihrt
    a, b = sphere(scenes), moved_sphere(scenes, "phase0.7")
    other = scenes.displaced_sphere(96, seed=11)

    def refused(fn, code=STATE):
        with pytest.raises(bihrt.BihrtError) as e:
            fn()
        assert e.value.code == code

    refused(renderer.refit)                                              # nothing loaded
    renderer.load_models(a)
    refused(renderer.refit)                                              # loaded, never built
    renderer.build()
    renderer.load_models(other)
    refused(renderer.refit)                                              # another mesh, the same n
    renderer.build()
    renderer.refit()
    try:
        renderer.set_option("morton_bits", 63)
        refused(renderer.refit)                                          # quality mode set, parity tree built
        renderer.build()
        renderer.set_option("morton_bits", 30)
        refused(renderer.refit)                                          # after a quality build
    finally:
        renderer.set_option("morton_bits", 30)
    renderer.load_models(a).build()
    refused(lambda: renderer.update_vertices(b[:-1]), INVALID)
    refused(lambda: renderer.update_vertices(np.concatenate([b, b[:1]])), INVALID)
    renderer.update_vertices(b)
    rays = random_rays(b, 256)
    q = queries(sample_points(b, np.random.default_rng(1), 64))
    cam = frame_camera(scenes, b)
    for name, fn in (("trace", lambda: renderer.trace(rays)), ("trace_counted", lambda: renderer.trace(rays, counted=True)),
                     ("trace_any", lambda: renderer.trace_any(rays)), ("intersect", lambda: renderer.intersect(rays8(rays))),
                     ("closest_point", lambda: renderer.closest_point(q)), ("winding_number", lambda: renderer.winding_number(q)),
                     ("render", lambda: renderer.render(cam, 64, 32)), ("render_hits", lambda: renderer.render_hits(cam, 64, 32)),
                     ("render_counted", lambda: renderer.render_counted(cam, 64, 32)),
                     ("render_samples", lambda: renderer.render_samples(cam, 64, 32, 4, 0, 2)),
                     ("render_interleaved", lambda: renderer.render_interleaved(cam, 64, 32, 4, 0, 2)),
                     ("reference_view", renderer.reference_view), ("bih_blob_bytes", renderer.bih_blob_bytes)):
        try:
            refused(fn)
        except AssertionError as e:
            raise AssertionError("%s after update_vertices: %s" % (name, e))
    renderer.refit()
    renderer.trace(rays)


def test_device_input_refits_as_host_input(renderer, oracle, scenes, tree):  # noqa: F811
    import torch
    a, b = sphere(scenes), moved_sphere(scenes, "shuffle")
    refit(renderer, a, b)
    host = blob_of(renderer).copy()
    renderer.load_models(a).build()
    renderer.update_vertices(torch.from_numpy(b).cuda())
    renderer.refit()
    np.testing.assert_array_equal(blob_of(renderer), host)
    assert_blob_equals(host, tree(refit_bih(oracle.Bih(a), b)), "device input")
