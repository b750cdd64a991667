"""Camera launches refilled in lock step: a warp traces one unit of 32 items at a time (lane i takes item i of the unit),
lanes of padding pixels sit the unit out, units of padding only are skipped, the next unit is fetched one unit ahead, and
a pixel of a lane group is written from a ballot (1 sample per lane) or a shuffle sum (several samples per lane).

The cases are the shapes that exercise those paths and that the other suites do not reach: several samples per lane
(64 spp: 32 lanes x 2 samples; 12 spp: 4 lanes x 3; 96 spp: past the colour table), frames smaller than one unit (most
warps' first unit is already past the end), odd frames whose units are half padding, per-SM queues, a reused tile order,
and the count paths (sample ranges and unit interleave) on an odd frame.  Every frame is compared with the oracle's
framebuffer of its own walk, every per-sample record (render_hits) with the oracle's walk, bit for bit."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def scene(scenes, oracle):
    tri = scenes.displaced_sphere(96)
    return tri, oracle.Bih(tri)


def expected(oracle, ob, cam, w, h, spp, jitter, seed=1984):
    rays = oracle.camera_rays(cam, w, h, spp=spp, jitter=jitter, seed=seed)
    t, s, p = ob.trace(rays, "box")
    return t, s, p, oracle.pack_framebuffer(s, w, h, spp).reshape(h, w)


def check_frame(renderer, oracle, ob, cam, w, h, spp, jitter=True, hits=True):
    t0, s0, p0, fb0 = expected(oracle, ob, cam, w, h, spp, jitter)
    fb = renderer.render(cam, w, h, spp=spp, jitter=jitter).framebuffer()
    np.testing.assert_array_equal(fb, fb0)
    if hits:
        t, s, p = renderer.render_hits(cam, w, h, spp=spp, jitter=jitter)
        np.testing.assert_array_equal(s, s0)
        np.testing.assert_array_equal(p, p0)
        np.testing.assert_array_equal(t, t0)
    return fb0


# (w, h, spp): several samples per lane, frames below one unit and below the grid, odd frames with half-padding units
FRAMES = [(40, 24, 64), (33, 17, 12), (21, 13, 96),
          (1, 1, 1), (1, 1, 16), (1, 1, 64), (3, 2, 1), (3, 2, 16), (3, 2, 64),
          (37, 23, 16), (45, 19, 16), (37, 23, 64), (45, 19, 64), (51, 29, 1)]


@pytest.mark.parametrize("w,h,spp", FRAMES)
def test_lockstep_frames_match_oracle(renderer, scenes, oracle, scene, w, h, spp):
    tri, ob = scene
    renderer.load_models(tri).build()
    check_frame(renderer, oracle, ob, scenes.pinhole_camera(aspect=w / h), w, h, spp)


def test_lockstep_per_sm_queues(renderer, scenes, oracle, scene):
    """1 spp through one queue per SM (units fetched when needed, no prefetch) on a frame of ragged edge tiles."""
    tri, ob = scene
    renderer.set_option("trace_sm_queues", 1)
    renderer.load_models(tri).build()
    w, h = 333, 197
    check_frame(renderer, oracle, ob, scenes.pinhole_camera(aspect=w / h), w, h, 1, jitter=False)
    check_frame(renderer, oracle, ob, scenes.pinhole_camera(aspect=w / h), w, h, 4, hits=False)


def test_lockstep_reused_tile_order(renderer, scenes, oracle, scene):
    """Tile order from the previous launch, over repeated launches: the prefetched unit is mapped through the order when
    it is taken, so every launch draws the same frame."""
    tri, ob = scene
    renderer.set_option("trace_tile_order", 2)
    renderer.load_models(tri).build()
    for w, h, spp in ((200, 120, 16), (131, 77, 1), (131, 77, 64)):
        cam = scenes.pinhole_camera(aspect=w / h)
        fb0 = expected(oracle, ob, cam, w, h, spp, True)[3]
        for _ in range(4):
            np.testing.assert_array_equal(renderer.render(cam, w, h, spp=spp, jitter=True).framebuffer(), fb0)


@pytest.mark.parametrize("spp", [16, 64])
def test_lockstep_count_paths(renderer, scenes, oracle, scene, spp):
    """Hit counts (atomics per pixel and unit) of sample ranges and of interleaved units on an odd frame, summed and
    resolved, equal the oracle's frame."""
    import torch
    from bihrt import multi
    tri, ob = scene
    renderer.load_models(tri).build()
    w, h = 75, 41
    cam = scenes.pinhole_camera(aspect=w / h)
    fb0 = expected(oracle, ob, cam, w, h, spp, True)[3]
    counts = torch.zeros((h, w), dtype=torch.int32, device="cuda")
    for k in range(3):
        s0, s1 = multi.sample_range(spp, k, 3)
        renderer.render_samples(cam, w, h, spp, s0, s1, jitter=True)
        renderer.sync()
        counts += multi.framebuffer_tensor(renderer)
        torch.cuda.synchronize()
    multi.framebuffer_tensor(renderer).copy_(counts)
    torch.cuda.synchronize()
    np.testing.assert_array_equal(renderer.framebuffer_resolve(spp).framebuffer(), fb0)
    for count in (2, 4):
        counts.zero_()
        for k in range(count):
            renderer.render_interleaved(cam, w, h, spp, k, count, jitter=True)
            renderer.sync()
            counts += multi.framebuffer_tensor(renderer)
            torch.cuda.synchronize()
        multi.framebuffer_tensor(renderer).copy_(counts)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(renderer.framebuffer_resolve(spp).framebuffer(), fb0)
