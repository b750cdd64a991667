"""Camera launches that take their units from the global counter a batch at a time: lane j of the warp resolves unit j of
the batch, the units with a pixel in the frame are traced lowest first, a batch of padding units only is skipped, and
the warp leaves at the first batch whose first unit is past the end.

The tile order is off (`trace_tile_order` 0), which puts every launch here on the batch path; the same frame rendered
with the tile order on (2: every launch of more than one tile measures tile costs) takes one unit per fetch.  Both must
equal the oracle's frame bit for bit.  The shapes: frames of fewer units than a batch, unit counts that are not a
multiple of it, edge tiles whose bottom rows make batches of padding only, 1 to 96 samples per pixel (several samples
per lane from 64 on), sample ranges, unit interleave across 2 and 4 ranks, per-sample records (render_hits) and a frame
rendered twice."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

BATCH_PATH, UNIT_PATH = 0, 2          # trace_tile_order: off (batches of units) / every launch cost-ordered (one unit)


@pytest.fixture(scope="module")
def scene(scenes, oracle):
    tri = scenes.displaced_sphere(96)
    return tri, oracle.Bih(tri)


def expected(oracle, ob, cam, w, h, spp, jitter, seed=1984):
    rays = oracle.camera_rays(cam, w, h, spp=spp, jitter=jitter, seed=seed)
    t, s, p = ob.trace(rays, "box")
    return t, s, p, oracle.pack_framebuffer(s, w, h, spp).reshape(h, w)


def on_both_paths(renderer, draw):
    """draw() on the batch path, then on the one-unit path."""
    out = []
    for order in (BATCH_PATH, UNIT_PATH):
        renderer.set_option("trace_tile_order", order)
        out.append(draw())
    return out


# (w, h, spp): a single pixel (one unit in the frame), frames of a few units, unit counts that are not a multiple of a
# batch, edge tiles of padding rows (33 x 5: the second tile holds one column), and several samples per lane
FRAMES = [(1, 1, 1), (1, 1, 16), (3, 2, 4), (9, 5, 1), (17, 9, 1), (33, 5, 1), (33, 5, 4), (33, 5, 16), (33, 5, 64),
          (65, 37, 1), (47, 29, 12), (39, 21, 16), (70, 40, 16), (29, 19, 64), (21, 13, 96)]


@pytest.mark.parametrize("w,h,spp", FRAMES)
def test_batched_frames_match_oracle_and_unit_path(renderer, scenes, oracle, scene, w, h, spp):
    tri, ob = scene
    renderer.load_models(tri).build()
    cam = scenes.pinhole_camera(aspect=w / h)
    jitter = spp > 1
    fb0 = expected(oracle, ob, cam, w, h, spp, jitter)[3]
    fbs = on_both_paths(renderer, lambda: renderer.render(cam, w, h, spp=spp, jitter=jitter).framebuffer().copy())
    for fb in fbs:
        np.testing.assert_array_equal(fb, fb0)


@pytest.mark.parametrize("w,h,spp", [(33, 5, 1), (17, 9, 16), (29, 19, 64)])
def test_batched_render_hits_match_oracle(renderer, scenes, oracle, scene, w, h, spp):
    """Per-sample records (MODE 2) on both paths equal the oracle's walk."""
    tri, ob = scene
    renderer.load_models(tri).build()
    cam = scenes.pinhole_camera(aspect=w / h)
    t0, s0, p0, _ = expected(oracle, ob, cam, w, h, spp, spp > 1)
    for t, s, p in on_both_paths(renderer, lambda: renderer.render_hits(cam, w, h, spp=spp, jitter=spp > 1)):
        np.testing.assert_array_equal(s, s0)
        np.testing.assert_array_equal(p, p0)
        np.testing.assert_array_equal(t, t0)


def test_batched_frame_twice(renderer, scenes, oracle, scene):
    """Two launches in a row on the batch path draw the same frame (the counter of batches starts again at 0)."""
    tri, ob = scene
    renderer.load_models(tri).build()
    renderer.set_option("trace_tile_order", BATCH_PATH)
    for w, h, spp in ((45, 19, 16), (33, 5, 1)):
        cam = scenes.pinhole_camera(aspect=w / h)
        fb0 = expected(oracle, ob, cam, w, h, spp, spp > 1)[3]
        for _ in range(2):
            np.testing.assert_array_equal(renderer.render(cam, w, h, spp=spp, jitter=spp > 1).framebuffer(), fb0)


@pytest.mark.parametrize("w,h,spp", [(33, 5, 16), (75, 41, 4), (75, 41, 64)])
def test_batched_count_paths(renderer, scenes, oracle, scene, w, h, spp):
    """Hit counts of sample ranges and of units interleaved over 2 and 4 ranks, summed and resolved, equal the oracle's
    frame on both paths."""
    import torch
    from bihrt import multi
    tri, ob = scene
    renderer.load_models(tri).build()
    cam = scenes.pinhole_camera(aspect=w / h)
    fb0 = expected(oracle, ob, cam, w, h, spp, True)[3]

    def resolved(launches):
        counts = torch.zeros((h, w), dtype=torch.int32, device="cuda")
        for launch in launches:
            launch()
            renderer.sync()
            counts += multi.framebuffer_tensor(renderer)
            torch.cuda.synchronize()
        multi.framebuffer_tensor(renderer).copy_(counts)
        torch.cuda.synchronize()
        return renderer.framebuffer_resolve(spp).framebuffer().copy()

    def ranges():
        return resolved([lambda k=k: renderer.render_samples(cam, w, h, spp, *multi.sample_range(spp, k, 3), jitter=True)
                         for k in range(3)])

    def interleaved(count):
        return resolved([lambda k=k: renderer.render_interleaved(cam, w, h, spp, k, count, jitter=True) for k in range(count)])

    for draw in (ranges, lambda: interleaved(2), lambda: interleaved(4)):
        for fb in on_both_paths(renderer, draw):
            np.testing.assert_array_equal(fb, fb0)
