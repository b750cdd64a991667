"""Framebuffer renders walk in the copy of the node phase that matches the warp's ray octant (csrc/trace.cu, OCTS).

A warp whose live lanes agree on the sign of 1/d on every axis takes each box's near and far planes by compile-time sign;
a warp that mixes signs takes the generic copy.  Every case below must give the image of the closest-hit oracle bit for
bit, and render_counted (which runs the same copies) must visit exactly the nodes and triangles of the coverage
restatement, exit "first" of tests/walk_oracle.c:
  * views from the 8 diagonal directions, so that every octant copy runs;
  * the config-2 camera at sizes where the centre row and column, whose rays change sign, fall inside warps, at 1, 4 and
    16 spp, with and without jitter, for several lane groupings (1 spp launches also refill warps partially);
  * a camera whose centre pixel column has dx == 0 exactly: a zero component in an otherwise uniform warp;
  * cameras inside the atrium, where warps of many octants and mixed warps meet.
"""
import itertools

import numpy as np
import pytest

from walk_oracle import tree  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu


def check_frame(renderer, oracle, tree, cam, w, h, spp, jitter, groups=(-1,)):  # noqa: F811
    """The renderer's tree is `tree` (a walk_oracle.Tree): the image is held to its closest walk and render_counted to its
    'first' walk."""
    rays = oracle.camera_rays(cam, w, h, spp=spp, jitter=jitter, seed=1984)
    s0 = tree.walk(rays)["slot"]
    exp = oracle.pack_framebuffer(s0, w, h, spp).reshape(h, w)
    what = "%dx%d spp %d jitter %s" % (w, h, spp, jitter)
    try:
        for g in groups:
            renderer.set_option("trace_lane_groups", g)
            fb = renderer.render(cam, w, h, spp=spp, seed=1984, jitter=jitter).framebuffer()
            np.testing.assert_array_equal(fb, exp, err_msg="%s groups %d" % (what, g))
    finally:
        renderer.set_option("trace_lane_groups", -1)
    cf = tree.walk(rays, "first")["counters"]
    cnt = renderer.render_counted(cam, w, h, spp=spp, seed=1984, jitter=jitter)
    assert cnt["rays"] == len(rays)
    assert (cnt["nodes"], cnt["tris"], cnt["max_stack"]) == (cf["nodes"], cf["tris"], cf["max_stack"]), what
    return rays, s0


def check_parity_frame(renderer, oracle, tree, tri, cam, w, h, spp, jitter, groups=(-1,)):  # noqa: F811
    """check_frame on the parity tree of `tri`, whose closest walk hits exactly where the reference's traversal ('ref') hits:
    the image is the reference's."""
    ob = oracle.Bih(tri)
    rays, s0 = check_frame(renderer, oracle, tree(ob), cam, w, h, spp, jitter, groups)
    np.testing.assert_array_equal(s0 >= 0, ob.trace(rays, "ref")[1] >= 0)
    return rays, s0


@pytest.mark.parametrize("signs", list(itertools.product((1, -1), repeat=3)))
def test_diagonal_views(renderer, scenes, oracle, tree, signs):  # noqa: F811
    """The sphere seen from (+-1, +-1, +-1): nearly every ray lies in the octant opposite the eye."""
    tri = scenes.displaced_sphere(187)
    renderer.load_models(tri).build()
    s = np.array(signs, np.float64)
    cam = scenes.look_at_camera(2.2 * s + np.array([0.05, 0.03, 0.0]), (0.0, 0.0, 0.0), 0.3, 1.5)
    for spp, jitter in ((1, False), (4, True), (16, True)):
        rays, s0 = check_parity_frame(renderer, oracle, tree, tri, cam, 120, 80, spp, jitter)
        assert (np.sign(rays[:, 3:]) == -s).all(axis=1).mean() > 0.95
        assert 0.2 < (s0 >= 0).mean() < 0.9


@pytest.mark.parametrize("w,h", [(97, 65), (160, 90), (75, 41)])
def test_sign_changes_inside_warps(renderer, scenes, oracle, tree, w, h):  # noqa: F811
    """Config-2 camera looking along +z: dx and dy change sign on the centre column and row of the frame."""
    tri = scenes.displaced_sphere(187)
    renderer.load_models(tri).build()
    cam = scenes.pinhole_camera(aspect=w / h)
    for spp in (1, 4, 16):
        for jitter in (False, True):
            rays, _ = check_parity_frame(renderer, oracle, tree, tri, cam, w, h, spp, jitter, groups=(-1, 1, 2))
            assert (rays[:, 3] < 0).any() and (rays[:, 3] > 0).any() and (rays[:, 4] < 0).any() and (rays[:, 4] > 0).any()


def test_zero_direction_component_in_a_uniform_warp(renderer, scenes, oracle, tree):  # noqa: F811
    """Pixel centres of column 48 of a 97-pixel-wide frame have dx == 0 exactly (origin x = 0, llc x = -0.5, horizontal
    x = 1): at 16 spp a warp holds pixels 48 and 49, one with dx == 0 and one with dx > 0."""
    tri = scenes.displaced_sphere(187)
    renderer.load_models(tri).build()
    w, h = 97, 64
    cam = scenes.pinhole_camera(origin=(0.0, 0.2, -3.0), half=0.5, aspect=1.0)
    for spp in (1, 16):
        rays, s0 = check_parity_frame(renderer, oracle, tree, tri, cam, w, h, spp, False, groups=(-1, 1))
        zero = rays[:, 3] == 0
        assert zero.sum() == h * spp and (s0[zero] >= 0).any()


@pytest.mark.parametrize("view", ["atrium_camera", "diagonal_down", "diagonal_up_back"])
def test_camera_inside_the_atrium(renderer, scenes, oracle, tree, view):  # noqa: F811
    tri = scenes.atrium(0.2)
    renderer.load_models(tri).build()
    cam = {"atrium_camera": lambda: scenes.atrium_camera(160 / 90),
           "diagonal_down": lambda: scenes.look_at_camera((-1.2, 0.3, 0.4), (0.0, -0.5, -0.4), 0.6, 160 / 90),
           "diagonal_up_back": lambda: scenes.look_at_camera((1.0, -0.4, 0.3), (-0.2, 0.4, 1.2), 0.6, 160 / 90)}[view]()
    for spp, jitter in ((1, False), (4, True), (16, False)):
        _, s0 = check_parity_frame(renderer, oracle, tree, tri, cam, 160, 90, spp, jitter, groups=(-1, 1))
        assert (s0 >= 0).mean() > 0.5
