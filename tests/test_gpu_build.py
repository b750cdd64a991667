"""GPU BIH build vs the oracle: every array of the reference's data model, bit for bit, through the C ABI."""
import json
import os

import numpy as np
import pytest

from conftest import assert_view_equals_oracle
from test_oracle_kat import GOLD, check_against_golden

pytestmark = pytest.mark.gpu


def build_view(renderer, tri):
    renderer.load_models(tri).build()
    return renderer.reference_view()


def test_kat_dodecahedron_matches_reference_dump(renderer, scenes, oracle):
    v = build_view(renderer, scenes.dodecahedron(True))
    gold = json.load(open(GOLD))
    check_against_golden(v["children"], v["is_leaf"], v["axis"], v["parent"], v["clip_planes"], gold["nodes"])
    assert_view_equals_oracle(v, oracle.Bih(scenes.dodecahedron(True)))


@pytest.mark.parametrize("name", ["cornell", "sphere16", "sphere187", "atrium", "soup", "duplicates", "flat", "sphere361"])
def test_build_bit_exact(renderer, scenes, oracle, name):
    tri = {
        "cornell": lambda: scenes.cornell_box(),
        "sphere16": lambda: scenes.displaced_sphere(16),
        "sphere187": lambda: scenes.displaced_sphere(187),
        "sphere361": lambda: scenes.displaced_sphere(361),
        "atrium": lambda: scenes.atrium(),
        "soup": lambda: scenes.random_soup(100000),
        "duplicates": lambda: np.repeat(scenes.dodecahedron(), 5, axis=0),
        "flat": lambda: scenes.quad_grid([0, 0, 0], [1, 0, 0], [0, 1, 0], 40, 30),
    }[name]()
    assert_view_equals_oracle(build_view(renderer, tri), oracle.Bih(tri))


@pytest.mark.parametrize("n", [1, 2, 3, 31, 32, 33, 255, 256, 257, 4095, 4096, 4097, 8193])
def test_ragged_sizes(renderer, scenes, oracle, n):
    tri = scenes.random_soup(n, size=0.1, seed=n)
    assert_view_equals_oracle(build_view(renderer, tri), oracle.Bih(tri))


def test_single_cell_and_empty(renderer, oracle):
    same = np.tile(np.array([[0, 0, 0, 1, 0, 0, 0, 1, 0]], np.float32), (7, 1))
    v = build_view(renderer, same)
    assert v["nu"] == 1 and v["n"] == 7 and len(v["axis"]) == 0
    assert_view_equals_oracle(v, oracle.Bih(same))
    renderer.load_models(np.zeros((0, 9), np.float32)).build()
    assert renderer.build_info()["nu"] == 0


def test_rebuild_is_idempotent_and_update_vertices(renderer, scenes, oracle):
    a, b = scenes.displaced_sphere(64, phase=0.0), scenes.displaced_sphere(64, phase=0.7)
    renderer.load_models(a).build()
    v1 = renderer.reference_view()
    renderer.build()
    v2 = renderer.reference_view()
    for k in ("morton_codes", "tris_indexes", "children", "clip_planes", "parent"):
        np.testing.assert_array_equal(v1[k], v2[k])
    renderer.update_vertices(b)
    renderer.build()                       # animation: clip planes must be rebuilt from scratch (SURVEY 0.9)
    assert_view_equals_oracle(renderer.reference_view(), oracle.Bih(b))


def test_device_pointer_input(renderer, scenes, oracle):
    import torch
    tri = scenes.displaced_sphere(48)
    d = torch.from_numpy(tri).cuda()
    renderer.load_models(d).build()
    assert_view_equals_oracle(renderer.reference_view(), oracle.Bih(tri))


def test_one_million_triangles(renderer, scenes, oracle):
    """BASELINE config 5 size: full comparison with the oracle (the CPU build takes < 1 s) plus the
    size-independent properties: sortedness, permutation, run structure, tree shape."""
    tri = scenes.displaced_sphere(708)
    v = build_view(renderer, tri)
    n, nu = v["n"], v["nu"]
    assert n == 1002528
    codes = v["morton_codes"]
    assert np.all(codes[1:] >= codes[:-1])
    assert np.array_equal(np.sort(v["tris_indexes"]), np.arange(n, dtype=np.uint32))
    eq = codes[1:] == codes[:-1]                      # stable: equal codes keep input order
    assert np.all(v["tris_indexes"][1:][eq] > v["tris_indexes"][:-1][eq])
    assert v["duplicates_cnts"].sum() == n and np.all(np.diff(v["unique_morton_codes"].astype(np.int64)) > 0)
    ch, lf = v["children"], v["is_leaf"]
    assert np.all(ch[:, 1] == ch[:, 0] + 1)
    assert lf.sum() == nu and (~lf.astype(bool)).sum() == nu - 2     # every leaf / non-root node has one parent
    assert_view_equals_oracle(v, oracle.Bih(tri))


def test_obj_loader(renderer, scenes, oracle, tmp_path):
    tri = scenes.dodecahedron()
    p = tmp_path / "d.obj"
    with open(p, "w") as f:
        f.write("# test\n")
        for t in tri.reshape(-1, 3):
            f.write("v %.9g %.9g %.9g\n" % tuple(t))
        for i in range(len(tri)):
            f.write("f %d/1/1 %d//2 %d\n" % (3 * i + 1, 3 * i + 2, 3 * i + 3))
        f.write("v 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nf -4 -3 -2 -1\n")     # quad -> fan of 2
    renderer.load_models(str(p)).build()
    quad = np.array([[0, 0, 0, 1, 0, 0, 1, 1, 0], [0, 0, 0, 1, 1, 0, 0, 1, 0]], np.float32)
    assert_view_equals_oracle(renderer.reference_view(), oracle.Bih(np.concatenate([tri, quad])))


def test_error_codes(renderer):
    import bihrt
    with pytest.raises(bihrt.BihrtError) as e:
        renderer.build()
    assert e.value.code == -4
    with pytest.raises(bihrt.BihrtError) as e:
        renderer.load_models("/nonexistent/file.obj")
    assert e.value.code == -5
    # retired trace-scheduling options are unknown names now (BIHRT_ERR_INVALID)
    for name in ("trace_refill_threshold", "trace_refill_incoherent", "trace_chunk_items", "trace_vote_wait", "trace_vote_walk"):
        with pytest.raises(bihrt.BihrtError) as e:
            renderer.set_option(name, 32)
        assert e.value.code == -1 and "unknown option" in str(e.value)


def test_refit_keeps_hits_correct(renderer, scenes, oracle):
    """bihrt_refit (non-parity fast path for animation): topology of the last build, new clip planes.  The
    BIH must stay valid: hits on the moved mesh equal brute force over the moved triangles."""
    import bihrt
    a, b = scenes.displaced_sphere(96, phase=0.0), scenes.displaced_sphere(96, phase=0.15)
    with pytest.raises(bihrt.BihrtError):
        renderer.load_models(a).refit()                 # needs a full build first
    renderer.build()
    topo = renderer.reference_view()["children"].copy()
    renderer.update_vertices(b)
    renderer.refit()
    v = renderer.reference_view()
    np.testing.assert_array_equal(v["children"], topo)                      # same topology ...
    rays = oracle.camera_rays(scenes.pinhole_camera(), 320, 180)
    t, s, p = renderer.trace(rays)
    # ... but bounds of the moved geometry: compare with brute force on the moved mesh, by primitive id
    ob = oracle.Bih(b)
    tb, sb, pb = ob.trace(rays, "brute")
    np.testing.assert_array_equal(p, pb)
    np.testing.assert_array_equal(t, tb)
    renderer.build()                                                        # a full rebuild is the parity path again
    from conftest import assert_view_equals_oracle
    assert_view_equals_oracle(renderer.reference_view(), ob)


@pytest.mark.parametrize("name", ["cornell", "sphere187", "atrium", "duplicates", "flat", "soup8193", "single", "two"])
def test_rebuild_and_refit_reproduce_the_blob(renderer, scenes, oracle, name):
    """The whole blob (header, 64-byte nodes with the children boxes, triangle records) is a function of the triangles alone:
    a second build over the scratch of the first and a refit of unmoved vertices rewrite it byte for byte."""
    tri = {
        "cornell": lambda: scenes.cornell_box(),
        "sphere187": lambda: scenes.displaced_sphere(187),
        "atrium": lambda: scenes.atrium(),
        "duplicates": lambda: np.repeat(scenes.dodecahedron(), 5, axis=0),
        "flat": lambda: scenes.quad_grid([0, 0, 0], [1, 0, 0], [0, 1, 0], 40, 30),
        "soup8193": lambda: scenes.random_soup(8193, size=0.1, seed=5),
        "single": lambda: np.tile(np.array([[0, 0, 0, 1, 0, 0, 0, 1, 0]], np.float32), (7, 1)),
        "two": lambda: scenes.random_soup(2, size=0.1, seed=2),
    }[name]()
    import torch
    from bihrt import multi

    def blob():
        ptr, nbytes = renderer.bih_region(len(tri))
        renderer.sync()
        return torch.as_tensor(multi._CudaView(ptr, (nbytes,), "|u1"), device="cuda:%d" % renderer.device).cpu().numpy()

    renderer.load_models(tri).build()
    assert_view_equals_oracle(renderer.reference_view(), oracle.Bih(tri))
    blob_ref = blob()
    renderer.build()
    assert_view_equals_oracle(renderer.reference_view(), oracle.Bih(tri))
    assert np.array_equal(blob(), blob_ref)
    renderer.refit()
    assert np.array_equal(blob(), blob_ref)


def test_builds_alternate_cleanly_between_parity_quality_and_refit(renderer, scenes, oracle):
    """k_front alternates between two scene-box accumulators (nothing is cleared before a build); the quality mode and the
    refit use a third one.  Any interleaving must give the reference's tree again, on a scene whose box CHANGES between builds."""
    a, b = scenes.displaced_sphere(48, phase=0.0), scenes.displaced_sphere(48, phase=0.9) * np.float32(1.7)
    oa, ob = oracle.Bih(a), oracle.Bih(b)
    renderer.load_models(a).build()
    assert_view_equals_oracle(renderer.reference_view(), oa)
    try:
        renderer.set_option("morton_bits", 63)
        renderer.build()                                    # quality build of a (own accumulator)
        renderer.set_option("morton_bits", 30)
        renderer.update_vertices(b)
        renderer.build()                                    # parity build of the larger scene
        assert_view_equals_oracle(renderer.reference_view(), ob)
        renderer.update_vertices(a)
        renderer.refit()                                    # refit back to a (non-parity tree, own accumulator) ...
        renderer.build()                                    # ... and two parity builds in a row
        assert_view_equals_oracle(renderer.reference_view(), oa)
        renderer.update_vertices(b)
        renderer.build()
        assert_view_equals_oracle(renderer.reference_view(), ob)
    finally:
        renderer.set_option("morton_bits", 30)
