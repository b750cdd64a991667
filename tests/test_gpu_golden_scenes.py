"""Pins the CPU oracle -- and through it the library -- to stored outputs on six scenes.

tests/golden/golden_scenes.json holds SHA-256 digests of every input and output of the oracle on these scenes: the
triangles, the camera rays, the BIH arrays of the reference's model (sorted codes, trisIndexes, uniqueMortonCodes,
duplicatesCnts, firstIdxs, children / isLeaf / axis / parent / clipPlanes, leafParents) and the literal TraverseTree
results (t, slot) of every ray.  These are the scenes on which the oracle was compared with the original project's own
CUDA kernels (oracle/ref_harness.cu) while those could be built: build arrays bit for bit, ids except the documented
edge ties, t within 1e-5 (DESIGN.md section 6).  The digests freeze the oracle, so a later change to the oracle,
the scene generators or the camera shows up here even when every library-vs-oracle test still agrees.  The library
is then held to the pinned oracle with the tolerances of that comparison.

Regenerate (CPU only, after a deliberate change of the oracle's results):  python tests/test_gpu_golden_scenes.py
"""
import hashlib
import json
import os
import sys

import numpy as np
import pytest

from conftest import assert_view_equals_oracle

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_scenes.json")
ID_MISMATCH_MAX = 1e-4      # ids exact except documented ties
T_REL_TOL = 1e-5

SCENES = {
    "dodecahedron": lambda S: (S.dodecahedron(), S.pinhole_camera(aspect=1.0), 128, 128),
    "cornell": lambda S: (S.cornell_box(), S.cornell_camera(), 256, 256),
    "sphere187": lambda S: (S.displaced_sphere(187), S.pinhole_camera(), 640, 360),
    "sphere361": lambda S: (S.displaced_sphere(361), S.pinhole_camera(), 320, 180),
    "atrium": lambda S: (S.atrium(0.3), S.atrium_camera(), 320, 180),
    "soup": lambda S: (S.random_soup(50000), S.pinhole_camera(), 320, 180),
}
BUILD = ("codes", "tris_idx", "umc", "cnt", "first", "children", "is_leaf", "axis", "parent", "leaf_parents", "clip")


def digest(a):
    a = np.ascontiguousarray(a)
    return "%s%s:%s" % (a.dtype.str, list(a.shape), hashlib.sha256(a.tobytes()).hexdigest())


def oracle_record(O, S, name):
    """Digests of the scene's inputs and of the oracle's build and trace; also returns what the test needs."""
    tri, cam, w, h = SCENES[name](S)
    ob = O.Bih(tri)
    rays = O.camera_rays(cam, w, h)
    t, slot, _ = ob.trace(rays, "ref")
    rec = {"triangles": digest(tri), "n": int(ob.n), "nu": int(ob.nu), "rays": digest(rays),
           "build": {k: digest(getattr(ob, k)) for k in BUILD}, "t": digest(t), "slot": digest(slot)}
    return rec, tri, ob, rays, t, slot


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCENES))
def test_oracle_and_library_match_stored_outputs(renderer, scenes, oracle, name):
    want = json.load(open(GOLD))["scenes"][name]
    got, tri, ob, rays, t0, s0 = oracle_record(oracle, scenes, name)
    # inputs first, so that a failure names the stage that moved
    for k in ("triangles", "rays", "n", "nu"):
        assert got[k] == want[k], k
    for k in BUILD:
        assert got["build"][k] == want["build"][k], "oracle build array %s differs from the stored one" % k
    assert got["slot"] == want["slot"] and got["t"] == want["t"], "oracle trace differs from the stored one"
    # the library against the pinned oracle: build bit for bit, trace within the tolerances above
    renderer.load_models(tri).build()
    assert_view_equals_oracle(renderer.reference_view(), ob)
    t, s, _ = renderer.trace(rays)
    bad = s != s0
    assert bad.sum() <= ID_MISMATCH_MAX * len(rays), "%d of %d ids differ from the stored trace" % (bad.sum(), len(rays))
    hit = ~bad & (s0 >= 0)
    np.testing.assert_allclose(t[hit], t0[hit], rtol=T_REL_TOL, atol=0)


if __name__ == "__main__":
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path[:0] = [root, os.path.join(root, "bih-gpu-raytracer_b200")]
    from bihrt import scenes as S
    from oracle import oracle as O
    out = {"what": "SHA-256 digests (dtype, shape, bytes) of the oracle's inputs and outputs on each scene; "
                   "written by tests/test_gpu_golden_scenes.py",
           "scenes": {nm: oracle_record(O, S, nm)[0] for nm in SCENES}}
    with open(GOLD, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("wrote", GOLD)
