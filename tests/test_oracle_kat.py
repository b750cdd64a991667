"""The oracle against the reference's only pinned result (SURVEY.md Appendix A, R/BIH1.txt)."""
import json
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(__file__), "golden", "dodecahedron_bih.json")

# SURVEY.md Appendix A: expected sorted order as (input triangle id, Morton code)
EXPECTED_SORTED = [
    (5, 0x035e8017), (4, 0x03c84932), (0, 0x0544a491), (8, 0x069d8027), (7, 0x06b0126c), (9, 0x0a7a125e),
    (10, 0x0bc84932), (1, 0x0c402490), (2, 0x0c6036d8), (14, 0x0f168005), (3, 0x11c06db0), (20, 0x1632124c),
    (17, 0x170d8003), (11, 0x19c06db0), (16, 0x1e090002), (15, 0x1e29124a), (21, 0x1f168005), (6, 0x22a05b68),
    (26, 0x2544a491), (28, 0x275a0016), (27, 0x27ccc933), (13, 0x2b048001), (12, 0x2b84c921), (25, 0x2c402490),
    (24, 0x2c6036d8), (32, 0x2ee85b7a), (31, 0x2f5a0016), (19, 0x32201248), (18, 0x32a05b68), (29, 0x35522494),
    (33, 0x370d8003), (22, 0x3b048001), (23, 0x3b84c921), (30, 0x3d522494), (34, 0x3e090002), (35, 0x3e29124a)]


def check_against_golden(children, is_leaf, axis, parent, clip, nodes):
    assert len(nodes) == 35 and len(axis) == 35
    for nd in nodes:
        i = nd["node"]
        assert parent[i] == nd["parent"], i
        assert list(children[i]) == nd["children"], i
        assert axis[i] == nd["axis"], i
        assert [bool(x) for x in is_leaf[i]] == nd["is_leaf"], i
        # the dump prints 6 significant digits
        assert abs(float(clip[i][0]) - nd["clip"][0]) <= 2e-6, i
        assert abs(float(clip[i][1]) - nd["clip"][1]) <= 2e-6, i


@pytest.mark.parametrize("rounded", [True, False])
def test_oracle_reproduces_reference_tree_dump(oracle, scenes, rounded):
    gold = json.load(open(GOLD))
    b = oracle.Bih(scenes.dodecahedron(rounded))
    assert b.nu == 36
    check_against_golden(b.children, b.is_leaf, b.axis, b.parent, b.clip, gold["nodes"])


def test_oracle_sorted_codes_match_appendix_a(oracle, scenes):
    b = oracle.Bih(scenes.dodecahedron(True))
    assert [(int(i), int(c)) for i, c in zip(b.tris_idx, b.codes)] == EXPECTED_SORTED
    assert np.all(b.cnt == 1) and np.array_equal(b.first, np.arange(36))

