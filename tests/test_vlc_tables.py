"""Pin tools/vlc_tables.py (ISO 11172-2 Annex B form) to the reference's tree tables.

tools/make_reference_golden.py walks the reference's trees (src/wasm/mpeg1.c:59-680 == src/mpeg1.js:1037-1663) the
way read_huffman does (src/wasm/mpeg1.c:1742-1748) and records in tests/golden/reference/vlc_trees.json every code
that reaches a leaf, with the leaf's value, and the reference's constant matrices.
"""
import pytest

import helpers
import vlc_tables as V


@pytest.mark.parametrize("name", sorted(V.ALL_VLC))
def test_prefix_free(name):
    V.check_prefix_free(V.ALL_VLC[name])


@pytest.mark.parametrize("name", sorted(V.ALL_VLC))
def test_codes_match_reference_trees(name):
    tree = helpers.reference_golden("vlc_trees")["trees"][name]
    table = V.ALL_VLC[name]
    for code, value in table.items():
        assert tree["codes"].get(code) == value, (name, code, tree["codes"].get(code), value)
    # same number of leaves => the tables are the same function on all valid codes
    assert tree["leaves"] == len(tree["codes"]) == len(table), (name, tree["leaves"], len(table))


def test_constant_matrices_match_reference():
    ref = helpers.reference_golden("vlc_trees")["matrices"]
    assert ref["ZIG_ZAG"] == V.ZIG_ZAG
    assert ref["DEFAULT_INTRA_QUANT_MATRIX"] == V.DEFAULT_INTRA_QUANT_MATRIX
    assert ref["DEFAULT_NON_INTRA_QUANT_MATRIX"] == V.DEFAULT_NON_INTRA_QUANT_MATRIX
    assert ref["PREMULTIPLIER_MATRIX"] == V.PREMULTIPLIER_MATRIX
    assert [round(x, 3) for x in ref["PICTURE_RATE"]] == [round(x, 3) for x in V.PICTURE_RATE]


def test_run_level_table_size():
    assert len(V.DCT_RUN_LEVEL_CODE) == 111  # ISO 11172-2 table B.5c-g
    assert sorted(V.ZIG_ZAG) == list(range(64))
