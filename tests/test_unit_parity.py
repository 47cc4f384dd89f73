"""Per-function parity of the oracle against the reference (SURVEY section 4): the reference's helper functions
are non-static (prototypes src/wasm/mpeg1.c:754-769), so tools/make_reference_golden.py calls its idct() directly
on the blocks below and records the results in tests/golden/reference/idct.json."""
import ctypes

import numpy as np

import helpers

COEF_MIN, COEF_MAX = -2048 * 62, 2047 * 62  # the full premultiplied coefficient range


def random_blocks(n=1200, seed=11):
    """Seeded random blocks: a quarter each over the full range and over the smaller magnitudes real streams give."""
    rng = np.random.default_rng(seed)
    scale = np.array([COEF_MAX, 2047, 255, 16])[np.arange(n) % 4, None]
    return np.clip(rng.integers(-scale, scale + 1, (n, 64)), COEF_MIN, COEF_MAX).astype(np.int32)


def sparse_and_extreme_blocks():
    rng = np.random.default_rng(0)
    cases = [[0] * 64, [255 << 8] + [0] * 63, [COEF_MIN] * 64, [COEF_MAX] * 64]
    for _ in range(200):
        blk = [0] * 64
        for i in rng.integers(0, 64, rng.integers(1, 6)):
            blk[int(i)] = int(rng.integers(COEF_MIN, COEF_MAX + 1))
        cases.append(blk)
    return np.array(cases, dtype=np.int32)


def idct_digests(idct, blocks):
    """digest of each block after idct (a ctypes function transforming 64 ints in place)."""
    out = []
    for blk in blocks:
        a = (ctypes.c_int * 64)(*blk.tolist())
        idct(a)
        out.append(helpers.digest(np.array(a, dtype=np.int32)))
    return out


def _check(kind, blocks):
    want = helpers.reference_golden("idct")[kind]
    assert helpers.digest(blocks) == want["inputs"], f"{kind}: the blocks are not the ones the reference transformed"
    got = idct_digests(helpers.oracle_lib().oracle_idct, blocks)
    bad = [k for k, (g, w) in enumerate(zip(got, want["outputs"])) if g != w]
    assert len(got) == len(want["outputs"]) and not bad, f"{kind}: {len(bad)} blocks differ, first {bad[:8]}"


def test_idct_matches_reference_on_random_blocks():
    """src/mpeg1.js:916-983 / src/wasm/mpeg1.c:1673-1740 on the full premultiplied coefficient range."""
    _check("random", random_blocks())


def test_idct_matches_reference_on_sparse_and_extreme_blocks():
    _check("sparse_and_extreme", sparse_and_extreme_blocks())


def vlc_trie_stream():
    import synth_es
    k = synth_es.Knobs(width=16, height=16, pictures=40, gop=1, slices="one", escape_prob=0.5, big_escape_prob=0.5,
                       max_coefs=30, dc_only_prob=0.05)
    return synth_es.SynthStream(k, 4242).generate()


def test_vlc_trie_matches_reference_read_huffman_on_random_bits():
    """Whole-stream comparisons already exercise the VLC paths; here the DCT coefficient table is
    hit with uniformly random bits through both decoders' block parsers by wrapping them in minimal
    one-macroblock intra pictures (every escape / long-code branch gets visited)."""
    es = vlc_trie_stream()
    orc_frames, orc_idx, od = helpers.decode_all(helpers.oracle_lib(), [(0.0, es)])
    assert len(orc_frames) == 40
    helpers.assert_matches_reference("vlc_trie", orc_frames, orc_idx, es)
    od.destroy()
