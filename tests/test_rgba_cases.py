"""SURVEY 8f rank 2 (planar -> RGBA, src/canvas2d.js:53-122) pinned to the TEXT of the reference: colours worked
out BY HAND from the JS statements, fed through the decoder as flat blocks.

An intra block whose only coefficient is its DC reconstructs to 64 samples of exactly the DC predictor value
(mpeg1.js:747 `blockData[0] <<= 8`, :838-841 `(blockData[0] + 128) >> 8`), so an I picture of DC-only blocks is a
picture of chosen (Y, Cb, Cr) triples: one colour per 8 x 8 luma block, Cb / Cr per macroblock.

canvas2d.js:85-91 (its `ccb` is the SECOND argument of render(), which the decoder fills with the Cr plane --
mpeg1.js:217 calls render(Y, Cr, Cb); SURVEY Q8 -- so below cr is the Cr-plane sample):
    r = (cr + ((cr * 103) >> 8)) - 179
    g = ((cb * 88) >> 8) - 44 + ((cr * 183) >> 8) - 91
    b = (cb + ((cb * 198) >> 8)) - 227
    R = clamp(Y + r)   G = clamp(Y - g)   B = clamp(Y + b)   A = 255      (Uint8ClampedArray, canvas2d.js:93-110)
"""
import os
import sys

import numpy as np
import pytest

import helpers

sys.path.insert(0, os.path.join(helpers.ROOT, "tools"))

# (Y, Cb, Cr) -> (R, G, B), each line worked out by hand from the statements above
HAND = [
    # grey: cr = cb = 128: r = 128 + (13184 >> 8 = 51) - 179 = 0; g = (11264 >> 8 = 44) - 44 + (23424 >> 8 = 91) - 91 = 0;
    #       b = 128 + (25344 >> 8 = 99) - 227 = 0
    ((128, 128, 128), (128, 128, 128)),
    ((16, 128, 128), (16, 16, 16)),
    ((235, 128, 128), (235, 235, 235)),
    # red-ish: cr = 240: r = 240 + (24720 >> 8 = 96) - 179 = 157; cb = 90: g = (7920 >> 8 = 30) - 44 + (43920 >> 8 = 171) - 91 = 66;
    #          b = 90 + (17820 >> 8 = 69) - 227 = -68.  Y = 81: R = 238, G = 81 - 66 = 15, B = 13
    ((81, 90, 240), (238, 15, 13)),
    # blue-ish: cb = 240: b = 240 + (47520 >> 8 = 185) - 227 = 198; cr = 110: r = 110 + (11330 >> 8 = 44) - 179 = -25;
    #           g = (21120 >> 8 = 82) - 44 + (20130 >> 8 = 78) - 91 = 25.  Y = 41: R = 16, G = 16, B = 239
    ((41, 240, 110), (16, 16, 239)),
    # clamping at both ends: cr = 255: r = 255 + (26265 >> 8 = 102) - 179 = 178; cb = 0: g = 0 - 44 + (46665 >> 8 = 182) - 91 = 47;
    #                        b = 0 + 0 - 227 = -227.  Y = 200: R = 378 -> 255, G = 153, B = -27 -> 0
    ((200, 0, 255), (255, 153, 0)),
    # cr = 0: r = 0 + 0 - 179 = -179; cb = 255: g = (22440 >> 8 = 87) - 44 + 0 - 91 = -48; b = 255 + (50490 >> 8 = 197) - 227 = 225.
    # Y = 100: R = -79 -> 0, G = 148, B = 325 -> 255
    ((100, 255, 0), (0, 148, 255)),
    ((0, 128, 128), (0, 0, 0)),
]


def flat_picture_es(width, height, colours):
    """One I picture of DC-only intra blocks.  colours[mb] = (y0, y1, y2, y3, cb, cr): the four luma blocks' values and
    the chroma values of macroblock mb (raster order).  One slice per picture, default matrices."""
    import synth_es as S
    mbw, mbh = (width + 15) // 16, (height + 15) // 16
    assert len(colours) == mbw * mbh
    w = S.BitWriter()
    w.start_code(0xB3)
    w.put(width, 12); w.put(height, 12); w.put(1, 4); w.put(5, 4); w.put(0x3FFFF, 18); w.put(1, 1); w.put(20, 10); w.put(0, 1)
    w.put(0, 1); w.put(0, 1)
    w.start_code(0x00)
    w.put(0, 10); w.put(1, 3); w.put(0xFFFF, 16); w.put(0, 1)
    w.start_code(0x01)
    w.put(8, 5)   # quantiser scale (DC is not quantised by it)
    w.put(0, 1)   # no extra information
    pred = {"y": 128, "cb": 128, "cr": 128}  # mpeg1.js:262-264

    def dc(value, key, luma):
        diff = value - pred[key]
        size = 0 if diff == 0 else abs(diff).bit_length()
        w.code((S.DC_LUMA_CODE if luma else S.DC_CHROMA_CODE)[size])
        if size:
            w.put(diff if diff > 0 else diff + (1 << size) - 1, size)
        pred[key] = value
        w.code("10")  # end_of_block

    for mb in range(mbw * mbh):
        w.code(S.MBA_CODE[1])
        w.code(S.TYPE_I_CODE[0x01])  # intra, no quantiser change
        y0, y1, y2, y3, cb, cr = colours[mb]
        for v in (y0, y1, y2, y3):
            dc(v, "y", True)
        dc(cb, "cb", False)  # block 4 -> the Cb plane
        dc(cr, "cr", False)  # block 5 -> the Cr plane (SURVEY Q8)
    w.align()
    w.start_code(0xB7)  # sequence end: the slice ends at a start code
    return w.tobytes()


def hand_picture():
    """48 x 32 (3 x 2 macroblocks): every hand-computed colour occurs as one 8 x 8 luma block; width 46 x height 30
    is displayed, so the last quad column / row of the coded picture is cropped (canvas2d.js:64-79)."""
    triples = [h[0] for h in HAND]
    mbs = []
    for mb in range(6):
        y, cb, cr = triples[mb % len(triples)]
        y2 = triples[(mb + 3) % len(triples)][0]
        mbs.append((y, y2, y2, y, cb, cr))
    return mbs


def expected_rgba(width, height, mbw, colours):
    out = np.full((height, width, 4), 255, np.uint8)
    table = {h[0]: h[1] for h in HAND}
    for Y in range((height >> 1) * 2):
        for X in range((width >> 1) * 2):
            mb = (Y // 16) * mbw + X // 16
            y0, y1, y2, y3, cb, cr = colours[mb]
            yy = (y0, y1, y2, y3)[((Y % 16) // 8) * 2 + (X % 16) // 8]
            if (yy, cb, cr) in table:
                out[Y, X, :3] = table[(yy, cb, cr)]
            else:  # a luma value paired with another macroblock's chroma: the formula itself
                r = (cr + ((cr * 103) >> 8)) - 179
                g = ((cb * 88) >> 8) - 44 + ((cr * 183) >> 8) - 91
                b = (cb + ((cb * 198) >> 8)) - 227
                out[Y, X, :3] = np.clip([yy + r, yy - g, yy + b], 0, 255)
    return out


def test_hand_computed_colours_follow_from_the_formula():
    """the table above really is the JS arithmetic (a typo in a hand-computed line would hide behind the formula branch)"""
    for (y, cb, cr), want in HAND:
        r = (cr + ((cr * 103) >> 8)) - 179
        g = ((cb * 88) >> 8) - 44 + ((cr * 183) >> 8) - 91
        b = (cb + ((cb * 198) >> 8)) - 227
        assert tuple(int(np.clip(v, 0, 255)) for v in (y + r, y - g, y + b)) == want, (y, cb, cr)


def flat_planes(colours):
    """The Y / Cr / Cb planes (48x32 coded) that hold exactly the chosen samples of hand_picture()."""
    Y, Cb, Cr = np.zeros((32, 48), np.uint8), np.zeros((16, 24), np.uint8), np.zeros((16, 24), np.uint8)
    for mb, (y0, y1, y2, y3, vb, vr) in enumerate(colours):
        r0, c0 = (mb // 3) * 16, (mb % 3) * 16
        Y[r0:r0 + 8, c0:c0 + 8], Y[r0:r0 + 8, c0 + 8:c0 + 16] = y0, y1
        Y[r0 + 8:r0 + 16, c0:c0 + 8], Y[r0 + 8:r0 + 16, c0 + 8:c0 + 16] = y2, y3
        Cb[r0 // 2:r0 // 2 + 8, c0 // 2:c0 // 2 + 8] = vb
        Cr[r0 // 2:r0 // 2 + 8, c0 // 2:c0 // 2 + 8] = vr
    return Y.ravel(), Cr.ravel(), Cb.ravel()


def test_flat_picture_decodes_to_the_chosen_samples_in_the_reference():
    """the construction: the reference decodes the flat picture to exactly the chosen Y / Cb / Cr values
    (its decode is recorded in tests/golden/reference/decodes.json)"""
    colours = hand_picture()
    es = flat_picture_es(46, 30, colours)
    helpers.assert_matches_reference("rgba/flat_picture", [flat_planes(colours)], None, es)


@pytest.mark.gpu
def test_fused_rgba_epilogue_gives_the_hand_computed_colours():
    from jsmpeg_b200.batch import OUT_RGBA, BatchDecoder
    colours = hand_picture()
    es = flat_picture_es(46, 30, colours)
    bd = BatchDecoder(1)
    bd.write(0, es)
    assert bd.decode(1, OUT_RGBA) == 1
    got = bd.read_rgba(0)
    want = expected_rgba(46, 30, 3, colours)
    assert np.array_equal(got, want), np.argwhere(got != want)[:8]
    bd.close()
