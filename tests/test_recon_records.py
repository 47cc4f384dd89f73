"""Stage 2 against a record-level model, on records no real stream produces.

The stream generators keep every motion vector's footprint inside the planes, and the GPU suite feeds stage 2
only what a real stream yields.  Here seeded, adversarial macroblock records -- vectors that leave the plane,
wrap into the neighbouring row or end exactly on its last sample, coefficients at the ends of the IDCT's range,
junk wherever the record format says "not read" -- go through:

  * a model written from the reference (src/mpeg1.js:459-687 copyMacroblock, :838-914 the DC-only shortcut and
    Copy/Add{Block,Value}ToDestination, :916-983 IDCT) and ISO 11172-2 2.4.4.3 for B pictures, in numpy and
    Python integers.  It does not call the oracle;
  * CPU tier: the oracle (oracle_reconstruct[_b]) and the device code compiled for the host
    (tests/emu/walk_emu.cpp: emu_reconstruct_picture[_b]);
  * GPU tier: all four stage-2 kernels through jsmpeg_b200_debug_reconstruct_batch, which runs ONE launcher call
    over many pictures of any sizes, as the engine does.  Every buffer is sized for the call's largest picture
    and its surplus holds canaries, so that a stray read or write stays inside the allocation and shows.

Record contract the generator keeps (stage 1 always writes records this way): an intra macroblock has cbp 0x3f,
and a DC-only block has zeros in coefficients 1..63.
"""
import ctypes

import numpy as np
import pytest

import helpers

# ---- the record format (jsmpeg_b200/csrc/records.h) -----------------------------------------------------------
MBF_PRESENT, MBF_INTRA, MBF_SKIPPED, MBF_MOTION_BWD, MBF_MOTION_FWD = 0x01, 0x02, 0x04, 0x08, 0x10
RECORD = np.dtype([("mv_h", "<i2"), ("mv_v", "<i2"), ("flags", "u1"), ("cbp", "u1"), ("dc_only", "u1"), ("qscale", "u1"),
                   ("bit_pos", "<u4"), ("bwd_h", "<i2"), ("bwd_v", "<i2")])
assert RECORD.itemsize == 16

# MPEG1.PREMULTIPLIER_MATRIX (src/mpeg1.js:1026-1035)
PREMULTIPLIER = np.array([
    32, 44, 42, 38, 32, 25, 17, 9, 44, 62, 58, 52, 44, 35, 24, 12, 42, 58, 55, 49, 42, 33, 23, 12,
    38, 52, 49, 44, 38, 30, 20, 10, 32, 44, 42, 38, 32, 25, 17, 9, 25, 35, 33, 30, 25, 20, 14, 7,
    17, 24, 23, 20, 17, 14, 9, 5, 9, 12, 12, 10, 9, 7, 5, 2], np.int64)

# per-launch task limits of the four kernels (recon.cuh / recon.cu)
KINDS = {"plain": (0, 80), "rgba": (1, 60), "b": (2, 64), "rgba_b": (3, 48)}

MB_WIDTHS = (1, 2, 3, 5, 16, 17, 31, 33, 45, 120, 256)
MB_HEIGHTS = (1, 2, 3, 9, 17)


# ---- the model -------------------------------------------------------------------------------------------------
def _i32(x):
    """JS ToInt32: what `>>` does to its left operand and what a store into an Int32Array keeps."""
    return ((x + (1 << 31)) & 0xFFFFFFFF) - (1 << 31)


def _idct8(v, row):
    """One 8-point pass of MPEG1.IDCT (mpeg1.js:925-981) on v[0..7] (arrays over all blocks and columns / rows)."""
    b1 = v[4]
    b3 = v[2] + v[6]
    b4 = v[5] - v[3]
    t1 = v[1] + v[7]
    t2 = v[3] + v[5]
    b6 = v[1] - v[7]
    b7 = t1 + t2
    m0 = v[0]
    x4 = (_i32(b6 * 473 - b4 * 196 + 128) >> 8) - b7
    x0 = x4 - (_i32((t1 - t2) * 362 + 128) >> 8)
    x1 = m0 - b1
    x2 = (_i32((v[2] - v[6]) * 362 + 128) >> 8) - b3
    x3 = m0 + b1
    y3, y4, y5, y6 = x1 + x2, x3 + b3, x1 - x2, x3 - b3
    y7 = -x0 - (_i32(b4 * 473 + b6 * 196 + 128) >> 8)
    out = (b7 + y4, x4 + y3, y5 - x0, y6 - y7, y6 + y7, x0 + y5, y3 - x4, y4 - b7)
    return [_i32(o + 128) >> 8 if row else _i32(o) for o in out]


def model_idct(blocks):
    """MPEG1.IDCT of premultiplied blocks, shape (..., 64) -> (..., 64) int64."""
    v = np.asarray(blocks, np.int64).reshape(-1, 8, 8).copy()
    cols = _idct8([v[:, k, :] for k in range(8)], row=False)  # column pass: all 8 columns at once
    for k in range(8):
        v[:, k, :] = cols[k]
    rows = _idct8([v[:, :, k] for k in range(8)], row=True)
    for k in range(8):
        v[:, :, k] = rows[k]
    return v.reshape(np.shape(blocks))


def _half_trunc(m):
    """motion / 2 truncated toward zero (mpeg1.js:562-565: (motionH / 2) >> 1 and & 1 act on ToInt32 of a half)."""
    return np.sign(m) * (np.abs(m) // 2)


def _predict(ref, stride, size, rows, cols, mh, mv):
    """copyMacroblock for one plane: (n, size, size) predicted samples.  The source index is flat
    ((row * size + V) * stride + col * size + H, mpeg1.js:479): a vector past the end of a row reads the next row.
    A tap outside the plane is `undefined` in JS; the sample's sum becomes NaN and NaN & 0xff = 0."""
    psize = len(ref)
    oh, ov = (mh & 1).astype(bool), (mv & 1).astype(bool)
    base = (rows * size + (mv >> 1)) * stride + cols * size + (mh >> 1)
    i = base[:, None, None] + np.arange(size)[None, :, None] * stride + np.arange(size)[None, None, :]
    oh, ov = oh[:, None, None], ov[:, None, None]

    def tap(t):
        return ref[np.clip(t, 0, psize - 1)].astype(np.int64), (t >= 0) & (t < psize)

    (a, ia), (b, ib), (c, ic), (d, id_) = tap(i), tap(i + 1), tap(i + stride), tap(i + stride + 1)
    ok = ia & (ib | ~oh) & (ic | ~ov) & (id_ | ~(oh & ov))
    val = np.where(oh & ov, (a + b + c + d + 2) >> 2, np.where(oh, (a + b + 1) >> 1, np.where(ov, (a + c + 1) >> 1, a)))
    return np.where(ok, val, 0)


def _planes(buf, W, H):
    ys = W * H * 256
    return buf[:ys], buf[ys:ys + ys // 4], buf[ys + ys // 4:ys * 3 // 2]  # Y, Cr, Cb


def model_reconstruct(W, H, rec, coef, fwd, cur, bwd=None):
    """One picture: records `rec` (RECORD, W*H), coefficients (W*H, 6, 64), plane sets Y | Cr | Cb.  Returns the new
    plane set (cur's first W*H*384 bytes with the picture written).  bwd given: a B picture (ISO 11172-2 2.4.4.3)."""
    n = W * H
    rec = rec[:n]
    coef = np.asarray(coef[:n], np.int64)
    out = np.array(cur[:n * 384], np.uint8)
    oy, ocr, ocb = _planes(out, W, H)
    fy, fcr, fcb = _planes(fwd, W, H)
    flags = rec["flags"].astype(np.int64)
    present = (flags & MBF_PRESENT) != 0
    intra = present & ((flags & MBF_INTRA) != 0)
    pred_mb = present & ~intra
    mbs = np.nonzero(present)[0]
    rows, cols = mbs // W, mbs % W
    k = len(mbs)

    # residual: (k, 6, 8, 8); a DC-only block is (c0 * 32 + 128) >> 8 everywhere (mpeg1.js:838-853)
    c = coef[mbs]
    bit = 0x20 >> np.arange(6)
    coded = (rec["cbp"][mbs, None].astype(np.int64) & bit) != 0
    dc_only = coded & ((rec["dc_only"][mbs, None].astype(np.int64) & bit) != 0)
    res = model_idct(c * PREMULTIPLIER).reshape(k, 6, 8, 8)
    dc = _i32(c[:, :, 0] * PREMULTIPLIER[0] + 128) >> 8
    res = np.where(dc_only[:, :, None, None], dc[:, :, None, None], res)
    res = np.where(coded[:, :, None, None], res, 0)
    assert not (intra[mbs][:, None] & ~coded).any(), "record contract: an intra macroblock has cbp 0x3f"

    # prediction: forward, backward, or their average with each direction rounded first
    def predict_from(planes, mh, mv):
        py = _predict(planes[0], W * 16, 16, rows, cols, mh, mv)
        ch, cv = _half_trunc(mh), _half_trunc(mv)
        return py, _predict(planes[1], W * 8, 8, rows, cols, ch, cv), _predict(planes[2], W * 8, 8, rows, cols, ch, cv)

    pf = predict_from((fy, fcr, fcb), rec["mv_h"][mbs].astype(np.int64), rec["mv_v"][mbs].astype(np.int64))
    if bwd is None:
        pred = pf
    else:
        pb = predict_from(_planes(bwd, W, H), rec["bwd_h"][mbs].astype(np.int64), rec["bwd_v"][mbs].astype(np.int64))
        use_b = (flags[mbs] & MBF_MOTION_BWD) != 0
        use_f = ~use_b | ((flags[mbs] & MBF_MOTION_FWD) != 0)  # neither bit: forward, like I/P records
        pred = tuple(np.where((use_f & use_b)[:, None, None], (f + b + 1) >> 1, np.where(use_b[:, None, None], b, f))
                     for f, b in zip(pf, pb))

    # luma blocks 0..3 -> the macroblock's 16 x 16; block 4 -> Cb, block 5 -> Cr (mpeg1.js:819-834)
    ry = np.zeros((k, 16, 16), np.int64)
    ry[:, :8, :8], ry[:, :8, 8:], ry[:, 8:, :8], ry[:, 8:, 8:] = res[:, 0], res[:, 1], res[:, 2], res[:, 3]
    isp = pred_mb[mbs][:, None, None]
    new_y = np.clip(np.where(isp, pred[0], 0) + ry, 0, 255)
    new_cr = np.clip(np.where(isp, pred[1], 0) + res[:, 5], 0, 255)
    new_cb = np.clip(np.where(isp, pred[2], 0) + res[:, 4], 0, 255)

    def scatter(plane, stride, size, val):
        idx = (rows[:, None, None] * size + np.arange(size)[None, :, None]) * stride + cols[:, None, None] * size + \
            np.arange(size)[None, None, :]
        plane[idx] = val

    scatter(oy, W * 16, 16, new_y)
    scatter(ocr, W * 8, 8, new_cr)
    scatter(ocb, W * 8, 8, new_cb)
    return out  # absent macroblocks keep what cur held


# ---- the record generator --------------------------------------------------------------------------------------
MB_TYPES_P = ("absent", "intra", "fwd")
MB_TYPES_B = ("absent", "intra", "fwd", "bwd", "both", "neither")
VEC_CATS = ("small", "wrap", "edge_luma", "edge_chroma", "edge_top", "out_top", "out_bottom", "out_far")
VEC_P = (0.3, 0.1, 0.12, 0.12, 0.1, 0.08, 0.08, 0.1)
COEF_CATS = ("sparse", "natural", "full2048", "saturating")
ROW_MODES = ("mixed", "fullpel", "dc_only")


def _vectors(rng, cat, rows, cols, W, H):
    """(mh, mv) per macroblock for its vector category (luma half-pel units, int16 as in the record)."""
    n = len(cat)

    def jig():  # one half-pel either way, or none
        return rng.integers(-1, 2, n)

    def toward_zero_pair(m):  # a luma component whose truncated half is m
        return 2 * m + np.where(m < 0, -1, 1) * rng.integers(0, 2, n)

    cand = {
        "small": rng.integers(-12, 13, (2, n)),
        # past the right or the left end of the row: the flat index reads the neighbouring row
        "wrap": (2 * np.where(rng.random(n) < 0.5, (W - cols) * 16 - rng.integers(1, 16, n), -cols * 16 - rng.integers(1, 16, n))
                 + rng.integers(0, 2, n), rng.integers(-6, 7, n)),
        # the footprint's last sample on the plane's last sample (luma), +- one half-pel
        "edge_luma": (2 * (W - 1 - cols) * 16 + jig(), 2 * (H - 1 - rows) * 16 + jig()),
        "edge_chroma": (toward_zero_pair(2 * (W - 1 - cols) * 8 + jig()), toward_zero_pair(2 * (H - 1 - rows) * 8 + jig())),
        # the footprint starting on sample 0, +- one half-pel
        "edge_top": (-2 * cols * 16 + jig(), -2 * rows * 16 + jig()),
        "out_top": (rng.integers(-6, 7, n), 2 * (-rows * 16 - rng.integers(1, 24, n)) + rng.integers(0, 2, n)),
        "out_bottom": (rng.integers(-6, 7, n), 2 * ((H - 1 - rows) * 16 + rng.integers(1, 24, n)) + rng.integers(0, 2, n)),
        "out_far": rng.integers(-4000, 4001, (2, n)),
    }
    mh, mv = np.zeros(n, np.int64), np.zeros(n, np.int64)
    for ci, name in enumerate(VEC_CATS):
        sel = cat == ci
        mh[sel], mv[sel] = np.asarray(cand[name][0])[sel], np.asarray(cand[name][1])[sel]
    return mh, mv


def _coefficients(rng, n, coded, dc_only, cat):
    """(n, 6, 64) int16: a category per coded block, junk in every block that is not coded."""
    junk = rng.integers(-32768, 32768, (n, 6, 64))
    sparse = np.where(rng.random((n, 6, 64)) < 0.06, rng.integers(-2048, 2048, (n, 6, 64)), 0)
    rc = np.add.outer(np.arange(8), np.arange(8)).reshape(64)
    natural = np.clip(np.rint(rng.normal(0, 1, (n, 6, 64)) * (600.0 / (1 + rc))), -2048, 2047).astype(np.int64)
    which = rng.integers(0, 3, (n, 6, 1))  # all -2048, all 2047, or random signs
    full = np.where(which == 0, -2048, np.where(which == 1, 2047, np.where(rng.random((n, 6, 64)) < 0.5, -2048, 2047)))
    saturating = natural // 4
    saturating[:, :, 0] = np.where(rng.random((n, 6)) < 0.5, -2048, 2047)
    gen = np.select([cat[..., None] == i for i in range(4)], [sparse, natural, full, saturating])
    dc = np.where(rng.random((n, 6)) < 0.3, np.where(rng.random((n, 6)) < 0.5, -2048, 2047), rng.integers(-2048, 2048, (n, 6)))
    dc_blocks = np.zeros((n, 6, 64), np.int64)
    dc_blocks[:, :, 0] = dc
    gen = np.where(dc_only[..., None], dc_blocks, gen)  # the contract: zeros behind a DC-only block's coefficient 0
    return np.where(coded[..., None], gen, junk).astype(np.int16)


def gen_picture(rng, W, H, b=False):
    """Seeded adversarial records for a W x H macroblock picture.  Returns (records, coefficients, labels): labels[mb]
    names the macroblock's categories, so that a failure says which case it was."""
    n = W * H
    mbs = np.arange(n)
    rows, cols = mbs // W, mbs % W
    row_mode = rng.choice(len(ROW_MODES), H, p=(0.6, 0.25, 0.15))
    row_mode[:3] = rng.permutation(len(ROW_MODES))[:H]  # every mode in every picture of three rows or more
    row_mode = row_mode[rows]
    types = MB_TYPES_B if b else MB_TYPES_P
    type_p = (0.1, 0.15, 0.3, 0.2, 0.2, 0.05) if b else (0.1, 0.2, 0.7)
    mtype = rng.choice(len(types), n, p=type_p)
    present, intra = mtype != 0, mtype == 1
    vcat = rng.choice(len(VEC_CATS), n, p=VEC_P)
    mh, mv = _vectors(rng, vcat, rows, cols, W, H)
    bcat = rng.choice(len(VEC_CATS), n, p=VEC_P)
    bh, bv = _vectors(rng, bcat, rows, cols, W, H)
    fullpel = row_mode == 1  # whole macroblock rows without a half-pel component (luma or chroma): the FULLPEL path
    mh, mv, bh, bv = (np.where(fullpel, m - m % 4, m) for m in (mh, mv, bh, bv))

    rec = np.zeros(n, RECORD)
    flags = np.where(present, MBF_PRESENT, 0) | np.where(intra, MBF_INTRA, 0) | np.where(rng.random(n) < 0.2, MBF_SKIPPED, 0)
    if b:
        name = np.array(types)[mtype]
        flags |= np.where(np.isin(name, ("fwd", "both")), MBF_MOTION_FWD, 0) | np.where(np.isin(name, ("bwd", "both")), MBF_MOTION_BWD, 0)
    junk_flags = rng.integers(0, 256, n) & ~MBF_PRESENT  # an absent record: nothing of it is read
    rec["flags"] = np.where(present, flags, junk_flags)
    uses_b = b & present & ~intra & ((rec["flags"] & MBF_MOTION_BWD) != 0)
    rec["mv_h"], rec["mv_v"] = mh, mv
    rec["bwd_h"] = np.where(uses_b, bh, rng.integers(-32768, 32768, n))  # mv_bwd is read only by B records that use it
    rec["bwd_v"] = np.where(uses_b, bv, rng.integers(-32768, 32768, n))
    rec["bit_pos"] = rng.integers(0, 1 << 32, n, dtype=np.uint64)
    rec["qscale"] = rng.integers(0, 256, n)

    cbp = np.where(intra, 0x3F, rng.integers(0, 64, n))
    bit = 0x20 >> np.arange(6)
    coded = present[:, None] & ((cbp[:, None] & bit) != 0)
    dc_only = coded & np.where((row_mode == 2)[:, None], True, rng.random((n, 6)) < 0.3)
    dcbits = (dc_only * bit).sum(1)
    rec["cbp"] = np.where(present, cbp, rng.integers(0, 64, n))
    rec["dc_only"] = dcbits | (rng.integers(0, 64, n) & ~np.where(present, cbp, 0))  # junk in the bits of uncoded blocks
    ccat = rng.choice(len(COEF_CATS), (n, 6))
    coef = _coefficients(rng, n, coded, dc_only, ccat)

    labels = []
    for m in range(n):
        t = types[mtype[m]]
        lab = f"mb {m} (row {rows[m]}, col {cols[m]}, {ROW_MODES[row_mode[m]]} row): {t}"
        if present[m] and not intra[m]:
            lab += f", vector {VEC_CATS[vcat[m]]} ({mh[m]}, {mv[m]})"
            if uses_b[m]:
                lab += f", backward {VEC_CATS[bcat[m]]} ({bh[m]}, {bv[m]})"
        if present[m]:
            lab += ", blocks " + " ".join(("dc" if dc_only[m, k] else COEF_CATS[ccat[m, k]]) if coded[m, k] else "-" for k in range(6))
        labels.append(lab)
    return rec, coef, labels


def _first_difference(W, H, got, want, labels, what):
    """None when equal, else a message naming the first differing sample's macroblock and its categories."""
    n = W * H * 384
    bad = np.nonzero(got[:n] != want[:n])[0]
    if not len(bad):
        return None
    i = int(bad[0])
    ys = W * H * 256
    if i < ys:
        plane, x, y, mb = "Y", i % (W * 16), i // (W * 16), (i // (W * 16) // 16) * W + (i % (W * 16)) // 16
    else:
        j = (i - ys) % (ys // 4)
        plane = "Cr" if i < ys + ys // 4 else "Cb"
        x, y = j % (W * 8), j // (W * 8)
        mb = (y // 8) * W + x // 8
    return (f"{what}: {len(bad)} samples differ; first: plane {plane} ({x}, {y}) got {got[i]} want {want[i]}; "
            f"{labels[mb]}")


# ---- CPU tier: model = oracle = the device code compiled for the host -------------------------------------------
class _Planes(ctypes.Structure):
    _fields_ = [("y", ctypes.c_void_p), ("cr", ctypes.c_void_p), ("cb", ctypes.c_void_p)]


def _planes_t(buf, W, H):
    return _Planes(*(p.ctypes.data for p in _planes(buf, W, H)))


def oracle_reconstruct(W, H, rec, coef, fwd, cur, bwd=None):
    lib = helpers.oracle_lib()
    seq = helpers.SeqParamsOracle()
    seq.mb_width, seq.mb_size = W, W * H
    out = np.array(cur[:W * H * 384], np.uint8)
    hdr = np.ascontiguousarray(rec)
    c = np.ascontiguousarray(coef, np.int16)
    f, o = _planes_t(fwd, W, H), _planes_t(out, W, H)
    if bwd is None:
        lib.oracle_reconstruct(ctypes.byref(seq), W * 16, H * 16, ctypes.c_void_p(hdr.ctypes.data), ctypes.c_void_p(c.ctypes.data),
                               ctypes.byref(f), ctypes.byref(o))
    else:
        bp = _planes_t(bwd, W, H)
        lib.oracle_reconstruct_b(ctypes.byref(seq), W * 16, H * 16, ctypes.c_void_p(hdr.ctypes.data), ctypes.c_void_p(c.ctypes.data),
                                 ctypes.byref(f), ctypes.byref(bp), ctypes.byref(o))
    return out


def emu_reconstruct(W, H, rec, coef, fwd, cur, bwd=None):
    from test_walk_emu import emu_lib
    lib = emu_lib()
    vp = ctypes.c_void_p
    pad = W * 16 + 64  # the planes' readable tail, as the product allocates it
    out = np.zeros(W * H * 384 + pad, np.uint8)
    out[:W * H * 384] = cur[:W * H * 384]
    hdr = np.ascontiguousarray(rec)
    c = np.ascontiguousarray(coef, np.int16)
    f = np.concatenate([fwd[:W * H * 384], np.zeros(pad, np.uint8)])
    if bwd is None:
        lib.emu_reconstruct_picture.argtypes = [vp, vp, vp, vp, ctypes.c_int, ctypes.c_int]
        lib.emu_reconstruct_picture(hdr.ctypes.data, c.ctypes.data, out.ctypes.data, f.ctypes.data, W, H)
    else:
        bb = np.concatenate([bwd[:W * H * 384], np.zeros(pad, np.uint8)])
        lib.emu_reconstruct_picture_b.argtypes = [vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int]
        lib.emu_reconstruct_picture_b(hdr.ctypes.data, c.ctypes.data, out.ctypes.data, f.ctypes.data, bb.ctypes.data, W, H)
    return out[:W * H * 384]


def _random_planes(rng, W, H, k):
    return [rng.integers(0, 256, W * H * 384, dtype=np.uint8) for _ in range(k)]


@pytest.mark.parametrize("b", [False, True], ids=["ip", "b"])
@pytest.mark.parametrize("W", MB_WIDTHS)
def test_model_oracle_and_host_compiled_device_code_agree(W, b):
    """Every height of MB_HEIGHTS at this width: the model, the oracle and recon.cuh compiled for the host give the
    same planes on the adversarial records."""
    for H in MB_HEIGHTS:
        rng = np.random.default_rng([W, H, int(b), 1])
        rec, coef, labels = gen_picture(rng, W, H, b)
        fwd, bwd, cur = _random_planes(rng, W, H, 3)
        bwd = bwd if b else None
        want = model_reconstruct(W, H, rec, coef, fwd, cur, bwd)
        for name, fn in (("oracle", oracle_reconstruct), ("host-compiled recon.cuh", emu_reconstruct)):
            got = fn(W, H, rec, coef, fwd, cur, bwd)
            msg = _first_difference(W, H, got, want, labels, f"{W}x{H} {'B' if b else 'P'}: {name} vs model")
            assert msg is None, msg


def test_generator_reaches_every_category():
    """The generated records do contain what they are for: vectors out of the plane, wrapping, exactly at the edge
    (inside and one half-pel out), negative odd chroma vectors, blocks at +-2048, and saturation at 0 and 255."""
    W, H = 17, 9
    rng = np.random.default_rng(5)
    rec, coef, labels = gen_picture(rng, W, H, b=True)
    fwd, bwd, cur = _random_planes(rng, W, H, 3)
    text = "\n".join(labels)
    for word in MB_TYPES_B + VEC_CATS + COEF_CATS + ("dc", "fullpel row", "dc_only row"):
        assert word in text, word
    mh = rec["mv_h"].astype(int)
    pred = (rec["flags"] & (MBF_PRESENT | MBF_INTRA)) == MBF_PRESENT
    assert ((mh < 0) & (mh % 2 == 1) & pred).any()  # odd negative: chroma truncation and flat-index wrap
    assert (coef == -2048).all(axis=2).any() and (coef == 2047).all(axis=2).any()
    out = model_reconstruct(W, H, rec, coef, fwd, cur, bwd)
    written = np.concatenate([out[:W * H * 384][cur[:W * H * 384] != out[:W * H * 384]]])
    assert (written == 0).any() and (written == 255).any()


def test_model_idct_is_the_reference_idct():
    """The model's transform reproduces the reference's idct() on both recorded block sets
    (tests/golden/reference/idct.json), so the model is pinned to the reference itself."""
    import test_unit_parity as U
    for kind, blocks in (("random", U.random_blocks()), ("sparse_and_extreme", U.sparse_and_extreme_blocks())):
        want = helpers.reference_golden("idct")[kind]
        assert helpers.digest(blocks) == want["inputs"]
        got = model_idct(blocks).astype(np.int32)
        bad = [k for k in range(len(blocks)) if helpers.digest(got[k]) != want["outputs"][k]]
        assert len(got) == len(want["outputs"]) and not bad, f"{kind}: {len(bad)} blocks differ, first {bad[:8]}"


def test_row_magic_divides_exactly():
    """reconstruct_block finds a slot's macroblock row as umulhi(slot, row_magic) with row_magic = floor(2^32 / 6W) + 1
    (recon.cu fill_task): exact for every width 1..256 and every slot of a picture up to 256 macroblock rows."""
    for W in range(1, 257):
        magic = (1 << 32) // (6 * W) + 1
        slots = np.arange(6 * W * 256, dtype=np.uint64)
        got = (slots * np.uint64(magic)) >> np.uint64(32)
        assert np.array_equal(got, slots // np.uint64(6 * W)), W


# ---- GPU tier: the four kernels through one launcher call ------------------------------------------------------
CANARY = 0xA5


def _task(rng, W, H, b, rgba, cap_mb, cap, rgba_cap):
    """Buffers of one task, sized for the call's largest picture, the surplus filled with canaries."""
    n = W * H
    rec, coef, labels = gen_picture(rng, W, H, b)
    hdr = np.zeros(cap_mb, RECORD)
    hdr[:n] = rec
    hdr["flags"][n:] = MBF_PRESENT | MBF_INTRA  # a record past the picture that a stray CTA would reconstruct
    hdr["cbp"][n:] = 0x3F
    cf = np.zeros((cap_mb, 6, 64), np.int16)
    cf[:n] = coef
    cf[n:] = rng.integers(1, 2048, (cap_mb - n, 6, 64))

    def planes():
        p = np.full(cap, CANARY, np.uint8)
        p[:n * 384] = rng.integers(0, 256, n * 384, dtype=np.uint8)
        return p

    t = dict(W=W, H=H, rec=rec, coef=coef, labels=labels, hdr=hdr, cf=cf, fwd=planes(), cur=planes(),
             bwd=planes() if b else None, width=0, height=0, rgba=None)
    if rgba:  # display sizes inside the last macroblock column / row: odd ones and ones with width % 4 != 0
        t["width"] = int(W * 16 - rng.choice([0, 1, 2, 3, 5, 7, 9, 15][:min(8, W * 16)]))
        t["height"] = int(H * 16 - rng.choice([0, 1, 3, 6, 11, 15]))
        t["rgba"] = np.full(rgba_cap, CANARY, np.uint8)
        t["rgba"][:t["width"] * t["height"] * 4] = 0xFF  # the opaque white the picture buffer is created with
    return t


def run_batch(kind, geoms, seed):
    """One jsmpeg_b200_debug_reconstruct_batch call over tasks of the given (W, H); checks every task."""
    from jsmpeg_b200 import capi
    code, _ = KINDS[kind]
    b, rgba = kind in ("b", "rgba_b"), kind in ("rgba", "rgba_b")
    rng = np.random.default_rng(seed)
    mw, mh = max(w for w, _ in geoms), max(h for _, h in geoms)
    cap_mb = mw * mh
    cap = cap_mb * 384 + mw * 16 + 64
    rgba_cap = cap_mb * 256 * 4 + 64
    tasks = [_task(rng, W, H, b, rgba, cap_mb, cap, rgba_cap) for W, H in geoms]
    before = [{k: (None if t[k] is None else t[k].copy()) for k in ("hdr", "cf", "fwd", "bwd", "cur", "rgba")} for t in tasks]
    geometry = np.array([(t["W"], t["H"], t["width"], t["height"]) for t in tasks], np.int32)

    def ptrs(key):
        return np.array([0 if t[key] is None else t[key].ctypes.data for t in tasks], np.uint64)

    arrays = {k: ptrs(k) for k in ("hdr", "cf", "fwd", "bwd", "cur", "rgba")}
    lib = capi.product_library()
    rc = lib.jsmpeg_b200_debug_reconstruct_batch(code, len(tasks), geometry.ctypes.data, cap_mb, cap, rgba_cap,
                                                 *(arrays[k].ctypes.data for k in ("hdr", "cf", "fwd", "bwd", "cur", "rgba")))
    assert rc == 0
    for i, (t, old) in enumerate(zip(tasks, before)):
        W, H = t["W"], t["H"]
        what = f"{kind}, task {i} of {len(tasks)} ({W}x{H} macroblocks)"
        for k in ("hdr", "cf", "fwd", "bwd"):
            assert t[k] is None or np.array_equal(t[k], old[k]), f"{what}: the launch wrote into its input {k}"
        want = model_reconstruct(W, H, t["rec"], t["coef"], old["fwd"], old["cur"], old["bwd"])
        msg = _first_difference(W, H, t["cur"], want, t["labels"], what)
        assert msg is None, msg
        tail = t["cur"][W * H * 384:]
        assert (tail == CANARY).all(), f"{what}: {(tail != CANARY).sum()} bytes written past the plane set"
        if rgba:
            w, h = t["width"], t["height"]
            y, cr, cb = _planes(want, W, H)
            exp = helpers.canvas2d_rgba(y, cr, cb, w, h)
            got = t["rgba"][:w * h * 4].reshape(h, w, 4)
            if not np.array_equal(got, exp):
                yy, xx = np.nonzero((got != exp).any(2))
                raise AssertionError(f"{what}, display {w}x{h}: {len(yy)} RGBA pixels differ, first at ({xx[0]}, {yy[0]}): "
                                     f"{got[yy[0], xx[0]]} vs {exp[yy[0], xx[0]]}")
            assert (t["rgba"][w * h * 4:] == CANARY).all(), f"{what}: RGBA written past the picture"


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(KINDS))
@pytest.mark.parametrize("W", MB_WIDTHS)
def test_kernel_matches_model_one_task(kind, W):
    """One task per call, every height of MB_HEIGHTS at this width."""
    for H in MB_HEIGHTS:
        run_batch(kind, [(W, H)], seed=[W, H, KINDS[kind][0], 2])


# a narrow, tall picture next to a wide, short one, and others between: the grid covers the widest and the tallest
MIXED = [(1, 40), (40, 1), (17, 3), (3, 17), (5, 9), (33, 2), (2, 2), (45, 1), (1, 1), (16, 17)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(KINDS))
def test_kernel_matches_model_mixed_geometry(kind):
    run_batch(kind, MIXED, seed=[KINDS[kind][0], 3])


@pytest.mark.gpu
@pytest.mark.parametrize("extra", [1, 3], ids=["cap+1", "2cap+3"])
@pytest.mark.parametrize("kind", list(KINDS))
def test_kernel_matches_model_past_the_launch_limit(kind, extra):
    """More tasks than one launch holds (cap + 1, 2 cap + 3): the launcher's split into launches, with sizes that
    differ within and between the launches."""
    cap = KINDS[kind][1]
    n = cap + 1 if extra == 1 else 2 * cap + 3
    rng = np.random.default_rng([KINDS[kind][0], n])
    geoms = [(int(rng.integers(1, 7)), int(rng.integers(1, 5))) for _ in range(n)]
    geoms[n // 2] = (1, 6)  # one tall, narrow picture in the middle of the list
    run_batch(kind, geoms, seed=[KINDS[kind][0], n, 4])


# ---- engine level: streams of different sizes in one batch, OUT_RGBA --------------------------------------------
@pytest.mark.gpu
def test_engine_rgba_batch_of_different_sizes():
    """I/P streams of different widths and heights decoded together with the fused RGBA epilogue: every picture's
    planes equal the oracle's, its RGBA the canvas2d formula applied to them."""
    specs = [(320, 240, 6, 1), (176, 144, 6, 2), (640, 368, 5, 3), (48, 320, 6, 4)]
    clips = [b"".join(p for _, p in helpers.clip_packets(w, h, n, seed=s)) for (w, h, n, s) in specs]
    _engine_rgba_run(clips, [(w, h) for w, h, _, _ in specs], helpers.oracle_lib(), {})


@pytest.mark.gpu
def test_engine_rgba_b_pictures_of_different_sizes():
    """Two B-picture clips of different sizes (their B pictures share steps: reconstruct_rgba_b_kernel with mixed
    sizes) beside a shorter I/P stream."""
    import test_b_pictures as TB
    lib = helpers.oracle_lib()
    lib.oracle_set_decode_b(1)
    try:
        a = TB.natural_clip(176, 144, frames=7)[0]
        b = TB.natural_clip(64, 240, frames=7, seed=77)[0]
        c = b"".join(p for _, p in helpers.clip_packets(320, 96, 7, seed=5))
        _engine_rgba_run([a, b, c], [(176, 144), (64, 240), (320, 96)], lib, {"decode_b": 1})
    finally:
        lib.oracle_set_decode_b(0)


def _engine_rgba_run(clips, sizes, oracle, opts):
    from jsmpeg_b200.batch import OUT_RGBA, BatchDecoder
    expected = [helpers.decode_all(oracle, [(0, es)])[0] for es in clips]
    bd = BatchDecoder(len(clips), **opts)
    for i, es in enumerate(clips):
        bd.write(i, es)
    step = 0
    while bd.decode(1, OUT_RGBA):
        for i, frames in enumerate(expected):
            if step < len(frames):
                y, cr, cb = bd.read_planes(i)
                helpers.assert_frames_equal([(y, cr, cb)], [frames[step]], f"stream {i} picture {step}")
                w, h = sizes[i]
                assert np.array_equal(bd.read_rgba(i), helpers.canvas2d_rgba(y, cr, cb, w, h)), f"stream {i} RGBA picture {step}"
        step += 1
    assert step == max(len(f) for f in expected)
    assert bd.stats()["parse_errors"] == 0
    bd.close()
