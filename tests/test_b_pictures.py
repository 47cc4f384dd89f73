"""The B-picture extension (SURVEY 8f rank 4) -- CPU side.

The reference skips B pictures (src/mpeg1.js:181-184), so there is nothing to run for parity:
  * the ORACLE's B-picture path (oracle/mpeg1_oracle.c, oracle_set_decode_b) is checked against FFmpeg's
    mpeg1video decoder on streams of natural content written by tools/mini_enc.py -- PSNR on the luma plane,
    since the two IDCTs differ (the same comparison gives 58 dB on FFmpeg-made I/P clips);
  * the PRODUCT's device code for B pictures (walk_b.cuh, stage 1b, recon.cuh<BIDIR>) is emulated on the host
    (tests/emu) and must equal the oracle bit for bit -- records, coefficients, planes -- on those streams and
    on the syntax-level generator's B cases (tools/synth_es.py: all macroblock types of table B.2d, skipped
    runs, both f_codes, full-pel vectors, several slices);
  * with the extension off, oracle and product treat a B picture exactly as before (consumed, nothing decoded).
The GPU twin is tests/test_gpu_zz_b_pictures.py.
"""
import ctypes
import functools
import os

import numpy as np
import pytest

import helpers
import synth_es
from test_walk_emu import emu_lib, picture_starts, stream_geometry

HERE = os.path.dirname(os.path.abspath(__file__))


def picture_types(es):
    return [(es[s + 1] >> 3) & 7 for s in picture_starts(es)]


def display_order(types):
    """Coded indices in display order: an I/P picture is shown after the B pictures that follow it in the stream."""
    out, held = [], None
    for k, t in enumerate(types):
        if t == 3:
            out.append(k)
        else:
            if held is not None:
                out.append(held)
            held = k
    if held is not None:
        out.append(held)
    return out


def psnr(a, b):
    d = a.astype(np.float64) - b.astype(np.float64)
    m = float((d * d).mean())
    return 99.0 if m == 0 else 10 * np.log10(255 * 255 / m)


@pytest.fixture
def oracle_b():
    lib = helpers.oracle_lib()
    lib.oracle_set_decode_b(1)
    yield lib
    lib.oracle_set_decode_b(0)


@functools.lru_cache(maxsize=None)
def natural_clip(width=176, height=144, frames=13, b_frames=2, seed=1234, f_codes=(3, 3), full_pel=(0, 0), one_slice=False):
    """(ES bytes, picture types in coded order, display index per coded picture, macroblock statistics)."""
    import mini_enc
    return mini_enc.make_b_clip(width, height, frames, b_frames, seed, f_codes=f_codes, full_pel=full_pel, one_slice=one_slice)


# (forward_f_code, backward_f_code), (full_pel_forward_vector, full_pel_backward_vector): each direction with its own
# vector range and unit (ISO 11172-2 2.4.2.5; mpeg1.js:395-457 once per direction)
VECTOR_FORMS = [((3, 3), (0, 0)), ((2, 4), (0, 1)), ((4, 2), (1, 0))]


# (b_frames, display pictures, vector form, one slice per picture -- what FFmpeg itself writes -- instead of one per row)
@pytest.mark.parametrize("b_frames,frames,form,one_slice", [(2, 13, 0, False), (1, 9, 0, False), (3, 9, 0, False), (2, 10, 1, False),
                                                            (2, 10, 2, False), (2, 10, 0, True)])
def test_oracle_b_pictures_against_ffmpeg(oracle_b, tmp_path, b_frames, frames, form, one_slice):
    cv2 = pytest.importorskip("cv2")
    f_codes, full_pel = VECTOR_FORMS[form]
    es, types, order, stats = natural_clip(frames=frames, b_frames=b_frames, f_codes=f_codes, full_pel=full_pel, one_slice=one_slice)
    assert types.count(3) >= 4 and all(stats[k] > 0 for k in ("fwd", "bwd", "bi", "intra", "skipped")), stats
    got, _, d = helpers.decode_all(oracle_b, [(0, es)])
    w, h = d.width, d.height
    assert len(got) == len(types)
    path = str(tmp_path / "clip.m1v")
    with open(path, "wb") as f:
        f.write(es)
    cap = cv2.VideoCapture(path, cv2.CAP_FFMPEG)
    cap.set(cv2.CAP_PROP_CONVERT_RGB, 0)  # the decoder's own luma plane, no colour conversion
    theirs = []
    while True:
        ok, frame = cap.read()
        if not ok:
            break
        theirs.append(frame[:h, :w].copy())
    shown = display_order(types)
    assert len(theirs) == len(shown), (len(theirs), len(shown))
    for k, ci in enumerate(shown):
        y = got[ci][0].reshape(-1, w)[:h]
        # 58 dB is what the I/P path (pinned bit-exactly to the reference) gives against FFmpeg; a wrong reference,
        # vector, rounding or skipped-macroblock rule in a B picture costs tens of dB
        assert psnr(y, theirs[k]) > 50.0, f"display {k} (coded {ci}, type {types[ci]}): {psnr(y, theirs[k]):.1f} dB"
    d.destroy()


def test_display_order_rendering_against_ffmpeg(oracle_b, tmp_path):
    """The host class with decodeBPictures + displayOrder hands the destination the pictures in the order a screen
    shows them -- the order FFmpeg's decoder returns them in: compared picture for picture (PSNR, as above), and the
    temporal_reference the library reports counts the display positions."""
    cv2 = pytest.importorskip("cv2")
    from jsmpeg_b200 import decoder
    es, types, order, _ = natural_clip()
    d = decoder.MPEG1Video({"decodeFirstFrame": False, "decodeBPictures": True, "displayOrder": True}, lib=oracle_b)
    rec = decoder.PlaneRecorder()
    d.connect(rec)
    d.write(0, [es])
    seen = []
    while d.decode():
        seen.append(d.lastPicture())
    d.flush()
    assert [t for t, _ in seen] == types and [r for _, r in seen] == order  # (one GOP header: temporal_reference = display index)
    w, h = d.width, d.height
    path = str(tmp_path / "clip.m1v")
    with open(path, "wb") as f:
        f.write(es)
    cap = cv2.VideoCapture(path, cv2.CAP_FFMPEG)
    cap.set(cv2.CAP_PROP_CONVERT_RGB, 0)
    k = 0
    while True:
        ok, frame = cap.read()
        if not ok:
            break
        assert psnr(rec.frames[k][0].reshape(-1, w)[:h], frame[:h, :w]) > 50.0, f"display picture {k}"
        k += 1
    assert k == len(rec.frames) == len(types)
    d.destroy()


def test_extension_off_b_pictures_are_consumed_and_not_decoded():
    lib = helpers.oracle_lib()
    lib.oracle_set_decode_b(0)
    es = synth_es.make_case("b_rows")
    types = picture_types(es)
    frames, idx, d = helpers.decode_all(lib, [(0, es)])
    assert len(frames) == len(types)  # decode() answers true for every picture (mpeg1.js:181-184)
    for k, t in enumerate(types):
        if t == 3 and k > 0:  # the wrapper re-renders the last I/P picture (mpeg1-wasm.js:103-119)
            assert all(np.array_equal(a, b) for a, b in zip(frames[k], frames[k - 1]))
    # and that is exactly what the reference does with the stream (picture 0: C planes start uninitialised, Q19)
    helpers.assert_matches_reference("b_rows/extension_off", frames, idx, es, first=1)
    d.destroy()


def _emulated_b_pipeline(es, name, damaged=False):
    """walk (I/P: lane-parallel; B: walk_b) -> stage 1b -> stage 2 (two references for B), the product's plane
    bookkeeping (engine.cu), against the oracle's records, coefficients and planes of every picture.
    damaged: planes are compared up to the first picture whose walk reports an error -- what stage 2 does with
    the half-parsed macroblock of such a picture is outside the parity domain (DESIGN.md, section 6), for I/P
    pictures as well; records and picture infos are compared throughout."""
    from jsmpeg_b200 import decoder
    olib = helpers.oracle_lib()
    d = decoder.MPEG1Video({"decodeFirstFrame": False}, lib=olib)
    d.write(0, [es])
    seq = olib.oracle_seq_params(d.decoder).contents
    mb = seq.mb_size
    lib = emu_lib()
    lib.emu_set_quant(bytes(seq.intra_q), bytes(seq.non_intra_q))
    vp = ctypes.c_void_p
    lib.emu_walk_picture_b.argtypes = [vp, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_int, ctypes.c_int, vp, vp, vp]
    lib.emu_expand_picture.argtypes = [vp, ctypes.c_uint32, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp]
    lib.emu_reconstruct_picture.argtypes = [vp, vp, vp, vp, ctypes.c_int, ctypes.c_int]
    lib.emu_reconstruct_picture_b.argtypes = [vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int]
    mbw, mbh = stream_geometry(es)
    buf = np.frombuffer(es + b"\0" * 16, dtype=np.uint8).copy()
    ysize = mb * 256
    size = ysize * 3 // 2 + mbw * 16 + 64
    planes = [np.zeros(size, dtype=np.uint8) for _ in range(2)]
    planes_b = [np.zeros(size, dtype=np.uint8) for _ in range(2)]
    cur = b_cur = 0
    n_b = checked = 0
    compare_planes = True
    while d.decode():
        info = olib.oracle_last_picture_info(d.decoder).contents
        want_hdr = np.ctypeslib.as_array(ctypes.cast(olib.oracle_last_mb_records(d.decoder), ctypes.POINTER(ctypes.c_uint32)),
                                         shape=(mb, 4)).copy()
        hdr = np.zeros(mb * 4, dtype=np.uint32)
        park = np.zeros(mb * 6 * 2, dtype=np.uint32)
        coef = np.zeros(mb * 6 * 32, dtype=np.uint32)
        pinfo = np.zeros(12, dtype=np.int32)
        is_b = ((es[info.start_byte + 1] >> 3) & 7) == 3  # the host's routing (engine.cu: decode_round)
        if is_b:
            lib.emu_walk_picture_b(buf.ctypes.data, len(es), info.start_byte, mbw, mbh, hdr.ctypes.data, park.ctypes.data, pinfo.ctypes.data)
        else:
            lib.emu_walk_picture(buf.ctypes.data, len(es), info.start_byte, mbw, mbh, hdr.ctypes.data, park.ctypes.data, pinfo.ctypes.data, 1)
        # (damaged: a block that runs past coefficient 63 AND then meets an invalid code is PARSE_ERR_COEF_INDEX to the
        # oracle and PARSE_ERR_INVALID_VLC to the walks, which flag the index when a block ends -- an error either way)
        assert (pinfo[1], pinfo[2], pinfo[3], pinfo[8] if not damaged else bool(pinfo[8]), pinfo[10]) == \
               (info.end_bit, info.status, info.picture_type, info.error if not damaged else bool(info.error), info.reserved[1]), \
               f"{name}: picture {checked}: info"
        if not damaged:  # (the two counters are statistics: where a damaged stream makes slices revisit addresses the
            #              walks count every visit, the oracle every address -- I/P pictures as well)
            assert (pinfo[6], pinfo[7]) == (info.n_present, info.n_coded_blocks), f"{name}: picture {checked}: counters"
        if pinfo[2] != 1:
            checked += 1
            continue
        assert np.array_equal(hdr.reshape(mb, 4), want_hdr), \
            f"{name}: picture {checked} (type {info.picture_type}): records differ at mb {np.nonzero((hdr.reshape(mb, 4) != want_hdr).any(axis=1))[0][:8]}"
        lib.emu_expand_picture(buf.ctypes.data, len(es), mbw, mbh, hdr.ctypes.data, park.ctypes.data, coef.ctypes.data, pinfo.ctypes.data)
        if is_b:
            out = planes_b[b_cur]
            lib.emu_reconstruct_picture_b(hdr.ctypes.data, coef.ctypes.data, out.ctypes.data, planes[cur].ctypes.data,
                                          planes[cur ^ 1].ctypes.data, mbw, mbh)
            b_cur ^= 1
            n_b += 1
        else:
            out = planes[cur]
            lib.emu_reconstruct_picture(hdr.ctypes.data, coef.ctypes.data, out.ctypes.data, planes[cur ^ 1].ctypes.data, mbw, mbh)
            cur ^= 1
        y, cr, cb = d.planes()
        if damaged and info.error:
            compare_planes = False
        for pname, got, want in (("Y", out[:ysize], y), ("Cr", out[ysize:ysize + ysize // 4], cr), ("Cb", out[ysize + ysize // 4:ysize * 3 // 2], cb)):
            if compare_planes and not np.array_equal(got, want):
                bad = np.nonzero(got != want)[0]
                raise AssertionError(f"{name}: picture {checked} (type {info.picture_type}) plane {pname}: {len(bad)} bytes differ, first {bad[:6]}")
        checked += 1
    d.destroy()
    return checked, n_b


@pytest.mark.parametrize("name", sorted(synth_es.B_CASES))
def test_b_device_code_matches_the_oracle_on_syntax_cases(oracle_b, name):
    es = synth_es.make_case(name)
    checked, n_b = _emulated_b_pipeline(es, name)
    assert checked == len(picture_starts(es)) and n_b == picture_types(es).count(3) > 0


@pytest.mark.parametrize("form", range(len(VECTOR_FORMS)))
def test_b_device_code_matches_the_oracle_on_a_natural_clip(oracle_b, form):
    pytest.importorskip("cv2")
    f_codes, full_pel = VECTOR_FORMS[form]
    es, types, order, stats = natural_clip(frames=13 if form == 0 else 10, f_codes=f_codes, full_pel=full_pel)
    checked, n_b = _emulated_b_pipeline(es, f"mini_enc 176x144 {f_codes} {full_pel}")
    assert checked == len(types) and n_b == types.count(3)


def test_b_device_code_on_one_slice_pictures(oracle_b):
    """One slice per picture (FFmpeg's layout): the I/P pictures take the lane-parallel walk proper (sub-sequences of
    one long slice), the B pictures one long chain each, skipped runs cross macroblock rows."""
    pytest.importorskip("cv2")
    es, types, order, stats = natural_clip(frames=10, one_slice=True)
    checked, n_b = _emulated_b_pipeline(es, "mini_enc 176x144, one slice per picture")
    assert checked == len(types) and n_b == types.count(3) > 0


FIXTURE_720P = os.path.join(HERE, "fixtures", "b_clip_1280x720.m1v")  # tools/mini_enc.py: make_b_clip(1280, 720, 13, 2, seed=1234)


def test_b_device_code_matches_the_oracle_at_720p(oracle_b):
    """The committed 1280x720 I/P/B clip (the one tools/time_b.py times on the GPU): 13 pictures, 8 of them B."""
    es = open(FIXTURE_720P, "rb").read()
    checked, n_b = _emulated_b_pipeline(es, "fixture 720p")
    assert (checked, n_b) == (13, 8)


def test_fixture_hashes_are_the_oracles(oracle_b):
    """tests/fixtures/b_clip_1280x720.json (what bench.py's b_pictures_720p leg and tools/time_b.py compare the GPU's
    pictures with) holds the oracle's picture hashes and bit indices."""
    import json

    import bench
    meta = json.load(open(FIXTURE_720P.replace(".m1v", ".json")))
    es = open(FIXTURE_720P, "rb").read()
    frames, idx, d = helpers.decode_all(oracle_b, [(0, es)])
    assert picture_types(es) == meta["picture_types"] and idx == meta["bit_index_after"]
    assert [format(bench.fnv1a64_planes(*f), "016x") for f in frames] == meta["fnv1a64"]
    d.destroy()


def test_b_walk_on_damaged_streams_matches_the_oracle(oracle_b):
    """Bit flips and a truncation in B-picture streams: the walk stops where the oracle's stops (same records, same
    end_bit, same error), stage 2 stays inside its planes."""
    rng = np.random.default_rng(9)
    es = synth_es.make_case("b_one_slice_fcodes")
    for trial in range(5):
        bad = bytearray(es)
        for pos in rng.integers(200, len(es), size=3):
            bad[pos] ^= 1 << int(rng.integers(0, 8))
        _emulated_b_pipeline(bytes(bad), f"corrupt {trial}", damaged=True)
    _emulated_b_pipeline(es[: len(es) * 3 // 5], "truncated", damaged=True)


def _random_knobs(rng):
    w = int(rng.integers(2, 14)) * 16 - int(rng.integers(0, 2)) * int(rng.integers(1, 15))
    h = int(rng.integers(2, 10)) * 16 - int(rng.integers(0, 2)) * int(rng.integers(1, 15))
    return dict(width=max(w, 17), height=max(h, 17), pictures=int(rng.integers(5, 12)), gop=int(rng.integers(1, 4)),
                slices=str(rng.choice(["one", "rows", "random"])), b_frames=int(rng.integers(1, 4)),
                f_codes=tuple(int(x) for x in rng.integers(1, 8, size=3)), b_f_codes=tuple(int(x) for x in rng.integers(1, 8, size=3)),
                full_pel_prob=float(rng.choice([0, 0.3, 1.0])), b_skip_prob=float(rng.choice([0, 0.2, 0.6])),
                b_intra_prob=float(rng.choice([0, 0.1, 0.5])), skip_prob=float(rng.choice([0, 0.15, 0.5])),
                stuffing_prob=float(rng.choice([0, 0.2])), escape_prob=float(rng.choice([0.05, 0.4])),
                custom_matrices=bool(rng.integers(0, 2)), max_coefs=int(rng.integers(1, 30)),
                slice_gap_prob=float(rng.choice([0, 0.3])), extension_user_data=bool(rng.integers(0, 2)))


@pytest.mark.parametrize("seed", [101, 102])
def test_random_streams_clean_and_damaged(oracle_b, seed):
    """A slice of the randomised campaign run during development (700 random knob sets x (clean + 2 bit-flipped copies),
    no difference): random sizes incl. non-multiples of 16, 1-3 B pictures between references, every f_code, full-pel,
    slice layouts, skipped runs, stuffing, escapes, custom matrices.  The B-picture device pipeline against the oracle
    (planes on clean streams; records, end_bit and error presence on damaged ones), and the three lane-parallel modes
    plus the slice walk against the serial walk."""
    from test_walk_emu import check_stream
    rng = np.random.default_rng(seed)
    for trial in range(8):
        knobs = _random_knobs(rng)
        es = synth_es.SynthStream(synth_es.Knobs(**knobs), int(rng.integers(0, 1 << 30))).generate()
        name = f"seed {seed} trial {trial} {knobs}"
        _emulated_b_pipeline(es, name)
        check_stream(emu_lib(), es, name)
        bad = bytearray(es)
        for pos in rng.integers(64, len(es), size=int(rng.integers(1, 6))):
            bad[pos] ^= 1 << int(rng.integers(0, 8))
        bad = bytes(bad)
        if bad.find(b"\x00\x00\x01\xb3") < 0:
            continue
        mbw, mbh = stream_geometry(bad)
        if 0 < mbw * mbh <= 4000:
            _emulated_b_pipeline(bad, name + " (bit flips)", damaged=True)
