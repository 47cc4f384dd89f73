"""GPU parity: the CUDA path (through the C ABI) against the oracle, bit-exact.

Every test here needs a B200 (``-m gpu``).  The oracle (oracle/liboracle.so, our CPU restatement
pinned to the reference by tests/test_oracle_vs_reference.py) and the reference's own decodes, recorded in
tests/golden/reference, are the checkers.
"""
import ctypes

import numpy as np
import pytest

import helpers
from helpers import assert_frames_equal, assert_matches_reference, clip_packets, decode_all, oracle_lib
from jsmpeg_b200 import capi
from jsmpeg_b200.batch import OUT_DEVICE, OUT_HOST, BatchDecoder

pytestmark = pytest.mark.gpu

SIZES = [(320, 240, 24), (1280, 720, 14)]


def _oracle_pictures(packets, n):
    """Decode n pictures with the oracle and capture, per picture, its records and planes."""
    lib = oracle_lib()
    from jsmpeg_b200 import decoder
    d = decoder.MPEG1Video({"decodeFirstFrame": False}, lib=lib)
    for pts, p in packets:
        d.write(pts, [p])
    seq = lib.oracle_seq_params(d.decoder).contents
    mb_size = seq.mb_size
    out = []
    while len(out) < n:
        start_index = d.bufferGetIndex()
        if not d.decode():
            break
        info = lib.oracle_last_picture_info(d.decoder).contents
        hdr = np.ctypeslib.as_array(ctypes.cast(lib.oracle_last_mb_records(d.decoder), ctypes.POINTER(ctypes.c_uint8)),
                                    shape=(mb_size * 16,)).copy()
        coef = np.ctypeslib.as_array(ctypes.cast(lib.oracle_last_coefficients(d.decoder), ctypes.POINTER(ctypes.c_int16)),
                                     shape=(mb_size * 384,)).copy()
        planes = tuple(p.copy() for p in d.planes())
        out.append(dict(start_byte=info.start_byte, end_bit=info.end_bit, status=info.status,
                        type=info.picture_type, n_coded=info.n_coded_blocks, n_present=info.n_present,
                        hdr=hdr, coef=coef, planes=planes))
    return d, seq, out


def _coded_mask(hdr, mb_size):
    """Boolean mask over the int16 coefficient plane: blocks whose cbp bit is set."""
    h = hdr.reshape(mb_size, 16)
    present = (h[:, 4] & 1).astype(bool)
    cbp = h[:, 5]
    mask = np.zeros((mb_size, 6, 64), bool)
    for blk in range(6):
        mask[:, blk, :] = (present & ((cbp & (0x20 >> blk)) != 0))[:, None]
    return mask.reshape(-1)


@pytest.mark.parametrize("w,h,n", SIZES)
def test_stage1_parse_matches_oracle_records(w, h, n):
    packets = clip_packets(w, h, n)
    es = b"".join(p for _, p in packets)
    d, seq, pics = _oracle_pictures(packets, n)
    lib = capi.product_library()
    mbw, mbh = (w + 15) // 16, (h + 15) // 16
    mb_size = mbw * mbh
    iq = bytes(seq.intra_q)
    nq = bytes(seq.non_intra_q)
    for k, pic in enumerate(pics):
        info = helpers.PictureInfo()
        hdr = np.zeros(mb_size * 16, np.uint8)
        coef = np.zeros(mb_size * 384, np.int16)
        rc = lib.jsmpeg_b200_debug_parse_picture(es, len(es), pic["start_byte"], mbw, mbh, iq, nq,
                                                 ctypes.addressof(info), hdr.ctypes.data, coef.ctypes.data)
        assert rc == 0
        assert (info.status, info.picture_type, info.end_bit) == (pic["status"], pic["type"], pic["end_bit"]), k
        assert info.error == 0
        assert info.n_coded_blocks == pic["n_coded"] and info.n_present == pic["n_present"]
        # header bytes 0..7 are the contract (mv, flags, cbp, dc_only, qscale); 8.. are diagnostics
        got = hdr.reshape(mb_size, 16)[:, :8]
        exp = pic["hdr"].reshape(mb_size, 16)[:, :8]
        assert np.array_equal(got, exp), f"picture {k}: macroblock headers differ at {np.nonzero((got != exp).any(1))[0][:8]}"
        m = _coded_mask(pic["hdr"], mb_size)
        assert np.array_equal(coef[m], pic["coef"][m]), f"picture {k}: coefficients differ"
    d.destroy()


@pytest.mark.parametrize("w,h,n", SIZES)
def test_stage2_reconstruct_matches_oracle_planes(w, h, n):
    packets = clip_packets(w, h, n)
    d, seq, pics = _oracle_pictures(packets, n)
    lib = capi.product_library()
    mbw, mbh = (w + 15) // 16, (h + 15) // 16
    ysz = mbw * mbh * 256
    fwd = (np.zeros(ysz, np.uint8), np.zeros(ysz // 4, np.uint8), np.zeros(ysz // 4, np.uint8))
    prev2 = tuple(p.copy() for p in fwd)
    for k, pic in enumerate(pics):
        cur = tuple(p.copy() for p in prev2)  # ping-pong: the set written now held picture k-2
        rc = lib.jsmpeg_b200_debug_reconstruct(mbw, mbh, pic["hdr"].ctypes.data, pic["coef"].ctypes.data,
                                               fwd[0].ctypes.data, fwd[1].ctypes.data, fwd[2].ctypes.data,
                                               cur[0].ctypes.data, cur[1].ctypes.data, cur[2].ctypes.data)
        assert rc == 0
        assert_frames_equal([cur], [pic["planes"]], f"stage 2, picture {k}")
        prev2, fwd = fwd, cur
    d.destroy()


@pytest.mark.parametrize("w,h,n", SIZES + [(1920, 1080, 5)])
def test_reference_abi_whole_clip_bit_exact(w, h, n):
    """write everything, decode() until false: planes and bit indices identical to the oracle
    and to the reference (its decode recorded in tests/golden/reference/decodes.json)."""
    packets = clip_packets(w, h, n)
    exp_frames, exp_idx, od = decode_all(oracle_lib(), packets)
    got_frames, got_idx, gd = decode_all(capi.product_library(), packets)
    assert got_idx == exp_idx
    assert_frames_equal(got_frames, exp_frames, "CUDA vs oracle")
    assert (gd.width, gd.height, gd.codedSize, gd.frameRate) == (od.width, od.height, od.codedSize, od.frameRate)
    assert abs(gd.decodedTime - od.decodedTime) < 1e-9
    assert_matches_reference(f"ffmpeg/{w}x{h}x{n}", got_frames, got_idx, b"".join(p for _, p in packets))
    od.destroy()
    gd.destroy()


def test_batch_streams_are_independent_and_bit_exact():
    """4 streams (different seeds and sizes) decoded together, device-resident, against the oracle."""
    specs = [(320, 240, 12, 1), (320, 240, 12, 2), (352, 288, 10, 3), (640, 368, 8, 4)]
    clips = [clip_packets(w, h, n, seed=s) for (w, h, n, s) in specs]
    bd = BatchDecoder(len(specs))
    for i, packets in enumerate(clips):
        bd.write(i, b"".join(p for _, p in packets))
    expected = [decode_all(oracle_lib(), packets)[0] for packets in clips]
    step = 0
    while True:
        got = bd.decode(1, OUT_DEVICE)
        if got == 0:
            break
        for i, frames in enumerate(expected):
            if step < len(frames):
                assert_frames_equal([bd.read_planes(i)], [frames[step]], f"stream {i} picture {step}")
        step += 1
    assert step == max(len(f) for f in expected)
    st = bd.stats()
    assert st["pictures"] == sum(len(f) for f in expected)
    assert st["parse_errors"] == 0
    bd.close()


def test_batch_multi_picture_steps_and_host_output():
    """decode(n>1): several pictures per call, copied out to the host ring; the last picture of
    every call is checked, and a rewind reproduces the same pictures."""
    packets = clip_packets(320, 240, 24)
    exp, _, od = decode_all(oracle_lib(), packets)
    bd = BatchDecoder(2)
    es = b"".join(p for _, p in packets)
    bd.write(0, es)
    bd.write(1, es)
    for rnd in range(2):
        done = 0
        for n in (1, 3, 5, 24):
            got = bd.decode(n, OUT_HOST)
            assert got % 2 == 0
            done += got // 2
            if got:
                for s in range(2):
                    assert_frames_equal([tuple(p.copy() for p in bd.host_planes(s))], [exp[done - 1]], f"round {rnd} picture {done - 1}")
        assert done == len(exp)
        bd.rewind()
    od.destroy()
    bd.close()


# ---- golden vectors produced by the reference itself (tests/golden, tools/make_golden.py) -------

import test_oracle_golden as golden  # noqa: E402


@pytest.mark.parametrize("name", golden.CASES)
def test_cuda_matches_reference_golden(name):
    """Every syntax-corner stream and FFmpeg clip in tests/golden through the reference ABI on the
    GPU: bit indices and plane checksums identical to what the reference C produced."""
    golden.check_against_golden(capi.product_library(), name)


@pytest.mark.parametrize("name", ["rows_ip", "random_slices_gaps", "ffmpeg_176x144_ip"])
def test_cuda_golden_chunked_writes(name):
    golden.check_against_golden(capi.product_library(), name, chunked=True)


def test_streaming_evict_interleaved_write_decode():
    """EVICT mode, 64 KiB buffer, write one PES packet then decode() until false -- the reference
    player's streaming loop (src/player.js:222-229).  Exercises eviction (index shifts, mirror
    re-upload), look-ahead invalidation and pictures that are complete only after a later write."""
    packets = clip_packets(320, 240, 24)
    opts = {"streaming": True, "videoBufferSize": 64 * 1024, "decodeFirstFrame": False}

    def run(lib):
        from jsmpeg_b200 import decoder
        d = decoder.MPEG1Video(opts, lib=lib)
        rec = decoder.PlaneRecorder()
        d.connect(rec)
        trace = []
        for pts, payload in packets:
            d.write(pts, [payload])
            while d.decode():
                trace.append(d.bufferGetIndex())
        d.destroy()
        return rec.frames, trace

    exp_frames, exp_trace = run(oracle_lib())
    got_frames, got_trace = run(capi.product_library())
    assert got_trace == exp_trace
    assert_frames_equal(got_frames, exp_frames, "EVICT streaming")


def test_partial_picture_then_more_data():
    """A picture cut in the middle is decoded as far as the data goes (SURVEY Q15); after the rest
    arrives and the index is set back, the full picture must come out -- the parsed-ahead records
    of the truncated attempt must not be reused."""
    packets = clip_packets(320, 240, 4)
    es = b"".join(p for _, p in packets)
    cut = len(packets[0][1]) + len(packets[1][1]) // 2

    def run(lib):
        from jsmpeg_b200 import decoder
        d = decoder.MPEG1Video({"decodeFirstFrame": False}, lib=lib)
        out = []
        d.write(0.0, [es[:cut]])
        while d.decode():
            out.append((d.bufferGetIndex(), tuple(p.copy() for p in d.planes())))
        d.write(0.1, [es[cut:]])
        d.bufferSetIndex(len(packets[0][1]) * 8)  # back to the start of picture 1
        while d.decode():
            out.append((d.bufferGetIndex(), tuple(p.copy() for p in d.planes())))
        d.destroy()
        return out

    exp = run(oracle_lib())
    got = run(capi.product_library())
    assert [i for i, _ in got] == [i for i, _ in exp]
    assert_frames_equal([f for _, f in got], [f for _, f in exp], "partial picture")
    assert len(exp) == 2 + 3


def _canvas2d_rgba(y, cr, cb, width, height):
    """numpy restatement of the reference's integer renderer (src/canvas2d.js:53-122); the
    renderer's `cb` parameter receives the decoder's Cr plane and vice versa (SURVEY Q8)."""
    cw = ((width + 15) >> 4) << 4
    Y = y.reshape(-1, cw).astype(np.int32)
    hw = cw >> 1
    CR = cr.reshape(-1, hw).astype(np.int32)
    CB = cb.reshape(-1, hw).astype(np.int32)
    out = np.full((height, width, 4), 255, np.uint8)
    cols, rows = width >> 1, height >> 1
    ccb = CR[:rows, :cols]  # what the renderer calls cb
    ccr = CB[:rows, :cols]
    r = (ccb + ((ccb * 103) >> 8)) - 179
    g = ((ccr * 88) >> 8) - 44 + ((ccb * 183) >> 8) - 91
    b = (ccr + ((ccr * 198) >> 8)) - 227
    for dy in range(2):
        for dx in range(2):
            yy = Y[dy:rows * 2:2, dx:cols * 2:2]
            out[dy:rows * 2:2, dx:cols * 2:2, 0] = np.clip(yy + r, 0, 255)
            out[dy:rows * 2:2, dx:cols * 2:2, 1] = np.clip(yy - g, 0, 255)
            out[dy:rows * 2:2, dx:cols * 2:2, 2] = np.clip(yy + b, 0, 255)
    return out


@pytest.mark.parametrize("name", ["ffmpeg_176x144_ip", "odd_size"])
def test_rgba_epilogue_matches_canvas2d_formula(name):
    from jsmpeg_b200.batch import OUT_RGBA
    es, info = golden.load_case(name)
    bd = BatchDecoder(1)
    bd.write(0, es)
    n = 0
    while bd.decode(1, OUT_RGBA):
        y, cr, cb = bd.read_planes(0)
        got = bd.read_rgba(0)
        exp = _canvas2d_rgba(y, cr, cb, info["width"], info["height"])
        assert np.array_equal(got, exp), f"{name}: RGBA picture {n} differs"
        n += 1
    assert n >= 6
    bd.close()


# ---- MPEG-TS demux on the device (SURVEY section 8f rank 1) ---------------------------------------

def test_device_ts_demux_matches_host_demuxer_and_decodes_bit_exact():
    """jsmpeg_b200_batch_write_ts against the host mirror of src/ts.js (jsmpeg_b200/ts.py): same
    elementary stream, same PES table (offsets + PTS), and the decoded pictures equal the oracle's."""
    import gen_streams
    from jsmpeg_b200 import ts
    data = gen_streams.make_clip_ts(320, 240, 24, seed=1234, noise=9)
    packets = ts.demux_video_es(data)
    es = b"".join(p for _, p in packets)
    bd = BatchDecoder(2)
    total, pes = bd.write_ts(0, data)
    assert total == len(es)
    # stream 1: the same clip in two pieces, the second after an ordinary write (mixed residency)
    cut = (len(data) // 188 // 2) * 188
    first_pes = [p for p in ts.demux_video_es(data[:cut])]
    t1, pes1 = bd.write_ts(1, data[:cut])
    t2, pes2 = bd.write_ts(1, data[cut:])
    assert t1 + t2 == len(es)
    # PES table: offsets are the running payload sizes, PTS as the host demuxer reports them
    offsets, acc = [], 0
    for _, p in packets:
        offsets.append(acc)
        acc += len(p)
    assert [o for o, _ in pes] == offsets
    assert all(abs(a - b) < 1e-9 for (_, a), (b, _) in zip(pes, packets))
    assert [o for o, _ in pes1 + pes2][:len(first_pes)] == offsets[:len(first_pes)]
    exp_frames, exp_idx, od = decode_all(oracle_lib(), packets)
    n = 0
    while bd.decode(1, OUT_DEVICE):
        for s in range(2):
            assert_frames_equal([bd.read_planes(s)], [exp_frames[n]], f"TS stream {s} picture {n}")
        n += 1
    assert n == len(exp_frames)
    assert bd.get_index(0) == exp_idx[-1] == bd.get_index(1)
    od.destroy()
    bd.close()


def test_device_ts_demux_resyncs_on_unaligned_input_and_decodes_bit_exact():
    """Three bytes of garbage in front of the clip, an odd chunking: the device demuxer finds the packet grid the
    way src/ts.js:155-189 does, carries partial packets over (ts.js:25-41), and the pictures decode bit-exact."""
    import gen_streams
    from jsmpeg_b200 import ts
    data = gen_streams.make_clip_ts(176, 144, 6, seed=3, noise=4)
    packets = ts.demux_video_es(data)
    es = b"".join(p for _, p in packets)
    dirty = b"\x00\x01\x02" + data
    bd = BatchDecoder(1)
    total = 0
    for o in range(0, len(dirty), 1777):
        total += bd.write_ts(0, dirty[o:o + 1777])[0]
    assert total == len(es)
    exp_frames, exp_idx, od = decode_all(oracle_lib(), packets)
    n = 0
    while bd.decode(1, OUT_DEVICE):
        assert_frames_equal([bd.read_planes(0)], [exp_frames[n]], f"resynced TS picture {n}")
        n += 1
    assert n == len(exp_frames) and bd.get_index(0) == exp_idx[-1]
    od.destroy()
    bd.close()


# ---- robustness: garbage in must be memory-safe and must terminate (SURVEY section 5) -------------

@pytest.mark.parametrize("seed", range(4))
def test_corrupted_streams_terminate_and_stay_in_bounds(seed):
    """Random byte corruption after the sequence header.  The reference gives no defined output for
    such streams (undefined table reads, SURVEY section 5), so only the contract is checked:
    decode() keeps returning (no hang, no fault), one call per picture start code at most, and a
    following clean stream on the same GPU still decodes bit-exactly."""
    rng = np.random.default_rng(100 + seed)
    es = bytearray(golden.load_case(["ffmpeg_176x144_ip", "rows_ip", "fcodes_fullpel", "skips_stuffing_escape_mba"][seed])[0])
    n_flip = max(8, len(es) // 200)
    for pos in rng.integers(64, len(es), n_flip):
        es[pos] = int(rng.integers(0, 256))
    if seed == 1:
        es = es[:len(es) // 2]  # and a truncated tail
    es = bytes(es)
    starts = es.count(b"\x00\x00\x01\x00")
    bd = BatchDecoder(1)
    bd.write(0, es)
    calls = 0
    while bd.decode(1, OUT_HOST):
        calls += 1
        assert calls <= starts + 1
    assert bd.get_index(0) <= len(es) * 8
    bd.close()
    golden.check_against_golden(capi.product_library(), "rows_ip")


# ---- both walks of stage 1a against the same checkers ---------------------------------------------

def test_clean_clip_is_walked_by_the_lane_parallel_walk():
    """Default configuration: the lane-parallel walk, not its serial fall-back, produces every picture
    of a clean clip (a silent fall-back would still be bit-exact, only slow)."""
    import os
    if os.environ.get("JSMPEG_B200_WALK") == "serial":
        pytest.skip("serial walk selected")
    es = b"".join(p for _, p in clip_packets(640, 480, 13))
    bd = BatchDecoder(1)
    bd.write(0, es)
    n = bd.decode(13, OUT_DEVICE)
    st = bd.stats()
    bd.close()
    assert n == 13 and st["lane_walk_pictures"] == 13, (n, st["lane_walk_pictures"])


def test_serial_walk_in_a_child_process():
    """The walk variant is chosen once per process (first launch), so the stage-1 record parity, the
    golden streams, a whole-clip decode and the corrupted-stream contract are repeated in a child
    process with JSMPEG_B200_WALK=serial (the one-chain-per-warp walk the lane-parallel one falls back
    to inside the same kernel)."""
    import os
    import subprocess
    import sys
    if os.environ.get("JSMPEG_B200_WALK") == "serial":
        pytest.skip("already running with the serial walk")
    env = dict(os.environ, JSMPEG_B200_WALK="serial")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-x", "-q", "-p", "no:cacheprovider",
                        "-k", "stage1_parse or golden or whole_clip or corrupted"],
                       env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
