"""Pin the oracle to the reference: every plane byte of every picture and every bit index must equal what the
unmodified reference C (src/wasm/mpeg1.c + buffer.c) produced on the same streams.  The reference's results are
recorded in tests/golden/reference/decodes.json (tools/make_reference_golden.py runs the reference to write it)."""
import numpy as np
import pytest

import helpers
import synth_es


@pytest.mark.parametrize("name", sorted(synth_es.CASES))
def test_synthetic_syntax_corners(name):
    es = synth_es.make_case(name)
    orc_frames, orc_idx, od = helpers.decode_all(helpers.oracle_lib(), [(0.0, es)])
    helpers.assert_matches_reference(f"synth/{name}", orc_frames, orc_idx, es)
    assert len(orc_frames) >= 6
    od.destroy()


def random_syntax_stream(seed):
    k = synth_es.Knobs(width=int(16 * (2 + seed)), height=int(16 * (1 + seed % 3)) + 2 * seed, pictures=7, gop=3,
                       slices=["one", "rows", "random"][seed % 3], slice_gap_prob=0.2, stuffing_prob=0.2,
                       skip_prob=0.3, f_codes=(1, 2, 3, 4), full_pel_prob=0.3, escape_prob=0.3,
                       custom_matrices=bool(seed & 1), extension_user_data=True, ignored_pictures=bool(seed & 2))
    return synth_es.SynthStream(k, 1000 + seed).generate()


@pytest.mark.parametrize("seed", range(6))
def test_random_syntax_streams(seed):
    """Random streams (not the committed ones): all corner knobs on at once."""
    es = random_syntax_stream(seed)
    orc_frames, orc_idx, od = helpers.decode_all(helpers.oracle_lib(), [(0.0, es)])
    helpers.assert_matches_reference(f"random/{seed}", orc_frames, orc_idx, es)
    od.destroy()


@pytest.mark.parametrize("w,h,n", [(320, 240, 24), (1280, 720, 6)])
def test_ffmpeg_clips(w, h, n):
    packets = helpers.clip_packets(w, h, n)
    orc_frames, orc_idx, od = helpers.decode_all(helpers.oracle_lib(), packets)
    assert len(orc_frames) == n
    helpers.assert_matches_reference(f"ffmpeg/{w}x{h}x{n}", orc_frames, orc_idx, b"".join(p for _, p in packets))
    od.destroy()


def decode_streaming(lib, packets):
    """EVICT mode with a small buffer, write-a-packet / decode-what-is-there, like the reference player's
    streaming loop (src/player.js:222-229).  Returns (frames, bit index after every decode)."""
    from jsmpeg_b200 import decoder
    d = decoder.MPEG1Video({"streaming": True, "videoBufferSize": 64 * 1024, "decodeFirstFrame": False}, lib=lib)
    rec = decoder.PlaneRecorder()
    d.connect(rec)
    trace = []
    for pts, payload in packets:
        d.write(pts, [payload])
        while d.decode():
            trace.append(d.bufferGetIndex())
    d.destroy()
    return rec.frames, trace


def test_streaming_evict_mode_matches_reference():
    """EVICT streaming: same pictures, same indices as the reference."""
    packets = helpers.clip_packets(320, 240, 24)
    orc_frames, orc_trace = decode_streaming(helpers.oracle_lib(), packets)
    helpers.assert_matches_reference("evict/320x240x24", orc_frames, orc_trace, b"".join(p for _, p in packets))
    assert len(orc_frames) >= 20


def test_stats_of_synthetic_cases_cover_the_corners():
    """The committed corner streams really contain what their names promise (checked on the
    oracle's records)."""
    import ctypes
    lib = helpers.oracle_lib()
    from jsmpeg_b200 import decoder
    seen = dict(skipped=0, intra_in_p=0, dc_only=0, absent=0, mv_odd_h=0, mv_odd_v=0, ignored=0)
    for name in ("skips_stuffing_escape_mba", "random_slices_gaps", "fcodes_fullpel", "ignored_pictures_userdata"):
        d = decoder.MPEG1Video({"decodeFirstFrame": False}, lib=lib)
        d.write(0.0, [synth_es.make_case(name)])
        mb_size = lib.oracle_seq_params(d.decoder).contents.mb_size
        while d.decode():
            info = lib.oracle_last_picture_info(d.decoder).contents
            if info.status != 1:
                seen["ignored"] += 1
                continue
            h = np.ctypeslib.as_array(ctypes.cast(lib.oracle_last_mb_records(d.decoder), ctypes.POINTER(ctypes.c_uint8)),
                                      shape=(mb_size, 16))
            flags = h[:, 4]
            mv = h[:, :4].copy().view(np.int16)
            seen["skipped"] += int(((flags & 4) != 0).sum())
            seen["absent"] += int(((flags & 1) == 0).sum())
            seen["dc_only"] += int((h[:, 6] != 0).sum())
            if info.picture_type == 2:
                seen["intra_in_p"] += int(((flags & 2) != 0).sum())
                seen["mv_odd_h"] += int((mv[:, 0] & 1).sum())
                seen["mv_odd_v"] += int((mv[:, 1] & 1).sum())
        d.destroy()
    assert all(v > 0 for v in seen.values()), seen
