"""GPU parity of the B-picture extension: the CUDA path (through the C ABI) against the oracle, bit-exact.

The oracle's B-picture path has no reference to be pinned to (the reference skips B pictures); it is
cross-checked against FFmpeg's decoder in tests/test_b_pictures.py, where the same device code is also emulated
on the host.  Here the real kernels run: walk_pictures_b_kernel, expand_blocks_kernel, reconstruct_b_kernel,
reconstruct_rgba_b_kernel, and the engine's routing / plane bookkeeping.
"""
import numpy as np
import pytest

import helpers
import synth_es
from helpers import assert_frames_equal, clip_packets, decode_all
from jsmpeg_b200 import capi
from jsmpeg_b200.batch import OUT_DEVICE, OUT_HOST, OUT_RGBA, BatchDecoder
from test_b_pictures import natural_clip, picture_types

pytestmark = pytest.mark.gpu


@pytest.fixture
def oracle_b():
    lib = helpers.oracle_lib()
    lib.oracle_set_decode_b(1)
    yield lib
    lib.oracle_set_decode_b(0)


def _streams():
    out = {name: synth_es.make_case(name) for name in synth_es.B_CASES}
    out["natural_176x144"] = natural_clip()[0]
    return out


@pytest.mark.parametrize("name", sorted(synth_es.B_CASES) + ["natural_176x144"])
def test_reference_abi_decodes_b_pictures_bit_exact(oracle_b, name):
    """decodeBPictures through the 15-function ABI: every picture (I, P and B, coded order) and every bit index
    equal to the oracle's; lastPicture() reports type and temporal_reference of each."""
    es = _streams()[name]
    types = picture_types(es)
    exp, exp_idx, od = decode_all(oracle_b, [(0, es)])
    got, got_idx, gd = decode_all(capi.product_library(), [(0, es)], options={"decodeBPictures": True})
    assert got_idx == exp_idx
    assert_frames_equal(got, exp, f"{name}: CUDA vs oracle (B pictures decoded)")
    assert len(got) == len(types) and types.count(3) > 0
    assert gd.lastPicture()[0] == types[-1]
    od.destroy()
    gd.destroy()


def test_display_order_rendering(oracle_b):
    """decodeBPictures + displayOrder of the host class over the CUDA library: the destination receives the oracle's
    pictures in display order, lastPicture() reports the same (type, temporal_reference) sequence."""
    from jsmpeg_b200 import decoder
    es, types, order, _ = natural_clip()
    runs = []
    for lib in (oracle_b, capi.product_library()):
        d = decoder.MPEG1Video({"decodeFirstFrame": False, "decodeBPictures": True, "displayOrder": True}, lib=lib)
        rec = decoder.PlaneRecorder()
        d.connect(rec)
        d.write(0, [es])
        seen = []
        while d.decode():
            seen.append(d.lastPicture())
        d.flush()
        runs.append((seen, rec.frames))
        d.destroy()
    assert runs[0][0] == runs[1][0] == list(zip(types, order))
    assert_frames_equal(runs[1][1], runs[0][1], "display order: CUDA vs oracle")


def test_extension_off_is_the_reference_behaviour():
    """Default: a B picture is consumed and nothing is decoded -- identical to the compiled reference."""
    es = synth_es.make_case("b_rows")
    lib = helpers.oracle_lib()
    lib.oracle_set_decode_b(0)
    exp, exp_idx, od = decode_all(lib, [(0, es)])
    got, got_idx, gd = decode_all(capi.product_library(), [(0, es)])
    assert got_idx == exp_idx
    assert_frames_equal(got, exp, "b_rows, extension off")
    helpers.assert_matches_reference("b_rows/extension_off", got, got_idx, es, first=1)
    od.destroy()
    gd.destroy()


def test_batch_mixes_b_streams_and_ip_streams(oracle_b):
    """B streams of different sizes and GOP shapes next to a plain I/P clip in one batch: a reconstruct step then
    holds I/P pictures of some streams and B pictures of others.  Device output, picture by picture."""
    streams = _streams()
    names = sorted(streams)
    data = [streams[n] for n in names] + [b"".join(p for _, p in clip_packets(320, 240, 8))]
    expected = [decode_all(oracle_b, [(0, es)])[0] for es in data]
    bd = BatchDecoder(len(data), decode_b=1)
    for i, es in enumerate(data):
        bd.write(i, es)
    step = 0
    while bd.decode(1, OUT_DEVICE):
        for i, frames in enumerate(expected):
            if step < len(frames):
                assert_frames_equal([bd.read_planes(i)], [frames[step]], f"stream {i} picture {step}")
                assert bd.last_picture(i)[0] == picture_types(data[i])[step]
        step += 1
    assert step == max(len(f) for f in expected)
    st = bd.stats()
    assert st["pictures"] == sum(len(f) for f in expected) and st["parse_errors"] == 0
    bd.close()


def test_batch_multi_picture_calls_host_output_and_rewind(oracle_b):
    """decode(n > 1) with copy-out: consecutive B pictures alternate between the two B plane sets while the copy
    engine drains them; a rewind reproduces the same pictures."""
    es = natural_clip()[0]
    exp = decode_all(oracle_b, [(0, es)])[0]
    bd = BatchDecoder(2, decode_b=1)
    bd.write(0, es)
    bd.write(1, es)
    for rnd in range(2):
        done = 0
        for n in (1, 2, 3, 4, 50):
            got = bd.decode(n, OUT_HOST)
            assert got % 2 == 0
            done += got // 2
            if got:
                for s in range(2):
                    assert_frames_equal([tuple(p.copy() for p in bd.host_planes(s))], [exp[done - 1]], f"round {rnd} picture {done - 1}")
        assert done == len(exp)
        bd.rewind()
    bd.close()


def test_whole_clip_in_one_call_ends_on_the_right_picture(oracle_b):
    """All pictures in one wave (B and I/P pictures parsed by their own kernels side by side)."""
    streams = _streams()
    names = sorted(streams)
    expected = [decode_all(oracle_b, [(0, streams[n])])[0] for n in names]
    bd = BatchDecoder(len(names), decode_b=1)
    for i, n in enumerate(names):
        bd.write(i, streams[n])
    assert bd.decode(1000, OUT_DEVICE) == sum(len(f) for f in expected)
    for i, frames in enumerate(expected):
        assert_frames_equal([bd.read_planes(i)], [frames[-1]], f"{names[i]}: last picture")
    bd.close()


def test_fused_rgba_epilogue_on_b_pictures(oracle_b):
    from test_gpu_parity import _canvas2d_rgba
    es = natural_clip()[0]
    exp = decode_all(oracle_b, [(0, es)])[0]
    bd = BatchDecoder(1, decode_b=1)
    bd.write(0, es)
    n = 0
    while bd.decode(1, OUT_RGBA):
        y, cr, cb = bd.read_planes(0)
        assert_frames_equal([(y, cr, cb)], [exp[n]], f"picture {n} (RGBA run)")
        assert np.array_equal(bd.read_rgba(0), _canvas2d_rgba(y, cr, cb, 176, 144)), f"RGBA picture {n} differs"
        n += 1
    assert n == len(exp)
    bd.close()


def test_switching_the_extension_between_calls(oracle_b):
    """set_option("decode_b") flushes what was parsed ahead under the other rule."""
    es = synth_es.make_case("b_three")
    types = picture_types(es)
    bd = BatchDecoder(1)
    bd.write(0, es)
    assert bd.decode(1, OUT_DEVICE) == 1          # the I picture, B pictures behind it parsed ahead as "ignored"
    first = bd.read_planes(0)
    bd.set_option("decode_b", 1)
    exp = decode_all(oracle_b, [(0, es)])[0]
    assert_frames_equal([first], [exp[0]], "picture 0")
    for k in range(1, len(types)):
        assert bd.decode(1, OUT_DEVICE) == 1
        assert_frames_equal([bd.read_planes(0)], [exp[k]], f"picture {k} after switching the extension on")
    bd.close()


def test_bench_shape_64_streams_720p_every_picture():
    """The shape bench.py's b_pictures_720p leg and tools/time_b.py time: 64 streams of the committed 1280x720 I/P/B
    clip.  Picture by picture (13 steps: I/P launches and B launches), every stream's planes against the hashes the
    oracle gave (tests/fixtures/b_clip_1280x720.json); then the whole clip in one call after a rewind."""
    import json
    import os

    import bench
    from test_b_pictures import FIXTURE_720P
    meta = json.load(open(FIXTURE_720P.replace(".m1v", ".json")))
    es = open(FIXTURE_720P, "rb").read()
    n_streams = int(os.environ.get("B_TEST_STREAMS", "64"))
    bd = BatchDecoder(n_streams, max_slots=n_streams * 13 + 8, decode_b=1)
    for s in range(n_streams):
        bd.write(s, es)
    for k, want in enumerate(meta["fnv1a64"]):
        assert bd.decode(1, OUT_DEVICE) == n_streams
        for s in range(n_streams):
            assert format(bench.fnv1a64_planes(*bd.read_planes(s)), "016x") == want, f"stream {s} picture {k}"
            assert bd.last_picture(s) == (meta["picture_types"][k], [0, 3, 1, 2, 6, 4, 5, 9, 7, 8, 12, 10, 11][k])
    assert bd.decode(1, OUT_DEVICE) == 0
    bd.rewind()
    assert bd.decode(13, OUT_DEVICE) == 13 * n_streams
    for s in range(n_streams):
        assert format(bench.fnv1a64_planes(*bd.read_planes(s)), "016x") == meta["fnv1a64"][-1]
    st = bd.stats()
    assert st["parse_errors"] == 0
    bd.close()
