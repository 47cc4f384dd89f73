"""Parity AT the benchmarked configuration (BASELINE configs[3]): 64 independent 1920x1080 streams, 64 distinct
seeds, 25 pictures each (two GOP boundaries: I pictures at 0, 12, 24), decoded

  * by ONE BatchDecoder as one wave with device-resident planes -- bench.py's `value` leg, the 1600-picture
    lane-parallel walk, 25 reconstruct launches of 64 pictures,
  * in calls of 5 pictures, and picture by picture for a few streams (every plane of every picture),
  * by 16 BatchDecoders of 4 streams on 16 host threads with OUT_HOST -- bench.py's `e2e` leg, through the
    pinned host rings,

every checked picture hashed (FNV-1a 64 over Y | Cr | Cb, coded size) against the UNMODIFIED reference C
(src/wasm/mpeg1.c:853-864, 947-995 is the loop it runs) decoding the same stream on the host: its hashes are
recorded in tests/golden/reference/picture_hashes.json (tools/make_reference_golden.py).
Round 1 checked five pictures of one 1080p stream; nothing looked at a byte of the benchmarked workload."""
import sys
import threading

import numpy as np
import pytest

import helpers

sys.path.insert(0, helpers.ROOT)

pytestmark = pytest.mark.gpu

STREAMS, PICTURES, W, H = 64, 25, 1920, 1080
SEEDS = [1234 + i for i in range(STREAMS)]


@pytest.fixture(scope="module")
def workload():
    import bench
    old = bench.PICTURES
    bench.PICTURES = PICTURES
    try:
        clips = bench.load_streams(SEEDS, W, H)
    finally:
        bench.PICTURES = old
    rec = helpers.reference_golden("picture_hashes")[f"{W}x{H}x{PICTURES}"]
    assert rec["seeds"] == SEEDS
    bad = [i for i, es in enumerate(clips) if helpers.digest(es) != rec["es"][i]]
    assert not bad, f"streams {bad[:8]} are not the ones the reference decoded"
    want = np.array([[int(h, 16) for h in row] for row in rec["fnv1a64"]], dtype=np.uint64)
    assert want.shape == (STREAMS, PICTURES)
    assert len({int(x) for x in want[:, -1]}) == STREAMS  # 64 distinct clips really are distinct
    return bench, clips, want


def _hash(bench, planes):
    y, cr, cb = planes
    return bench.fnv1a64_planes(np.ascontiguousarray(y), np.ascontiguousarray(cr), np.ascontiguousarray(cb))


def test_one_wave_of_64_streams_device_output(workload):
    from jsmpeg_b200.batch import OUT_DEVICE, BatchDecoder
    bench, clips, want = workload
    bd = BatchDecoder(STREAMS, max_slots=STREAMS * PICTURES + 8)
    for i, es in enumerate(clips):
        bd.write(i, es)
    bd.reset_stats()
    assert bd.decode(PICTURES, OUT_DEVICE) == STREAMS * PICTURES  # the bench's value leg: one call, one wave
    st = bd.stats()
    assert st["lane_walk_pictures"] == STREAMS * PICTURES and st["parse_errors"] == 0
    bad = [i for i in range(STREAMS) if _hash(bench, bd.read_planes(i)) != int(want[i, PICTURES - 1])]
    assert not bad, f"last picture differs from the reference in streams {bad}"
    # the same wave with the parse/reconstruct pipeline cut into chunks of 6 pictures
    bd.set_option("chunk_pictures", 6)
    bd.rewind()
    assert bd.decode(PICTURES, OUT_DEVICE) == STREAMS * PICTURES
    bad = [i for i in range(STREAMS) if _hash(bench, bd.read_planes(i)) != int(want[i, PICTURES - 1])]
    assert not bad, f"chunked pipeline: last picture differs in streams {bad}"
    bd.set_option("chunk_pictures", 0)
    # in calls of 5 pictures: pictures 4, 9, 14, 19, 24 of every stream
    bd.rewind()
    for k in range(PICTURES // 5):
        assert bd.decode(5, OUT_DEVICE) == STREAMS * 5
        bad = [i for i in range(STREAMS) if _hash(bench, bd.read_planes(i)) != int(want[i, 5 * k + 4])]
        assert not bad, f"picture {5 * k + 4} differs in streams {bad}"
    # picture by picture, every picture of eight streams
    bd.rewind()
    for k in range(PICTURES):
        assert bd.decode(1, OUT_DEVICE) == STREAMS
        for i in range(0, STREAMS, 8):
            assert _hash(bench, bd.read_planes(i)) == int(want[i, k]), f"stream {i} picture {k}"
    bd.close()


def test_sixteen_threaded_decoders_host_output(workload):
    """bench.py's e2e leg: 16 decoders of 4 streams, one host thread each, OUT_HOST; write -> decode twice (the
    second round after reset(), like the bench's steady state)."""
    from jsmpeg_b200.batch import OUT_HOST, BatchDecoder
    bench, clips, want = workload
    groups = [list(range(g, STREAMS, 16)) for g in range(16)]
    decs = [BatchDecoder(len(g), max_slots=len(g) * PICTURES + 8) for g in groups]
    errors = []

    def work(k):
        try:
            dec = decs[k]
            for rnd in range(2):
                dec.reset()
                for j, i in enumerate(groups[k]):
                    dec.write(j, clips[i])
                n = dec.decode(PICTURES, OUT_HOST)
                assert n == len(groups[k]) * PICTURES, (k, rnd, n)
                for j, i in enumerate(groups[k]):
                    got = _hash(bench, dec.host_planes(j))
                    assert got == int(want[i, PICTURES - 1]), f"round {rnd}: stream {i}: host planes of the last picture differ"
            # picture by picture through the host ring for this group's first stream set
            if k == 0:
                dec.reset()
                for j, i in enumerate(groups[k]):
                    dec.write(j, clips[i])
                for p in range(PICTURES):
                    assert dec.decode(1, OUT_HOST) == len(groups[k])
                    for j, i in enumerate(groups[k]):
                        assert _hash(bench, dec.host_planes(j)) == int(want[i, p]), f"stream {i} picture {p} (host ring)"
        except Exception as e:  # noqa: BLE001 -- reported in the main thread
            errors.append(repr(e))

    ths = [threading.Thread(target=work, args=(k,)) for k in range(16)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    for d in decs:
        d.close()
    assert not errors, errors[:4]
