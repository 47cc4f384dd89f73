"""GPU parity of the slice walk (walk_pictures_slices_kernel, option "slice_walk"): one lane per slice for I/P
pictures of many slices.  Same records as the default walk, so every check is bit-exact against the oracle; the CPU
twin (the same device code emulated) is in tests/test_walk_emu.py.
"""
import json
import os

import numpy as np
import pytest

import helpers
import synth_es
import test_oracle_golden as golden
from helpers import assert_frames_equal, decode_all
from jsmpeg_b200.batch import OUT_DEVICE, OUT_HOST, BatchDecoder

pytestmark = pytest.mark.gpu


def _decode_batch(es_list, **options):
    bd = BatchDecoder(len(es_list), **options)
    for i, es in enumerate(es_list):
        bd.write(i, es)
    frames = [[] for _ in es_list]
    while bd.decode(1, OUT_DEVICE):
        for i in range(len(es_list)):
            frames[i].append(tuple(p.copy() for p in bd.read_planes(i)))
    st = bd.stats()
    bd.close()
    return frames, st


@pytest.mark.parametrize("name", golden.CASES)
def test_golden_vectors_with_the_slice_walk(name):
    """Every golden stream (a slice per row, slices starting mid-row, gaps, stuffing, one slice per picture, ignored
    pictures ...) with the option on: the pictures the reference produced."""
    es, info = golden.load_case(name)
    exp = decode_all(helpers.oracle_lib(), [(0, es)])[0]
    got, st = _decode_batch([es], slice_walk=1)
    n = min(len(exp), len(got[0]))
    assert n == len(exp)
    for k in range(n):  # (decode(1) steps also count ignored pictures: the planes then repeat, like the oracle's frames)
        assert_frames_equal([got[0][k]], [exp[k]], f"{name}: picture {k}")


def test_row_sliced_streams_in_one_wave_with_b_pictures():
    """64 x the committed 1280x720 I/P/B clip (45 slices per picture): I/P pictures through the slice walk, B pictures
    through theirs, both beside each other; every picture of every stream against the oracle's hashes."""
    import bench
    from test_b_pictures import FIXTURE_720P
    meta = json.load(open(FIXTURE_720P.replace(".m1v", ".json")))
    es = open(FIXTURE_720P, "rb").read()
    n_streams = 64
    bd = BatchDecoder(n_streams, max_slots=n_streams * 13 + 8, decode_b=1, slice_walk=1)
    for s in range(n_streams):
        bd.write(s, es)
    assert bd.decode(13, OUT_DEVICE) == 13 * n_streams
    for s in range(n_streams):
        assert format(bench.fnv1a64_planes(*bd.read_planes(s)), "016x") == meta["fnv1a64"][-1]
    st = bd.stats()
    assert st["parse_errors"] == 0 and st["lane_walk_pictures"] == 5 * n_streams  # the 5 I/P pictures of every stream
    bd.rewind()
    for k, want in enumerate(meta["fnv1a64"]):
        assert bd.decode(1, OUT_HOST) == n_streams
        for s in (0, 17, n_streams - 1):
            y, cr, cb = (p.copy() for p in bd.host_planes(s))
            assert format(bench.fnv1a64_planes(y, cr, cb), "016x") == want, f"stream {s} picture {k}"
    bd.close()


def test_mixed_batch_and_damaged_streams():
    """One-slice clips (which stay with the lane-parallel walk), row-sliced ones and bit-flipped copies in one batch:
    identical to the same batch decoded without the option."""
    rng = np.random.default_rng(3)
    base = [synth_es.make_case(n) for n in ("rows_ip", "fcodes_fullpel", "random_slices_gaps", "skips_stuffing_escape_mba")]
    base.append(b"".join(p for _, p in helpers.clip_packets(320, 240, 6)))
    damaged = []
    for es in base[:3]:
        bad = bytearray(es)
        for pos in rng.integers(200, len(es), size=4):
            bad[pos] ^= 1 << int(rng.integers(0, 8))
        damaged.append(bytes(bad))
    streams = base + damaged
    want, _ = _decode_batch(streams)
    got, st = _decode_batch(streams, slice_walk=1)
    for i in range(len(streams)):
        assert_frames_equal(got[i], want[i], f"stream {i}")
