"""Shared test helpers: library loading, clip access, oracle record access."""
import ctypes
import hashlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from jsmpeg_b200 import capi, decoder  # noqa: E402

ORACLE_LIB = os.path.join(ROOT, "oracle", "liboracle.so")
REF_LIB = os.path.join(ROOT, "oracle", "_ref", "libjsmpeg_ref.so")
REF_GOLDEN = os.path.join(ROOT, "tests", "golden", "reference")


class PictureInfo(ctypes.Structure):
    _fields_ = [("start_byte", ctypes.c_uint32), ("end_bit", ctypes.c_uint32), ("status", ctypes.c_int32),
                ("picture_type", ctypes.c_int32), ("full_pel", ctypes.c_int32), ("f_code", ctypes.c_int32),
                ("n_present", ctypes.c_int32), ("n_coded_blocks", ctypes.c_int32), ("error", ctypes.c_int32),
                ("reserved", ctypes.c_int32 * 3)]


class SeqParamsOracle(ctypes.Structure):
    _fields_ = [("mb_width", ctypes.c_int), ("mb_size", ctypes.c_int),
                ("intra_q", ctypes.c_uint8 * 64), ("non_intra_q", ctypes.c_uint8 * 64)]


def build_oracle():
    if not os.path.exists(ORACLE_LIB) or os.path.getmtime(ORACLE_LIB) < os.path.getmtime(
            os.path.join(ROOT, "oracle", "mpeg1_oracle.c")):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")])


_oracle = None


def oracle_lib():
    global _oracle
    if _oracle is None:
        build_oracle()
        lib = capi.load_library(ORACLE_LIB)
        lib.oracle_last_picture_info.restype = ctypes.POINTER(PictureInfo)
        lib.oracle_last_picture_info.argtypes = [ctypes.c_void_p]
        lib.oracle_last_mb_records.restype = ctypes.c_void_p
        lib.oracle_last_mb_records.argtypes = [ctypes.c_void_p]
        lib.oracle_last_coefficients.restype = ctypes.c_void_p
        lib.oracle_last_coefficients.argtypes = [ctypes.c_void_p]
        lib.oracle_seq_params.restype = ctypes.POINTER(SeqParamsOracle)
        lib.oracle_seq_params.argtypes = [ctypes.c_void_p]
        # the product's extension entry points, same names (B pictures: decodeBPictures / lastPicture of the host class)
        lib.jsmpeg_b200_decoder_set_option.restype = ctypes.c_int
        lib.jsmpeg_b200_decoder_set_option.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int]
        lib.jsmpeg_b200_decoder_last_picture.restype = ctypes.c_int
        lib.jsmpeg_b200_decoder_last_picture.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]
        _oracle = lib
    return _oracle


def ref_lib():
    """The compiled reference (oracle/_ref), where tools/make_reference_golden.py records from it; None elsewhere."""
    if not os.path.exists(REF_LIB):
        return None
    return capi.load_library(REF_LIB)


def digest(data):
    """Short content hash (sha256, 64 bits) of bytes or of an array's memory."""
    if not isinstance(data, (bytes, bytearray)):
        data = np.ascontiguousarray(data).tobytes()
    return hashlib.sha256(data).hexdigest()[:16]


def record_decode(frames, idx, es=None):
    """What a reference decode is recorded as in tests/golden/reference/decodes.json."""
    out = {"index": list(idx), "planes": [[digest(p) for p in f] for f in frames]}
    if es is not None:
        out["es"] = digest(es)
    return out


def reference_golden(name):
    """tests/golden/reference/<name>.json: what the compiled reference computed on the tests' inputs."""
    with open(os.path.join(REF_GOLDEN, name + ".json")) as f:
        return json.load(f)


def assert_matches_reference(key, frames, idx, es=None, first=0):
    """frames / bit indices of a decode against the reference's decode of the same stream (decodes.json[key]);
    idx None: planes only; `first` skips pictures whose planes the C reference leaves uninitialised."""
    want = reference_golden("decodes")[key]
    if es is not None:
        assert digest(es) == want["es"], f"{key}: the input stream is not the one the reference decoded"
    assert idx is None or list(idx) == want["index"], f"{key}: bit indices differ from the reference"
    got = [[digest(p) for p in f] for f in frames]
    assert len(got) == len(want["planes"]), f"{key}: {len(got)} vs {len(want['planes'])} pictures"
    for k in range(first, len(got)):
        assert got[k] == want["planes"][k], f"{key}: picture {k} differs from the reference (Y, Cr, Cb digests)"


def decode_all(lib, packets, options=None, keep=True, max_frames=None):
    """Drive a 15-function-ABI library through the decoder surface: write everything, then decode()
    until it returns False.  Returns (frames, bit indices after each decode, decoder)."""
    opts = {"decodeFirstFrame": False}
    opts.update(options or {})
    d = decoder.MPEG1Video(opts, lib=lib)
    rec = decoder.PlaneRecorder(keep=keep)
    d.connect(rec)
    for pts, payload in packets:
        d.write(pts, [payload])
    idx = []
    while (max_frames is None or len(idx) < max_frames) and d.decode():
        idx.append(d.bufferGetIndex())
    return rec.frames, idx, d


def assert_frames_equal(a, b, what=""):
    assert len(a) == len(b), f"{what}: {len(a)} vs {len(b)} pictures"
    for k, (x, y) in enumerate(zip(a, b)):
        for name, p, q in zip(("Y", "Cr", "Cb"), x, y):
            if not np.array_equal(p, q):
                w = np.nonzero(p != q)[0]
                raise AssertionError(f"{what}: picture {k} plane {name}: {len(w)} bytes differ, first at {w[:8]}: "
                                     f"{p[w[:8]]} vs {q[w[:8]]}")


def clip_packets(width, height, frames, seed=1234, noise=9):
    import gen_streams
    return gen_streams.make_clip_es(width, height, frames, seed, noise)
