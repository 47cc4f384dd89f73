"""Child process of tests/test_bitbuffer.py (libasan preloaded): drives jsmpeg_b200/csrc/bitbuffer.h
(through tests/emu/bitbuffer_test.cpp, exact-size malloc) with growing and random writes in both
modes; every byte the protocol hands out is written, so AddressSanitizer aborts the process on any
byte the returned pointer does not cover.  Where the REFERENCE's own arithmetic leaves enough room, the
state (capacity, length, index, content) must equal that of the reference's bit_buffer_* functions
(src/wasm/buffer.c:48-71, 157-190).

    bitbuffer_check.py <bitbuffer_test lib> <states.json>             compare with the recorded reference states
    bitbuffer_check.py <bitbuffer_test lib> <states.json> <ref lib>   run the reference beside it and record them

Prints "bitbuffer ok: N writes" on success."""
import ctypes
import hashlib
import json
import sys

import numpy as np

lib = ctypes.CDLL(sys.argv[1])
STATES = sys.argv[2]
ref = ctypes.CDLL(sys.argv[3]) if len(sys.argv) > 3 else None
recorded = None if ref is not None else json.load(open(STATES))["trials"]
lib.bbt_create.restype = ctypes.c_void_p
lib.bbt_create.argtypes = [ctypes.c_uint, ctypes.c_int]
lib.bbt_destroy.argtypes = [ctypes.c_void_p]
lib.bbt_write.restype = ctypes.c_long
lib.bbt_write.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_uint]
lib.bbt_set_index.argtypes = [ctypes.c_void_p, ctypes.c_uint]
lib.bbt_state.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint)]
lib.bbt_bytes.restype = ctypes.POINTER(ctypes.c_ubyte)
lib.bbt_bytes.argtypes = [ctypes.c_void_p]


class RefBuffer(ctypes.Structure):  # src/wasm/buffer.h:13-19
    _fields_ = [("bytes", ctypes.POINTER(ctypes.c_ubyte)), ("index", ctypes.c_uint), ("byte_capacity", ctypes.c_uint),
                ("byte_length", ctypes.c_uint), ("mode", ctypes.c_int)]


if ref is not None:
    ref.bit_buffer_create.restype = ctypes.POINTER(RefBuffer)
    ref.bit_buffer_create.argtypes = [ctypes.c_uint, ctypes.c_int]
    ref.bit_buffer_get_write_ptr.restype = ctypes.c_void_p
    ref.bit_buffer_get_write_ptr.argtypes = [ctypes.POINTER(RefBuffer), ctypes.c_uint]
    ref.bit_buffer_did_write.argtypes = [ctypes.POINTER(RefBuffer), ctypes.c_uint]
    ref.bit_buffer_destroy.argtypes = [ctypes.POINTER(RefBuffer)]


def state(t):
    out = (ctypes.c_uint * 4)()
    lib.bbt_state(t, out)
    return tuple(out)


def content(t):
    cap, length, _, _ = state(t)
    return bytes(lib.bbt_bytes(t)[:length])


def trace_digest(states):
    return hashlib.sha256(repr(states).encode()).hexdigest()[:16]


writes = 0
# the advisor's case: capacity 1000, 900 bytes buffered, then 1500 (the reference sizes the expansion at 2000)
for mode in (2, 1):
    t = lib.bbt_create(1000, mode)
    a, b = bytes(range(256)) * 4, bytes(reversed(range(256))) * 6
    assert lib.bbt_write(t, a[:900], 900) == 0
    off = lib.bbt_write(t, b[:1500], 1500)
    cap, length, index, moved = state(t)
    if mode == 2:
        assert (off, cap, length) == (900, 2400, 2400), (off, cap, length)
        assert content(t) == a[:900] + b[:1500]
    else:  # nothing read yet and no room even after dropping everything: evacuate, then grow
        assert (off, length, index) == (0, 1500, 0) and cap >= 1500, (off, cap, length, index)
        assert content(t) == b[:1500]
    lib.bbt_destroy(t)
    writes += 2

# growing chunks, a whole file in one write, zero-size buffer
for mode in (2, 1):
    t = lib.bbt_create(0, mode)
    model = b""
    for n in (1, 7, 64, 1000, 5, 70000, 3):
        chunk = bytes((i * 7 + n) & 255 for i in range(n))
        off = lib.bbt_write(t, chunk, n)
        assert off >= 0
        if mode == 2:
            model += chunk
            assert content(t) == model
        else:
            assert content(t).endswith(chunk)
        writes += 1
    lib.bbt_destroy(t)

# random traffic; against the reference wherever the reference itself stays inside its allocation
rng = np.random.default_rng(7)
trials = []
for trial in range(300):
    mode = int(rng.integers(1, 3))
    cap = int(rng.integers(1, 4000))
    t = lib.bbt_create(cap, mode)
    r = ref.bit_buffer_create(cap, mode) if ref is not None else None
    in_domain = True
    states = []  # (capacity, length, index, content digest) after every write inside the reference's domain
    for step in range(int(rng.integers(1, 40))):
        n = int(rng.integers(0, 3000)) if rng.random() < 0.8 else int(rng.integers(0, 40))
        chunk = bytes(rng.integers(0, 256, n, dtype=np.uint8))
        assert lib.bbt_write(t, chunk, n) >= 0
        writes += 1
        cap_t, len_t, idx_t, _ = state(t)
        assert content(t).endswith(chunk) and len_t <= cap_t
        if in_domain and r is None:
            if step == recorded[trial]["steps"]:
                in_domain = False
            else:
                states.append((cap_t, len_t, idx_t, hashlib.sha256(content(t)).hexdigest()[:16]))
        elif in_domain:
            ref.bit_buffer_get_write_ptr(r, n)
            if r.contents.byte_capacity - r.contents.byte_length < n:
                in_domain = False  # the reference would now write past its allocation: no parity defined from here on
            else:
                ctypes.memmove(ctypes.addressof(r.contents.bytes.contents) + r.contents.byte_length, chunk, n)
                ref.bit_buffer_did_write(r, n)
                assert (cap_t, len_t, idx_t) == (r.contents.byte_capacity, r.contents.byte_length, r.contents.index), \
                    (trial, step, (cap_t, len_t, idx_t), (r.contents.byte_capacity, r.contents.byte_length, r.contents.index))
                assert content(t) == bytes(r.contents.bytes[:len_t])
                states.append((cap_t, len_t, idx_t, hashlib.sha256(content(t)).hexdigest()[:16]))
        # the decoder consumes some of what is buffered
        idx = int(rng.integers(idx_t >> 3, len_t + 1)) << 3
        lib.bbt_set_index(t, idx)
        if in_domain and r is not None:
            r.contents.index = idx
    lib.bbt_destroy(t)
    if r is not None:
        ref.bit_buffer_destroy(r)
        trials.append({"steps": len(states), "states": trace_digest(states)})
    else:
        assert trace_digest(states) == recorded[trial]["states"], \
            f"trial {trial}: capacity / length / index / content differ from the reference's within its first {len(states)} writes"
if ref is not None:
    with open(STATES, "w") as f:
        json.dump({"trials": trials}, f, indent=0, separators=(",", ":"))
        f.write("\n")
print("bitbuffer ok:", writes, "writes", "(reference recorded)" if ref is not None else "(reference compared)")
