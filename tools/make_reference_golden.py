#!/usr/bin/env python
"""Record what the reference computes on the tests' inputs into tests/golden/reference/, so that the tests that pin
the oracle and the CUDA path to the reference run wherever the repository is checked out.

Needs oracle/_ref/libjsmpeg_ref.so (`make -C oracle REF=<reference checkout>`) and that checkout's
src/wasm/mpeg1.c for the VLC trees:

    python tools/make_reference_golden.py <reference checkout>

Writes
    decodes.json         per stream: digest of the input, bit index after every decode(), digests of Y / Cr / Cb
    idct.json            the reference's idct() on the blocks of tests/test_unit_parity.py
    vlc_trees.json       every code that reaches a leaf of the reference's VLC trees, and its constant matrices
    bitbuffer.json       the reference's bit buffer states under the traffic of tests/emu/bitbuffer_check.py
    picture_hashes.json  the reference harness's per-picture FNV-1a 64 (oracle/ref_bench.c) on the clips the GPU
                         tests decode at the benchmarked shape
"""
import ctypes
import json
import os
import re
import subprocess
import sys
import threading

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

import helpers  # noqa: E402
import synth_es  # noqa: E402

OUT = helpers.REF_GOLDEN


def decodes(ref):
    import test_gpu_parity
    import test_oracle_vs_reference as ovr
    import test_rgba_cases
    import test_unit_parity
    out = {}

    def add(key, packets, first=0):
        es = b"".join(p for _, p in packets)
        frames, idx, d = helpers.decode_all(ref, packets)
        out[key] = helpers.record_decode(frames, idx, es)
        d.destroy()

    for name in sorted(synth_es.CASES):
        add(f"synth/{name}", [(0.0, synth_es.make_case(name))])
    for seed in range(6):
        add(f"random/{seed}", [(0.0, ovr.random_syntax_stream(seed))])
    for w, h, n in sorted(set([(320, 240, 24), (1280, 720, 6)] + test_gpu_parity.SIZES + [(1920, 1080, 5)])):
        add(f"ffmpeg/{w}x{h}x{n}", helpers.clip_packets(w, h, n))
    packets = helpers.clip_packets(320, 240, 24)
    frames, trace = ovr.decode_streaming(ref, packets)
    out["evict/320x240x24"] = helpers.record_decode(frames, trace, b"".join(p for _, p in packets))
    add("vlc_trie", [(0.0, test_unit_parity.vlc_trie_stream())])
    add("b_rows/extension_off", [(0.0, synth_es.make_case("b_rows"))])
    add("rgba/flat_picture", [(0, test_rgba_cases.flat_picture_es(46, 30, test_rgba_cases.hand_picture()))])
    return out


def idct(ref):
    import test_unit_parity as t
    return {kind: {"inputs": helpers.digest(blocks), "outputs": t.idct_digests(ref.idct, blocks)}
            for kind, blocks in (("random", t.random_blocks()), ("sparse_and_extreme", t.sparse_and_extreme_blocks()))}


def vlc_trees(reference):
    import vlc_tables
    src = open(os.path.join(reference, "src", "wasm", "mpeg1.c")).read()
    arrays = {}
    for m in re.finditer(r"static const (?:int|uint8_t|float) (\w+)\[\] = \{(.*?)\};", src, re.S):
        body = re.sub(r"//[^\n]*", "", m.group(2))
        arrays[m.group(1)] = [eval(tok) for tok in (t.strip() for t in body.replace("\n", " ").split(",")) if tok]

    def codes(tree):  # read_huffman (src/wasm/mpeg1.c:1742-1748) over every bit string
        out = {}

        def walk(state, code):
            for bit in "01":
                nxt = tree[state + int(bit)]
                if nxt < 0:
                    continue
                if tree[nxt] == 0:
                    out[code + bit] = tree[nxt + 2]
                elif len(code) < 32:
                    walk(nxt, code + bit)
        walk(0, "")
        return out

    trees = {name: {"codes": codes(arrays[name]),
                    "leaves": sum(1 for i in range(0, len(arrays[name]), 3) if arrays[name][i] == 0 and i != 0)}
             for name in sorted(vlc_tables.ALL_VLC)}
    matrices = {k: arrays[k] for k in ("ZIG_ZAG", "DEFAULT_INTRA_QUANT_MATRIX", "DEFAULT_NON_INTRA_QUANT_MATRIX",
                                       "PREMULTIPLIER_MATRIX")}
    matrices["PICTURE_RATE"] = [round(x, 3) for x in arrays["PICTURE_RATE"]]
    return {"trees": trees, "matrices": matrices}


def bitbuffer():
    lib = os.path.join("/tmp", f"libbitbuffer_test_{os.getpid()}.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-o", lib,
                           os.path.join(ROOT, "tests", "emu", "bitbuffer_test.cpp")])
    path = os.path.join(OUT, "bitbuffer.json")
    try:
        subprocess.check_call([sys.executable, os.path.join(ROOT, "tests", "emu", "bitbuffer_check.py"), lib, path,
                               helpers.REF_LIB])
    finally:
        os.remove(lib)


def picture_hashes():
    import bench
    import test_gpu_bench_config as t
    lib = bench.ref_library()

    def hashes(es, n):
        buf = (ctypes.c_uint64 * n)()
        assert lib.ref_picture_hashes(es, len(es), buf, n) == n
        return [format(int(h), "016x") for h in buf]

    es = b"".join(p for _, p in helpers.clip_packets(176, 144, 5, seed=3, noise=4))
    out = {"176x144x5": {"es": helpers.digest(es), "fnv1a64": hashes(es, 5)}}
    old = bench.PICTURES
    bench.PICTURES = t.PICTURES
    try:
        clips = bench.load_streams(t.SEEDS, t.W, t.H)
    finally:
        bench.PICTURES = old
    per = [None] * len(clips)
    workers = bench.host_cores()["usable"]

    def work(k):
        for c in range(k, len(clips), workers):
            per[c] = hashes(clips[c], t.PICTURES)
    ths = [threading.Thread(target=work, args=(k,)) for k in range(workers)]
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    out[f"{t.W}x{t.H}x{t.PICTURES}"] = {"seeds": t.SEEDS, "es": [helpers.digest(c) for c in clips], "fnv1a64": per}
    return out


def main():
    if len(sys.argv) != 2 or helpers.ref_lib() is None:
        raise SystemExit(__doc__)
    ref = helpers.ref_lib()
    os.makedirs(OUT, exist_ok=True)
    for name, make in (("decodes", lambda: decodes(ref)), ("idct", lambda: idct(ref)),
                       ("vlc_trees", lambda: vlc_trees(sys.argv[1])), ("picture_hashes", picture_hashes)):
        with open(os.path.join(OUT, name + ".json"), "w") as f:
            json.dump(make(), f, indent=0, separators=(",", ":"), sort_keys=True)
            f.write("\n")
        print("wrote", name)
    bitbuffer()


if __name__ == "__main__":
    main()
