#!/usr/bin/env python
"""bench.py -- MPEG-1 video decode throughput (frames/s, Gpix/s) on N B200s vs the reference on host cores.

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own C on the host cores

Workload (BASELINE.json configs[3], weak-scaled to configs[4]): STREAMS_PER_GPU = 64 independent
1920x1080 MPEG-1 I+P elementary streams of PICTURES = 60 pictures each per GPU, every stream its OWN
clip (seed 1234 + rank * 64 + i; SURVEY 8(d) config 4), demuxed from synthetic MPEG-TS made by
tools/gen_streams.py (seeded content encoded by cv2's FFmpeg, GOP 12, one slice per picture).
One STEP = every picture of every stream once: start-code scan + VLC parse (stage 1) + IDCT/MC
reconstruction (stage 2).

  value  frames/s with the elementary streams already resident in HBM (jsmpeg_b200_batch_rewind
         forgets the start-code index and all parsed records, so scan + parse + reconstruct are
         all inside the timed region), planes left in HBM.
  e2e    the same through the reference-facing call sequence with HOST buffers: per step every
         stream is written again from host memory (get_write_ptr/memcpy/did_write -> H2D) and
         every decoded picture's Y/Cr/Cb planes are copied back to pinned host memory (D2H).
         The streams are driven as several independent BatchDecoders from host threads, so
         that one group's PCIe copy-out overlaps another group's write + parse.  The rank is bound
         to the CPUs of its GPU's NUMA node first (pinned rings are then node-local).
  verified  after the timed region the LAST picture of every stream of the rank (60 pictures deep into
         the P chains) is read back and its FNV-1a hash compared with the unmodified reference C
         (oracle/_ref; where that was not built, the oracle, pinned to it by the tests) decoding the same
         stream on the host; the run FAILS (exit 1) on any difference or if any picture fell back from the
         lane-parallel walk.
  roofline  stage-2 kernel: algorithmic bytes (DESIGN.md) / CUDA-event time of its launches on the
         stream they run on; in the value leg nothing else runs beside them.
  cpu_baseline  oracle/_ref (the unmodified reference C, compiled in place) on the host cores this
         process may really use: min(affinity, cgroup cpu.max quota) -- os.cpu_count() alone overstates
         a container's share.
  config_720p, single_stream_1080p  (N = 1 only) BASELINE configs[1] / [2]: the same legs at 64 x
         1280x720, and ONE 1080p stream through the 15-function reference ABI (ms per
         mpeg1_decoder_decode, look-ahead 16 and 1) beside one host core of the reference.
  b_pictures_720p  (N = 1 only) the opt-in B-picture extension on 64 x a committed 1280x720 I/P/B clip, last
         pictures hashed against the oracle's values; beside it the same call skipping B like the reference.

Timing: wall clock between torch.cuda.synchronize() + barrier on both sides of exactly K steps
(every step ends host-synchronised), max over ranks; per-kernel times are CUDA events recorded on
the launching stream inside the library.  Inputs are much larger than L2 (ES ~0.8 GB, records
~20 GB per step), so no explicit L2 flush is needed.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

WIDTH = int(os.environ.get("BENCH_WIDTH", 1920))    # the env overrides exist for the CPU smoke test of this file
HEIGHT = int(os.environ.get("BENCH_HEIGHT", 1080))
STREAMS_PER_GPU = int(os.environ.get("BENCH_STREAMS", 64))
PICTURES = int(os.environ.get("BENCH_PICTURES", 60))
DISTINCT = int(os.environ.get("BENCH_DISTINCT", 0)) or STREAMS_PER_GPU  # distinct clips per rank
NOISE = 9
E2E_GROUPS = int(os.environ.get("BENCH_E2E_GROUPS", 16))
VALUE_GROUPS = int(os.environ.get("BENCH_VALUE_GROUPS", 1))
EXTRAS = os.environ.get("BENCH_EXTRAS", "1") != "0"   # config_720p + single_stream_1080p (N = 1 only)


def env_int(name, default):
    return int(os.environ.get(name, default))


# ------------------------------------------------------------------------------------------------
# host: how many cores this process really has

def host_cores():
    """os.cpu_count() says what the machine has; a container gets its scheduler affinity and, on top,
    a cgroup CPU quota (cpu.max = '<quota> <period>').  usable = min(affinity, quota)."""
    out = {"cpu_count": os.cpu_count(), "affinity": len(os.sched_getaffinity(0)), "cgroup_quota_cpus": None}
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    out["cgroup_quota_cpus"] = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    out["cgroup_quota_cpus"] = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except (OSError, ValueError, IndexError):
            continue
    usable = out["affinity"]
    if out["cgroup_quota_cpus"]:
        usable = min(usable, max(1, int(math.floor(out["cgroup_quota_cpus"] + 1e-6))))
    out["usable"] = max(1, usable)
    return out


# ------------------------------------------------------------------------------------------------
# synthetic streams

def _encode_one(args):
    import gen_streams
    w, h, n, seed = args
    gen_streams.make_clip_ts(w, h, n, seed=seed, noise=NOISE)
    return seed


def load_streams(seeds, width=None, height=None, workers=None):
    """One elementary stream (bytes) per seed; the clips are encoded in parallel processes first
    (cached under /tmp, so the reference arm and this arm of one box encode once)."""
    import gen_streams
    width, height = width or WIDTH, height or HEIGHT
    from concurrent.futures import ProcessPoolExecutor
    workers = workers or host_cores()["usable"]
    with ProcessPoolExecutor(max_workers=max(1, min(len(seeds), workers))) as ex:
        list(ex.map(_encode_one, [(width, height, PICTURES, s) for s in seeds]))
    out = []
    for s in seeds:
        packets = gen_streams.make_clip_es(width, height, PICTURES, seed=s, noise=NOISE)
        out.append(b"".join(p for _, p in packets))
    return out


def rank_seeds(rank, n=None):
    n = n or STREAMS_PER_GPU
    return [1234 + rank * STREAMS_PER_GPU + (i % DISTINCT) for i in range(n)]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None
        self.t_mark = 0.0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def mark(self):
        """Samples that arrive from now on belong to the timed region."""
        self.t_mark = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, power = [], 0, set(), 0.0
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t_arrival, line in self.lines:
            if t_arrival < self.t_mark:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx = max(mx, float(f[2]))
                power = max(power, float(f[3]))
            except ValueError:
                continue
            for name, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None,
                "power_w_max": power or None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic():
    """dram bytes per stage-2 launch from the committed ncu --set full capture, if any."""
    path = os.path.join(ROOT, "profiles", "recon_traffic.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return None


# ------------------------------------------------------------------------------------------------
# the reference on the host: reference arm / cpu baseline / checker

REF_LIB = os.path.join(ROOT, "oracle", "_ref", "libjsmpeg_ref.so")
_ref = None


def ref_library():
    """oracle/_ref/libjsmpeg_ref.so: the unmodified reference C (built from /root/reference/src/wasm/*.c
    in the build container; travels with the tree) + our pthread harness oracle/ref_bench.c."""
    global _ref
    if _ref is None and os.path.exists(REF_LIB):
        lib = ctypes.CDLL(REF_LIB, mode=os.RTLD_LOCAL | os.RTLD_NOW)
        lib.ref_bench_run.restype = ctypes.c_long
        lib.ref_bench_run.argtypes = [ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(ctypes.c_uint), ctypes.c_int,
                                      ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_double)]
        lib.ref_picture_hashes.restype = ctypes.c_long
        lib.ref_picture_hashes.argtypes = [ctypes.c_char_p, ctypes.c_uint, ctypes.POINTER(ctypes.c_uint64), ctypes.c_long]
        lib.ref_hash_bytes.restype = ctypes.c_uint64
        lib.ref_hash_bytes.argtypes = [ctypes.c_uint64, ctypes.c_void_p, ctypes.c_size_t]
        _ref = lib
    return _ref


def run_reference_cpu(clips, threads, loops):
    """The reference's own C decoder on `threads` host threads, clip c on thread c % threads; only the
    decode() loops are inside the timed region (decoders are created and written before it).  Falls
    back to our CPU port of it (oracle/) when the reference build is absent.  Returns (frames, seconds, kind)."""
    n = len(clips)
    lib = ref_library()
    if lib is not None:
        arr = (ctypes.c_char_p * n)(*clips)
        lens = (ctypes.c_uint * n)(*[len(c) for c in clips])
        sec = ctypes.c_double()
        frames = lib.ref_bench_run(arr, lens, n, threads, loops, ctypes.byref(sec))
        return frames, sec.value, "reference"
    # port: the oracle through ctypes from Python threads (ctypes releases the GIL in the C calls)
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")])
    from jsmpeg_b200 import capi
    lib = capi.load_library(os.path.join(ROOT, "oracle", "liboracle.so"))
    counts = [0] * threads
    spent = [0.0] * threads

    def work(t):
        for _ in range(loops):
            for c in range(t, n, threads):
                d = lib.mpeg1_decoder_create(len(clips[c]) + 16, 2)
                ctypes.memmove(lib.mpeg1_decoder_get_write_ptr(d, len(clips[c])), clips[c], len(clips[c]))
                lib.mpeg1_decoder_did_write(d, len(clips[c]))
                t0 = time.perf_counter()
                while lib.mpeg1_decoder_decode(d):
                    counts[t] += 1
                spent[t] += time.perf_counter() - t0
                lib.mpeg1_decoder_destroy(d)

    ths = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    return sum(counts), max(spent), "port"


def oracle_last_hash(lib, es):
    """(pictures, hash of the LAST picture) of one clip decoded by the oracle through the 15-function ABI."""
    d = lib.mpeg1_decoder_create(len(es) + 16, 2)
    ctypes.memmove(lib.mpeg1_decoder_get_write_ptr(d, len(es)), es, len(es))
    lib.mpeg1_decoder_did_write(d, len(es))
    n = 0
    while lib.mpeg1_decoder_decode(d):
        n += 1
    ysz = lib.mpeg1_decoder_get_coded_size(d)
    h = 1469598103934665603
    for ptr, size in ((lib.mpeg1_decoder_get_y_ptr(d), ysz), (lib.mpeg1_decoder_get_cr_ptr(d), ysz >> 2),
                      (lib.mpeg1_decoder_get_cb_ptr(d), ysz >> 2)):
        h = lib.oracle_hash_bytes(h, ptr, size)
    lib.mpeg1_decoder_destroy(d)
    return n, int(h) if n > 0 else None


def reference_last_hashes(clips, workers):
    """(pictures, hash of the LAST picture) of each clip, decoded on `workers` host threads by the reference
    (oracle/_ref) or, where that was not built, by the oracle, which the test suite pins to the reference."""
    lib = ref_library()
    olib = None
    if lib is None:
        olib = oracle_library()
        olib.mpeg1_decoder_destroy(olib.mpeg1_decoder_create(16, 2))  # its VLC tables are built once, here
    out = [None] * len(clips)

    def work(k):
        for c in range(k, len(clips), workers):
            if olib is not None:
                out[c] = oracle_last_hash(olib, clips[c])
                continue
            buf = (ctypes.c_uint64 * (PICTURES + 4))()
            n = lib.ref_picture_hashes(clips[c], len(clips[c]), buf, PICTURES + 4)
            out[c] = (int(n), int(buf[min(n, PICTURES + 4) - 1]) if n > 0 else None)

    ths = [threading.Thread(target=work, args=(k,)) for k in range(workers)]
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    return out


_oracle = None


def oracle_library():
    """oracle/liboracle.so: our CPU restatement of the reference (built by build()); here for its FNV-1a 64."""
    global _oracle
    if _oracle is None:
        from jsmpeg_b200 import capi
        lib = capi.load_library(os.path.join(ROOT, "oracle", "liboracle.so"))
        lib.oracle_hash_bytes.restype = ctypes.c_uint64
        lib.oracle_hash_bytes.argtypes = [ctypes.c_uint64, ctypes.c_void_p, ctypes.c_size_t]
        _oracle = lib
    return _oracle


def fnv1a64_planes(y, cr, cb):
    """FNV-1a 64 of Y | Cr | Cb, the hash oracle/ref_bench.c gives the reference's pictures (the hash is inherently
    serial; Python ints would take seconds per picture, so the byte loop runs in C: oracle_hash_bytes)."""
    lib = oracle_library()
    h = 1469598103934665603
    for a in (y, cr, cb):
        a = np.ascontiguousarray(a)
        h = lib.oracle_hash_bytes(h, a.ctypes.data, a.size)
    return int(h)


def truncate_pictures(es, n_pictures):
    """The first n_pictures pictures of an elementary stream (cut at the next picture start code)."""
    pos, count = 0, 0
    while True:
        pos = es.find(b"\x00\x00\x01\x00", pos)
        if pos < 0:
            return es
        if count == n_pictures:
            return es[:pos]
        count += 1
        pos += 4


# ------------------------------------------------------------------------------------------------
# the GPU legs

class Legs:
    """The timed legs over one set of streams (one resolution) on this rank's GPU."""

    def __init__(self, streams, width, height, local_rank, world, e2e_groups):
        import torch
        import torch.distributed as dist
        from jsmpeg_b200.batch import OUT_DEVICE, OUT_HOST, BatchDecoder
        self.torch, self.dist = torch, dist
        self.OUT_DEVICE, self.OUT_HOST = OUT_DEVICE, OUT_HOST
        self.streams, self.width, self.height = streams, width, height
        self.local_rank, self.world = local_rank, world
        n = len(streams)
        # value: VALUE_GROUPS decoders share the streams; with more than one, each is driven by its own host thread
        self.vgroups = [list(range(g, n, VALUE_GROUPS)) for g in range(VALUE_GROUPS)]
        self.value_decoders = [BatchDecoder(len(g), device=local_rank, max_slots=len(g) * PICTURES + 8) for g in self.vgroups]
        for dec, g in zip(self.value_decoders, self.vgroups):
            for j, i in enumerate(g):
                dec.write(j, streams[i])
            dec.upload()  # elementary streams resident in HBM before the timed region
        # e2e: smaller decoders, one host thread each (ctypes releases the GIL in the C calls)
        e2e_groups = max(1, min(e2e_groups, n))
        self.groups = [list(range(g, n, e2e_groups)) for g in range(e2e_groups)]
        self.e2e_decoders = [BatchDecoder(len(g), device=local_rank, max_slots=len(g) * PICTURES + 8) for g in self.groups]
        for dec, g in zip(self.e2e_decoders, self.groups):  # sequence headers parsed once, like a decoder that has seen its stream start
            for j, i in enumerate(g):
                dec.write(j, streams[i])

    def close(self):
        for d in self.value_decoders + self.e2e_decoders:
            d.close()

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def run_device(self, n_steps):
        if VALUE_GROUPS == 1:
            total = 0
            for _ in range(n_steps):
                self.value_decoders[0].rewind()
                total += self.value_decoders[0].decode(PICTURES, self.OUT_DEVICE)
            return total
        counts = [0] * VALUE_GROUPS

        def work(k):
            dec = self.value_decoders[k]
            for _ in range(n_steps):
                dec.rewind()
                counts[k] += dec.decode(PICTURES, self.OUT_DEVICE)

        threads = [threading.Thread(target=work, args=(k,)) for k in range(VALUE_GROUPS)]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
        return sum(counts)

    def run_e2e(self, n_steps):
        """n_steps whole-workload steps: every group's thread runs its n_steps back to back (no
        per-step join), so one group's PCIe copy-out overlaps the others' write + parse."""
        counts = [0] * len(self.groups)

        def work(k):
            dec = self.e2e_decoders[k]
            for _ in range(n_steps):
                dec.reset()
                for j, i in enumerate(self.groups[k]):
                    dec.write(j, self.streams[i])
                counts[k] += dec.decode(PICTURES, self.OUT_HOST)

        threads = [threading.Thread(target=work, args=(k,)) for k in range(len(self.groups))]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
        return sum(counts)

    def timed(self, run, steps, warmup, decoders):
        """run(n) performs n steps and returns the pictures decoded."""
        torch, dist = self.torch, self.dist
        sampler = ClockSampler(self.local_rank)
        sampler.start()  # started before the warm-up so that it is already streaming samples
        run(warmup)
        self.barrier()
        for d in decoders:
            d.reset_stats()
        sampler.mark()
        t0 = time.perf_counter()
        frames = run(steps)
        self.barrier()
        dt = time.perf_counter() - t0
        clocks = sampler.stop()
        st = {}
        for d in decoders:
            for k, v in d.stats().items():
                st[k] = st.get(k, 0) + v
        if self.world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            fr = torch.tensor([frames], dtype=torch.float64, device="cuda")
            dist.all_reduce(fr, op=dist.ReduceOp.SUM)
            dt, frames = float(t.item()), int(fr.item())
        return frames, dt, st, clocks

    def verify(self, seeds, workers):
        """The last picture of every stream, as the value leg left it in HBM, against the reference's
        decode of the same stream (FNV-1a 64 over Y | Cr | Cb).  Returns a dict for the JSON line."""
        # distinct clips only once on the host
        uniq = {}
        for i, s in enumerate(seeds):
            uniq.setdefault(s, i)
        order = list(uniq.values())
        want = reference_last_hashes([self.streams[i] for i in order], workers)
        want_by_seed = {seeds[i]: w for i, w in zip(order, want)}
        bad, checked = [], 0
        for dec, g in zip(self.value_decoders, self.vgroups):
            for j, i in enumerate(g):
                y, cr, cb = dec.read_planes(j)
                n_ref, h_ref = want_by_seed[seeds[i]]
                checked += 1
                if n_ref != PICTURES or fnv1a64_planes(y, cr, cb) != h_ref:
                    bad.append(i)
        return {"verified": not bad, "streams_checked": checked, "pictures_deep": PICTURES, "mismatching_streams": bad[:16],
                "checker": ("oracle/_ref (unmodified reference C)" if ref_library() is not None else "oracle (C restatement of the reference)")
                           + " on the host, FNV-1a 64 of Y|Cr|Cb of each stream's last picture"}


DUMP_BYTES = 56 << 20  # the sampled planes; with their positions < 64 MB in all


def dump_outputs(directory, legs, prefix=""):
    """What the value leg's last step left for its caller: per stream the Y / Cr / Cb planes of its last picture
    (jsmpeg_b200_batch_read_planes).  All of them would be ~200 MB at 64 x 1080p, so every stream's planes are
    sampled at the same fixed, seeded positions: <name>.npy is float32 [streams, samples], <name>_positions.npy the
    sample positions in the plane (float64)."""
    os.makedirs(directory, exist_ok=True)
    planes = [None] * len(legs.streams)
    for dec, g in zip(legs.value_decoders, legs.vgroups):
        for j, i in enumerate(g):
            planes[i] = dec.read_planes(j)
    per_stream = DUMP_BYTES // 4 // len(planes)
    rng = np.random.default_rng(0)
    for k, name in enumerate(("y", "cr", "cb")):
        size = planes[0][k].size
        pos = np.sort(rng.choice(size, min(size, per_stream * (4 if k == 0 else 1) // 6), replace=False))
        np.save(os.path.join(directory, f"{prefix}{name}.npy"), np.stack([p[k][pos] for p in planes]).astype(np.float32))
        np.save(os.path.join(directory, f"{prefix}{name}_positions.npy"), pos.astype(np.float64))


def roofline_block(st, peak, peak_src, traffic):
    recon_s = st["recon_ms"] / 1e3
    achieved = st["algorithmic_bytes"] / recon_s / 1e9 if recon_s > 0 else 0.0
    return {
        "kernel": "reconstruct_kernel (stage 2: IDCT + motion compensation + add/clamp)",
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak if peak else None, "peak_source": peak_src,
        "algorithmic_bytes_per_launch": st["algorithmic_bytes"] / max(1, st["recon_launches"]),
        "avg_launch_ms": st["recon_ms"] / max(1, st["recon_launches"]),
        "launches": st["recon_launches"],
        "timed": "CUDA events on the reconstruct stream around each chunk's launches; nothing runs beside them in this leg",
        "traffic": traffic["dram_bytes_per_launch"] if traffic else None,
        "traffic_source": traffic["source"] if traffic else None,
    }


def single_stream_leg(es, width, height, device):
    """ONE stream through the 15-function reference ABI (the drop-in use, src/player.js:226-228):
    whole clip written once, then mpeg1_decoder_decode() until false, each call timed on the host."""
    from jsmpeg_b200 import capi
    lib = capi.product_library()
    lib.jsmpeg_b200_set_default_device(device)
    out = {}
    for look in (16, 1):
        os.environ["JSMPEG_B200_LOOKAHEAD"] = str(look)
        per_call = []
        for rep in range(3):  # first repetition = warm-up (allocations, table upload)
            d = lib.mpeg1_decoder_create(len(es) + 16, capi.BIT_BUFFER_MODE_EXPAND)
            ctypes.memmove(lib.mpeg1_decoder_get_write_ptr(d, len(es)), es, len(es))
            lib.mpeg1_decoder_did_write(d, len(es))
            calls = []
            while True:
                t0 = time.perf_counter()
                ok = lib.mpeg1_decoder_decode(d)
                dt = time.perf_counter() - t0
                if not ok:
                    break
                calls.append(dt * 1e3)
            lib.mpeg1_decoder_destroy(d)
            if rep > 0:
                per_call += calls
        per_call.sort()
        n = len(per_call)
        out[f"lookahead_{look}"] = {
            "fps": 1e3 * n / sum(per_call) if per_call else None, "calls": n,
            "ms_per_decode_mean": sum(per_call) / n if n else None,
            "ms_per_decode_p50": per_call[n // 2] if n else None,
            "ms_per_decode_p99": per_call[min(n - 1, int(0.99 * n))] if n else None,
        }
    os.environ.pop("JSMPEG_B200_LOOKAHEAD", None)
    f, s, kind = run_reference_cpu([es], 1, 2)
    out["reference_one_core"] = {"fps": f / s if s > 0 else None, "kind": kind}
    out["what"] = (f"one {width}x{height} stream, {PICTURES} pictures, mpeg1_decoder_create/get_write_ptr/did_write once, then "
                   "mpeg1_decoder_decode() until false; every call ends with the picture's planes in pinned host memory")
    return out


def b_pictures_leg(device, streams, reps=4):
    """The B-picture extension (DESIGN 3.4; the reference skips B pictures): `streams` copies of the committed
    1280x720 I/P/B clip (tests/fixtures/b_clip_1280x720.m1v, written by tools/mini_enc.py), ES resident, the whole
    clip of every stream in one call, device output; the last picture of every stream is hashed against the value
    the oracle gives (tests/fixtures/b_clip_1280x720.json).  Beside it: the same call with the extension off
    (the B pictures consumed and skipped, what the reference does with this stream)."""
    from jsmpeg_b200.batch import OUT_DEVICE, BatchDecoder
    here = os.path.join(ROOT, "tests", "fixtures")
    es = open(os.path.join(here, "b_clip_1280x720.m1v"), "rb").read()
    meta = json.load(open(os.path.join(here, "b_clip_1280x720.json")))
    types = meta["picture_types"]
    out = {"workload": f"{streams} x 1280x720 I/P/B, {types.count(1)} I + {types.count(2)} P + {types.count(3)} B pictures per stream, "
                       "ES resident, one decode call, device output", "unit": "frames/s"}
    # the clip has a slice per macroblock row (45 per picture): third run = the same with the I/P pictures on the
    # one-lane-per-slice walk (option "slice_walk", DESIGN 3.1c)
    for decode_b, slice_walk in ((1, 0), (0, 0), (1, 1)):
        bd = BatchDecoder(streams, device=device, max_slots=streams * len(types) + 8, decode_b=decode_b, slice_walk=slice_walk)
        for s in range(streams):
            bd.write(s, es)
        bd.upload()
        best = None
        for rep in range(reps + 1):  # first repetition = warm-up
            bd.rewind()
            bd.reset_stats()
            t0 = time.perf_counter()
            n = bd.decode(len(types), OUT_DEVICE)
            dt = time.perf_counter() - t0
            st = bd.stats()
            if rep and (best is None or dt < best["wall_ms"] / 1e3):
                best = {"pictures_consumed": n, "pictures_decoded": st["pictures_decoded"], "wall_ms": dt * 1e3,
                        "value": st["pictures_decoded"] / dt, "parse_ms": st["parse_ms"], "reconstruct_ms": st["recon_ms"],
                        "launches": st["kernel_launches"], "parse_errors": st["parse_errors"]}
        if decode_b:
            want = int(meta["fnv1a64"][-1], 16)
            best["verified"] = all(fnv1a64_planes(*bd.read_planes(s)) == want for s in range(streams))
        out[("decode_b_slice_walk" if slice_walk else "decode_b") if decode_b else "skip_b_like_the_reference"] = best
        bd.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="value leg only (used for the ncu launch list)")
    ap.add_argument("--no-extras", action="store_true", help="skip config_720p / single_stream_1080p")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write the value leg's decoded pictures (a fixed sample) as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = env_int("RANK", 0)
    local_rank = env_int("LOCAL_RANK", 0)
    world = env_int("WORLD_SIZE", 1)
    local_world = env_int("LOCAL_WORLD_SIZE", world)
    pix = WIDTH * HEIGHT
    cores = host_cores()
    base_config = {
        "workload": f"{STREAMS_PER_GPU} independent {WIDTH}x{HEIGHT} MPEG-1 I+P elementary streams x {PICTURES} pictures per GPU "
                    f"(BASELINE configs[3]; weak-scaled x N GPUs = configs[4]), GOP 12, one slice per picture",
        "streams_per_gpu": STREAMS_PER_GPU, "pictures_per_stream": PICTURES, "distinct_clips_per_gpu": DISTINCT,
        "parallelism": f"streams sharded {STREAMS_PER_GPU} per GPU, no collective",
        "l2": "inputs larger than L2 (ES + records per step >> 126 MB); no explicit flush",
    }

    if args.impl == "reference":
        if rank != 0:
            return 0
        threads = cores["usable"]
        clips = load_streams(rank_seeds(0, min(threads, STREAMS_PER_GPU)))
        sample = [clips[i % len(clips)] for i in range(threads)]  # one whole clip (all PICTURES pictures) per thread
        for _ in range(min(args.warmup, 1)):
            run_reference_cpu(sample, threads, 1)
        frames, seconds, kind = 0, 0.0, "reference"
        for _ in range(args.steps):
            f, s, kind = run_reference_cpu(sample, threads, 1)
            frames += f
            seconds += s
        fps = frames / seconds
        desc = (f"{threads} threads (usable cores: affinity {cores['affinity']}, cgroup quota {cores['cgroup_quota_cpus']}, "
                f"cpu_count {cores['cpu_count']}) x 1 clip x all {PICTURES} pictures per step ({len(clips)} distinct {WIDTH}x{HEIGHT} "
                f"clips, same streams as the GPU arm); only the decode() loops are timed")
        print(json.dumps({
            "impl": "reference", "metric": "MPEG-1 video decode frames/s", "value": fps, "unit": "frames/s",
            "gpix_per_s": fps * pix / 1e9, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * seconds / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": base_config,
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": kind, "sample": desc, "host": cores},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }))
        return 0

    # NCCL is used for the barrier / counter reduction only; keep its banner off stdout (one JSON line)
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    # this rank's share of the host: the cgroup quota (or the CPU set) divided among the ranks of the node
    per_rank_cores = max(1, cores["usable"] // max(1, local_world))
    # the clips are encoded (worker PROCESSES, cv2) before anything touches CUDA: nothing CUDA is ever forked
    seeds = rank_seeds(rank)
    streams = load_streams(sorted(set(seeds)), workers=per_rank_cores)
    by_seed = dict(zip(sorted(set(seeds)), streams))
    streams = [by_seed[s] for s in seeds]
    streams_720 = None
    if world == 1 and EXTRAS and not args.no_extras:
        s2 = load_streams(sorted(set(seeds)), 1280, 720, workers=per_rank_cores)
        by2 = dict(zip(sorted(set(seeds)), s2))
        streams_720 = [by2[s] for s in seeds]
    # this rank's host side lives on its GPU's NUMA node: threads, pinned bit buffers and plane rings
    from jsmpeg_b200 import capi
    numa = capi.bind_host_to_device(local_rank)
    cores_rank = host_cores()
    cores_rank["per_rank"] = per_rank_cores
    import torch
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.barrier()
    e2e_groups = max(1, min(E2E_GROUPS, per_rank_cores))
    legs = Legs(streams, WIDTH, HEIGHT, local_rank, world, e2e_groups)

    frames, dt, st, clocks = legs.timed(legs.run_device, args.steps, args.warmup, legs.value_decoders)
    verdict = {"verified": None, "why": "--no-verify"}
    if not args.no_verify:
        verdict = legs.verify(seeds, per_rank_cores)
        verdict["lane_walk_pictures_equal_pictures"] = st.get("lane_walk_pictures", 0) == st.get("pictures", -1)
        if world > 1:
            ok = torch.tensor([1.0 if verdict["verified"] and verdict["lane_walk_pictures_equal_pictures"] else 0.0], device="cuda")
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            verdict["all_ranks"] = bool(ok.item() > 0.5)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, legs, "" if world == 1 else f"rank{rank}_")
    e_steps = args.steps
    if args.no_e2e:
        e_frames, e_dt, e_st, e_clocks = 0, 1.0, {"h2d_bytes": 0, "d2h_bytes": 0}, None
    else:
        e_frames, e_dt, e_st, e_clocks = legs.timed(legs.run_e2e, e_steps, 3, legs.e2e_decoders)
    legs.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    fps = frames / dt
    e_fps = e_frames / e_dt
    peak, peak_src = measured_peak()
    traffic = recorded_traffic()
    out = {
        "metric": "MPEG-1 video decode frames/s", "value": fps, "unit": "frames/s",
        "gpix_per_s": fps * pix / 1e9,
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": base_config,
        "clocks": clocks,
        "verified": verdict.get("verified"), "verification": verdict,
        "e2e": {"value": e_fps, "unit": "frames/s", "gpix_per_s": e_fps * pix / 1e9,
                "h2d_bytes_per_step": e_st["h2d_bytes"] // e_steps,
                "d2h_bytes_per_step": e_st["d2h_bytes"] // e_steps,
                "ms_per_step": 1e3 * e_dt / e_steps, "steps": e_steps, "warmup": 3,
                "host_threads": e2e_groups, "numa": numa, "clocks": e_clocks},
        "gpu_launches": st["kernel_launches"], "value_host_threads": VALUE_GROUPS,
        "roofline": roofline_block(st, peak, peak_src, traffic),
        "stage_ms_per_step": {"scan": st["scan_ms"] / args.steps, "parse": st["parse_ms"] / args.steps,
                              "reconstruct": st["recon_ms"] / args.steps},
        "stage1": {"es_mbit_per_s": st["es_bytes"] * 8 / (st["parse_ms"] / 1e3) / 1e6 if st["parse_ms"] else None,
                   "pictures_per_s": st["pictures"] / (st["parse_ms"] / 1e3) if st["parse_ms"] else None,
                   "parse_errors": st["parse_errors"],
                   "walk": os.environ.get("JSMPEG_B200_WALK") or "lanes",
                   "lane_walk_pictures_per_step": st.get("lane_walk_pictures", 0) / args.steps},
        "host": cores_rank,
    }
    if world == 1 and EXTRAS and not args.no_extras:
        # BASELINE configs[1]: 1280x720, the same legs
        w2, h2 = 1280, 720
        legs2 = Legs(streams_720, w2, h2, local_rank, 1, e2e_groups)
        f2, dt2, st2, _ = legs2.timed(legs2.run_device, args.steps, args.warmup, legs2.value_decoders)
        v2 = legs2.verify(seeds, per_rank_cores) if not args.no_verify else {"verified": None}
        if args.no_e2e:
            ef2, edt2 = 0, 1.0
        else:
            ef2, edt2, _, _ = legs2.timed(legs2.run_e2e, e_steps, 3, legs2.e2e_decoders)
        legs2.close()
        out["config_720p"] = {
            "workload": f"{STREAMS_PER_GPU} x {w2}x{h2} x {PICTURES} pictures (BASELINE configs[1] shape, batched like configs[3])",
            "value": f2 / dt2, "unit": "frames/s", "gpix_per_s": f2 / dt2 * w2 * h2 / 1e9, "ms_per_step": 1e3 * dt2 / args.steps,
            "e2e": {"value": ef2 / edt2, "unit": "frames/s", "gpix_per_s": ef2 / edt2 * w2 * h2 / 1e9},
            "roofline": roofline_block(st2, peak, peak_src, None), "verified": v2.get("verified"),
            "stage_ms_per_step": {"scan": st2["scan_ms"] / args.steps, "parse": st2["parse_ms"] / args.steps,
                                  "reconstruct": st2["recon_ms"] / args.steps},
        }
        # BASELINE configs[2]: one 1080p stream through the reference ABI
        out["single_stream_1080p"] = single_stream_leg(streams[0], WIDTH, HEIGHT, local_rank)
        try:  # the opt-in B-picture extension: a side number, never a reason for the bench line to be missing
            out["b_pictures_720p"] = b_pictures_leg(local_rank, STREAMS_PER_GPU)
        except Exception as e:  # noqa: BLE001
            out["b_pictures_720p"] = {"error": f"{type(e).__name__}: {e}"}
    if not args.no_cpu_baseline and world == 1:
        threads = cores_rank["usable"]
        sample = [streams[i % len(streams)] for i in range(threads)]
        f, s, kind = run_reference_cpu(sample, threads, 1)
        out["cpu_baseline"] = {"value": f / s, "unit": "frames/s", "gpix_per_s": f / s * pix / 1e9, "cores": threads,
                               "kind": kind, "host": cores_rank,
                               "sample": f"{threads} threads (usable cores = min(affinity, cgroup quota)) x 1 clip x all {PICTURES} "
                                         f"pictures of the same {WIDTH}x{HEIGHT} clips; only the decode() loops are timed"}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()
    bad = verdict.get("verified") is False or verdict.get("lane_walk_pictures_equal_pictures") is False
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
