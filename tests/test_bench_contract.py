"""bench.py's reference arm and JSON contract, on a tiny configuration (no GPU needed)."""
import json
import os
import subprocess
import sys

import helpers

REQUIRED = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline", "impl"]


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ, BENCH_WIDTH="320", BENCH_HEIGHT="240", BENCH_PICTURES="12", BENCH_DISTINCT="2",
               BENCH_STREAMS="4", BENCH_REF_PICTURES="6")
    out = subprocess.run([sys.executable, os.path.join(helpers.ROOT, "bench.py"), "--impl", "reference", "--gpus", "1",
                          "--steps", "2", "--warmup", "1"], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in REQUIRED:
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert "workload" in d["config"]
    # the core count is the honest one: never more than the scheduler affinity or the cgroup CPU quota allow
    host = d["cpu_baseline"]["host"]
    assert d["cpu_baseline"]["cores"] == host["usable"] <= host["affinity"] <= host["cpu_count"]
    if host["cgroup_quota_cpus"]:
        assert host["usable"] <= max(1, int(host["cgroup_quota_cpus"] + 1e-6))
    assert d["value"] * d["ms_per_step"] > 0


def test_checker_hash_is_fnv1a64_of_the_planes():
    """bench.py's `verified` and the GPU tests compare pictures by FNV-1a 64 of Y | Cr | Cb; pin the function to the
    textbook FNV-1a 64 on a small buffer, and the hashes of a clip's pictures to the ones the reference's harness
    (oracle/ref_bench.c: ref_picture_hashes, recorded in tests/golden/reference/picture_hashes.json) gave."""
    import numpy as np
    sys.path.insert(0, helpers.ROOT)
    import bench
    data = np.frombuffer(b"jsmpeg_b200 fnv check", dtype=np.uint8).copy()
    h = 1469598103934665603
    for byte in data.tobytes():
        h = ((h ^ byte) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    assert bench.oracle_library().oracle_hash_bytes(1469598103934665603, data.ctypes.data, data.size) == h
    es = b"".join(p for _, p in helpers.clip_packets(176, 144, 5, seed=3, noise=4))
    want = helpers.reference_golden("picture_hashes")["176x144x5"]
    assert helpers.digest(es) == want["es"]
    frames, _, d = helpers.decode_all(helpers.oracle_lib(), [(0, es)])
    assert [format(bench.fnv1a64_planes(*f), "016x") for f in frames] == want["fnv1a64"]
    d.destroy()
    # the last-picture hash bench.py's `verified` computes where the reference build is absent
    assert bench.oracle_last_hash(bench.oracle_library(), es) == (5, int(want["fnv1a64"][-1], 16))


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(helpers.ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         env=env, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == ""
