import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")


def _cuda_problem():
    """None when the product library is built and finds a usable CUDA device, else the reason."""
    try:
        from jsmpeg_b200 import capi
        lib = capi.product_library()
    except (OSError, FileNotFoundError) as e:
        return f"libjsmpeg_b200.so not loadable: {e}"
    saved = os.dup(2)  # a dead decoder announces itself on stderr; keep the collection output clean
    devnull = os.open(os.devnull, os.O_WRONLY)
    os.dup2(devnull, 2)
    try:
        b = lib.jsmpeg_b200_batch_create(1, int(os.environ.get("JSMPEG_B200_DEVICE", "0")), 2)
        err = lib.jsmpeg_b200_batch_last_error(b)
        lib.jsmpeg_b200_batch_destroy(b)
    finally:
        os.dup2(saved, 2)
        os.close(saved)
        os.close(devnull)
    return err.decode(errors="replace") if err else None


def pytest_collection_modifyitems(config, items):
    gpu_items = [item for item in items if "gpu" in item.keywords]
    problem = _cuda_problem() if gpu_items else None
    for item in gpu_items:
        if problem:  # a plain `pytest tests` on a box without a GPU runs the CPU suite and skips these
            item.add_marker(pytest.mark.skip(reason=f"no usable CUDA device: {problem[:120]}"))
