import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device")
    config.addinivalue_line("markers", "multigpu: needs at least 2 CUDA devices; skipped elsewhere")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        # tests that need several GPUs skip on a single-GPU machine; their single-GPU stand-ins are
        # tests/test_tp_loopback_gpu.py
        if torch.cuda.device_count() < 2:
            skip_multi = pytest.mark.skip(reason="needs at least 2 CUDA devices")
            for item in items:
                if "multigpu" in item.keywords:
                    item.add_marker(skip_multi)
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)
