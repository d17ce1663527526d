"""pytest configuration: markers and import path."""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch

        has_gpu = torch.cuda.is_available()
    except Exception:  # pragma: no cover
        has_gpu = False
    skip_gpu = pytest.mark.skip(reason="no CUDA device")
    # tools/run_gpu_tests_on_standin.py: the kernels are replaced by tests/fake_ops.py, so the estimator-level gpu
    # tests can check the host logic on a CPU-only machine
    if os.environ.get("CCAB_TESTS_ON_STANDIN") == "1":
        has_gpu = True
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(skip_gpu)
