import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# Kimera-VIO's shipped rig files and test fixtures, stored by tests/golden/make_reference_fixtures.py
REF = os.path.join(ROOT, "tests", "golden", "reference")
REF_DATA = os.path.join(REF, "data")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


def pytest_collection_modifyitems(config, items):
    # GPU tests are skipped (not failed) when no CUDA device is visible.
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device visible")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)
