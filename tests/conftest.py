import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (a B200)")
    config.addinivalue_line("markers", "needs_reference: needs the original MuDPT project at MUDPT_REFERENCE_ROOT")


def pytest_collection_modifyitems(config, items):
    import torch
    from oracle import ref_shims
    has_gpu = torch.cuda.is_available()
    has_ref = ref_shims.reference_available()
    for it in items:
        if "gpu" in it.keywords and not has_gpu:
            it.add_marker(pytest.mark.skip(reason="no CUDA device"))
        if "needs_reference" in it.keywords and not has_ref:
            it.add_marker(pytest.mark.skip(reason="MUDPT_REFERENCE_ROOT does not name a MuDPT checkout"))
