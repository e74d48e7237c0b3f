import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on the B200 box)")
    import torch
    # the CPU oracle is many small torch ops: on a 100+-core host the default thread count is several times SLOWER than 16 threads
    torch.set_num_threads(min(torch.get_num_threads(), 16))


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)
