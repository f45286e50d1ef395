import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: test needs a real B200 (run with -m gpu)")
    # the oracle runs on the host: many-core boxes with a small CPU quota crawl when torch spawns one thread per visible core
    import torch

    torch.set_num_threads(max(1, min(16, os.cpu_count() or 1)))


@pytest.fixture(scope="session")
def golden_dir():
    return os.path.join(ROOT, "tests", "golden")
