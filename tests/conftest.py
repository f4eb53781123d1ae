import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "pytorch-studiogan_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session", autouse=True)
def golden_cpu_threads():
    """The golden vectors were recorded on 8 CPU threads.  Some CPU results round differently with the thread count (the
    LAPACK QR behind the seeded orthogonal initialisation, the reductions behind analytically-zero bias gradients), and the
    tests that pin them bit for bit or at round-off level hold only at that count."""
    import torch
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


@pytest.fixture(scope="session")
def golden_dir():
    return os.path.join(ROOT, "tests", "golden")
