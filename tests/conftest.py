import os
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session", autouse=True)
def _built():
    """CPU-side artefacts (oracle, host-sim, product .so) are built once per session; idempotent."""
    import __graft_entry__ as g
    g.build()
    yield
