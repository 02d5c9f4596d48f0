import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on a B200 with -m gpu)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch

        have_gpu = torch.cuda.is_available()
    except Exception:  # pragma: no cover
        have_gpu = False
    for item in items:
        if "gpu" in item.keywords and not have_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))


@pytest.fixture(autouse=True)
def _pin_global_rngs():
    """Every test starts from the same global numpy / torch (CPU and CUDA) generator state: a test that draws without an explicit
    generator sees the same problem instance whatever ran before it."""
    import numpy as np

    np.random.seed(12345)
    try:
        import torch

        torch.manual_seed(12345)
    except Exception:  # pragma: no cover
        pass
    yield
