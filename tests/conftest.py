import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(autouse=True)
def _reset_kernel_options(request):
    """GPU tests flip process-wide kernel selectors (omt_set_option); restore the defaults afterwards."""
    yield
    if request.node.get_closest_marker("gpu") is None:
        return
    try:
        from omnitokenizer_b200 import _cabi
        if _cabi._lib is not None:
            for name, value in _cabi.DEFAULT_OPTIONS.items():
                _cabi.set_option(name, value)
    except Exception:
        pass
