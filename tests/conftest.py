import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
GOLDEN_THREADS = 8


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        have_gpu = torch.cuda.is_available()
    except Exception:  # pragma: no cover
        have_gpu = False
    # a GPU test that deadlocks (a device-side wait that never returns blocks the host in a CUDA call) must not take the whole
    # session with it for longer than this: pytest-timeout's thread method ends the process (default per-test budget, overridable)
    have_timeout = config.pluginmanager.hasplugin("timeout") and not config.getoption("timeout", None)
    for it in items:
        if have_timeout and "gpu" in it.keywords and it.get_closest_marker("timeout") is None:
            it.add_marker(pytest.mark.timeout(300, method="thread"))
        if "gpu" in it.keywords and not have_gpu:
            it.add_marker(pytest.mark.skip(reason="no CUDA device"))


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


@pytest.fixture(scope="module")
def golden_threads():
    """Bit-exact comparisons with the goldens run with the intra-op thread count the goldens were written with
    (tests/golden/make_golden*.py): ATen's CPU convolutions and reductions split their sums by thread count, so on a host
    that defaults to another count the last bits differ."""
    import torch
    saved = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(saved)
