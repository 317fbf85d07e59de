import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# a checkout of the original Rust project (rusty-marcher), for the tests that need its sources; they skip without one
REFERENCE = os.environ.get("RM_REFERENCE_DIR", "")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


def pytest_collection_modifyitems(config, items):
    """A GPU test that hangs (a kernel that never retires blocks the host in cudaStreamSynchronize, out of reach of
    Python) must cost minutes, not the session: with pytest-timeout present every GPU test gets a hard limit enforced
    from a watchdog thread, which ends the process."""
    if not config.pluginmanager.hasplugin("timeout"):
        return
    for item in items:
        if item.get_closest_marker("gpu") and not item.get_closest_marker("timeout"):
            item.add_marker(pytest.mark.timeout(300, method="thread"))


def has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.fixture(scope="session")
def reference_dir():
    if not os.path.isdir(REFERENCE):
        pytest.skip("RM_REFERENCE_DIR does not name a checkout of the original rusty-marcher project")
    return REFERENCE


@pytest.fixture(scope="session")
def rm_gpu():
    """The product package bound to cuda:0 -- fails loudly (no fallback) if there is no GPU."""
    import rusty_marcher_b200 as rm
    rm.init(0)
    return rm
