import os
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: test needs a CUDA device (a B200)")


def pytest_collection_modifyitems(config, items):
    import torch

    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.hookimpl(hookwrapper=True)
def pytest_runtest_protocol(item, nextitem):
    """Tests not marked ``gpu`` are the CPU tier: they run on the CPU also where a GPU is visible (layers would otherwise
    default to it), in this process and in the processes they start, so that they check the same code on every
    machine.  Set around the whole protocol so that module-scoped fixtures are built on the CPU too."""
    if "gpu" in item.keywords:
        yield
        return
    import torch

    with pytest.MonkeyPatch.context() as mp:
        mp.setenv("CUDA_VISIBLE_DEVICES", "")
        mp.setattr(torch.cuda, "is_available", lambda: False)
        yield


@pytest.fixture(autouse=True)
def _fresh_topology():
    """Every test starts from the default (single process) topology."""
    from libai_b200.utils import distributed as dutil

    dutil.reset_dist_util()
    yield
    dutil.reset_dist_util()
