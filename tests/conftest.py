"""pytest wiring: `-m "not gpu"` runs on the CPU-only build container, `-m gpu` on a B200 box."""
import os
import sys

import pytest

REPO = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
PKG = os.path.join(REPO, "second.pytorch_b200")
for p in (REPO, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def oracle():
    """the CPU oracle `spconv` package (test infrastructure), loaded under an alias."""
    from b2second import loader
    return loader.oracle_spconv()


@pytest.fixture(scope="session")
def product():
    """the CUDA `spconv` drop-in; loading fails loudly if libb2second.so is missing."""
    from b2second import loader
    mod = loader.product_spconv()
    mod._lib.load()
    return mod


@pytest.fixture(scope="session")
def out_dir():
    d = os.path.join(REPO, "gpurun_out")
    os.makedirs(d, exist_ok=True)
    return d

