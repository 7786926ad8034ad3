import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    import torch

    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def golden():
    import torch

    def load(name):
        g = torch.load(os.path.join(GOLDEN, name), weights_only=False)
        # a fixture that would exceed 1 MB keeps some top-level entries in side files <stem>.<key>.pt (oracle/make_golden.py)
        for key in g.pop("_parts", ()):
            g[key] = torch.load(os.path.join(GOLDEN, f"{name[:-3]}.{key}.pt"), weights_only=False)
        return g

    return load
