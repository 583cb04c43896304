import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def oracles():
    """The CPU checkers (test infrastructure). Builds them if needed; `ref` may be unavailable."""
    import oracle

    oracle.build(ref=oracle.reference_sources_present())
    return oracle


@pytest.fixture(scope="session")
def handle():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import libbicos_b200 as lb

    if not os.path.exists(lb.capi.LIB_PATH):
        import __graft_entry__

        __graft_entry__.build()
    return lb.Handle(0)
