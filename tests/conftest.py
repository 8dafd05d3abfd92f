import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `pytest -m gpu`)")


@pytest.hookimpl(hookwrapper=True)
def pytest_runtest_makereport(item, call):
    rep = (yield).get_result()
    if call.when == "call":
        item.passed_call = rep.passed


@pytest.fixture
def reftape(request):
    """the reference side of a comparison, live from oracle/_ref or replayed from tests/golden/ref (tests/_reftape.py)"""
    import _reftape
    t = _reftape.Tape(request.node.path.stem, request.node.name)
    yield t
    if getattr(request.node, "passed_call", False):
        t.close()


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _has_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)
