import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def pkg():
    import importlib
    return importlib.import_module("creating-2d-laser-slam-from-scratch_b200")


@pytest.hookimpl(hookwrapper=True)
def pytest_runtest_makereport(item, call):
    rep = (yield).get_result()
    if rep.when == "call":
        item.call_passed = rep.passed


@pytest.fixture
def reference(request):
    """The reference build (oracle/_ref/) where it was compiled, its recorded answers elsewhere (reference_replay.py)."""
    import reference_replay
    from oracle import ref, ref_gmapping, ref_hector
    live = ref.available() and ref_gmapping.available() and ref_hector.available()
    s = reference_replay.Session(request.module.__name__, request.node.name, live,
                                 record=os.environ.get("B2S_RECORD_REFERENCE") == "1")
    yield s
    if getattr(request.node, "call_passed", False):
        s.finish()
