import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture
def ref(request):
    """The reference CPU path (oracle/ref.py) for this test: its stored outputs, or the live library while recording
    them (tests/reference_outputs.py). Checker only."""
    from reference_outputs import Reference
    node = request.node
    return Reference(os.path.relpath(str(node.path), ROOT).replace(os.sep, "/") + "::" + node.name)


def pytest_sessionfinish(session):
    from reference_outputs import RECORD, STORE
    if RECORD and STORE.recorded:
        STORE.save()
