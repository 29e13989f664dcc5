import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# games whose device implementation exists (extended as games land)
IMPLEMENTED = ["maze", "coinrun", "bossfight", "climber", "chaser", "caveflyer", "jumper"]


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box: pytest -m gpu)")


@pytest.fixture
def reference(request):
    """Reference environments for a parity test (tests/reference.py): the compiled reference when oracle/_ref is built,
    else the host-sim stand-in; what they return is checked against the test's recorded tape when it ends."""
    from oracle import build_ref
    from tests.reference import Reference
    build_ref.build()
    ref = Reference(request.node.nodeid)
    yield ref
    ref.finish()


def golden(game):
    import numpy as np
    return np.load(os.path.join(ROOT, "tests", "golden", "%s.npz" % game))
