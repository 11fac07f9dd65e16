import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: executes the unmodified reference checkout at oracle/_ref/ (skipped when absent)")


@pytest.fixture(scope="session")
def small_scene():
    from dynamicfusion_body_b200 import synth
    return synth.make_scene(res=48, k=4, n_nodes=300, seed=0, rows=120, cols=160)
