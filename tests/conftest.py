import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session", autouse=True)
def _built():
    """Build what is buildable here: the oracle always, the reference when its sources are
    mounted, the product library when the .so is missing (nvcc cross-compiles without a GPU)."""
    from oracle import oracle as O
    O.build()
    import gmerlin_avdecoder_b200 as g
    if not os.path.exists(g.LIB_PATH) or not os.path.exists(g.PLUGIN_PATH):
        g.build_library()
    yield

