"""pytest configuration: the `gpu` marker, and one-time builds of the product library and the
oracle (the checker).  `-m "not gpu"` runs here on CPU; `-m gpu` runs on a B200."""
import os
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    # build the product (.so in-tree), the C restatement and, where oracle/reference/ holds the reference, oracle/_ref
    from nmslib_zig_b200 import build as nb_build
    nb_build.build()
    from oracle import oracle as O
    O.build()


def pytest_collection_modifyitems(config, items):
    import nmslib_zig_b200 as nb
    have_gpu = nb.device_available()
    skip = pytest.mark.skip(reason="no CUDA device visible")
    for item in items:
        if "gpu" in item.keywords and not have_gpu:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden_dir():
    return ROOT / "tests" / "golden"
