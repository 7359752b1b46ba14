import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
# the original GA3C's ga3c/ source directory; not part of this repository
REFERENCE = os.environ.get("GA3C_REFERENCE", "")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (sm_100a)")
    config.addinivalue_line("markers", "reference: imports the original GA3C's own Python from $GA3C_REFERENCE "
                                       "(skipped where it is not set)")


def pytest_collection_modifyitems(config, items):
    have_ref = os.path.isdir(REFERENCE)
    for item in items:
        if "reference" in item.keywords and not have_ref:
            item.add_marker(pytest.mark.skip(reason="GA3C_REFERENCE does not name the original GA3C's ga3c/ directory"))


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN
