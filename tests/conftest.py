import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: needs a checkout of the reference project (SMZ_REFERENCE_ROOT)")


def pytest_collection_modifyitems(config, items):
    from oracle import ref_import
    have_ref = ref_import.available()
    skip_ref = pytest.mark.skip(reason="SMZ_REFERENCE_ROOT does not name a checkout of the reference project")
    for item in items:
        if "reference" in item.keywords and not have_ref:
            item.add_marker(skip_ref)
