import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run them with: pytest -m gpu)")
    config.addinivalue_line("markers", "needs_reference: needs the original project's code (oracle/ref_shim.py REFERENCE_ROOT)")


def pytest_collection_modifyitems(config, items):
    from oracle import ref_shim
    if ref_shim.reference_available():
        return
    skip_ref = pytest.mark.skip(reason=f"the original project is not at {ref_shim.REFERENCE_ROOT} (RCD_REFERENCE_ROOT names it)")
    for item in items:
        if "needs_reference" in item.keywords:
            item.add_marker(skip_ref)
