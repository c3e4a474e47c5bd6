import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def compiled_reference():
    """The unmodified reference (oracle/_ref/libkaori_ref.so), built only where its sources exist: for the tests that
    check the C restatement against it."""
    from oracle import kref as m
    if not m.available():
        pytest.skip("oracle/_ref/libkaori_ref.so not built")
    return m


@pytest.fixture(scope="session")
def kref(port):
    """The yardstick of the product's tests: the compiled reference where it was built, else the C restatement, which
    tests/test_golden_fixtures.py pins to the reference's stored outputs, so that these tests run on any checkout."""
    from oracle import kref as m
    return m if m.available() else port


@pytest.fixture(scope="session")
def port():
    from oracle import port as m
    if not m.available():
        import subprocess
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "liboracle.so"])
    return m
