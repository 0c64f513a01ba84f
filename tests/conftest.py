import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def built():
    """Everything compiled: product library, host check helper, oracle (and _ref when possible)."""
    import __graft_entry__ as ge
    ge.build()
    return True


@pytest.fixture(scope="session")
def oracle(built):
    from oracle import Oracle
    return Oracle()


@pytest.fixture(scope="session")
def reference_digests():
    """What the unmodified reference computes on the inputs of the tests that compare with it (SHA-256 digests,
    written by tests/golden/make_reference_digests.py): those tests run without a build of the reference."""
    import json
    with open(os.path.join(GOLDEN, "reference_digests.json")) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def fixture_jpeg():
    with open(os.path.join(GOLDEN, "JPEG_example_JPG_RIP_050.jpg"), "rb") as f:
        return f.read()


@pytest.fixture(scope="session")
def decoder(built):
    import ocljpegdecoder_b200 as b2j
    return b2j.Decoder(0)
