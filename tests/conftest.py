import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def built_lib():
    from squid_b200 import build
    return build.build(verbose=False)


REFERENCE_MISSING = "oracle/_ref/squid_ref is missing: it is built from the reference's own sources, which are not part of this repository"


@pytest.fixture(scope="session")
def reference_build():
    """The reference's own sources built against the shims (oracle/_ref/squid_ref), for the tests that check that build itself or
    files only it writes.  SQUID_REQUIRE_ORACLE=1 turns its absence into a failure."""
    from oracle import pyref
    pyref.build()
    if not pyref.available():
        if os.environ.get("SQUID_REQUIRE_ORACLE"):
            pytest.fail(REFERENCE_MISSING, pytrace=False)
        pytest.skip(REFERENCE_MISSING)
    return pyref


@pytest.fixture(scope="session")
def ref_oracle():
    """What the parity tests compare with: the reference build where it is present, else the CPU restatement
    (oracle.pyref.Restated), so that a missing reference never turns a parity test into a skip."""
    from oracle import pyref
    pyref.build()
    if pyref.available():
        return pyref
    if os.environ.get("SQUID_REQUIRE_ORACLE"):
        pytest.fail(REFERENCE_MISSING, pytrace=False)
    pyref.build_restate()
    return pyref.Restated
