import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

_REF_RECORDING = {}


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def oracle():
    from oracle import pyoracle
    return pyoracle.Oracle()


@pytest.fixture(scope="session")
def _ref_source(oracle):
    """libref.so where it is built or buildable, else the oracle's stand-in for it (tests/refrecord.py)."""
    from oracle import pyoracle
    from tests import refrecord
    return refrecord.Ref() if pyoracle.have_ref() else refrecord.StandIn(oracle)


@pytest.fixture
def ref(request, _ref_source):
    """The reference, every call recorded (CPROC_REF_RECORD=<file>) or checked against tests/golden/ref_calls.json."""
    from tests import refrecord
    module_rng = getattr(request.module, "rng", None)
    key = request.node.nodeid
    if os.environ.get("CPROC_REF_RECORD"):
        entry = _REF_RECORDING.setdefault(key, {"calls": []})
        if module_rng is not None:
            entry["rng"] = module_rng.bit_generator.state
        return refrecord.Recorded(_ref_source, entry["calls"], "record")
    entry = refrecord.load().get(key)
    if entry is None:
        if isinstance(_ref_source, refrecord.StandIn):
            pytest.fail("%s has no record in tests/golden/ref_calls.json: write it with tests/golden/gen_golden_ref.py" % key)
        return _ref_source                                               # a new test, run against libref.so alone
    if module_rng is not None and "rng" in entry:
        module_rng.bit_generator.state = entry["rng"]                   # the draws of a whole-file run, whatever runs before
    return refrecord.Recorded(_ref_source, entry["calls"], "check")


def pytest_sessionfinish(session):
    path = os.environ.get("CPROC_REF_RECORD")
    if path and _REF_RECORDING:
        from tests import refrecord
        refrecord.save(path, _REF_RECORDING)
