import json
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tests import reference  # noqa: E402

_recorded = {}


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.hookimpl(hookwrapper=True)
def pytest_runtest_makereport(item, call):
    rep = (yield).get_result()
    setattr(item, "rep_" + rep.when, rep)


@pytest.fixture(autouse=True)
def reference_digest(request):
    """Folds what the test compares against into one digest and checks it against the one recorded from the reference
    (tests/reference.py)."""
    pins = reference.CURRENT[0] = reference.Pins()
    yield
    rep = getattr(request.node, "rep_call", None)
    if rep is None or not rep.passed:
        return
    if pins.n == 0:
        assert reference.LIVE or not pins.used, "the test used the reference's stand-in but pinned none of its results"
        return
    key = f"{os.path.basename(str(request.node.fspath))}::{request.node.name}"
    if reference.LIVE:
        _recorded[key] = pins.hexdigest()
    want = reference.stored().get(key)
    if want is None and reference.LIVE:
        return
    assert want is not None, f"no digest of the reference's results for {key} in {reference.DIGESTS}"
    assert pins.hexdigest() == want, f"{key}: results differ from the reference's (digest {pins.hexdigest()} != {want})"


def pytest_sessionfinish(session):
    path = os.environ.get("MAB_RECORD_REFERENCE")
    if path and _recorded:
        with open(path, "w") as f:
            json.dump(_recorded, f, indent=0, sort_keys=True)


@pytest.fixture(scope="session")
def built():
    """Everything compiled: product library, oracle port, generator (and oracle/_ref when sources exist)."""
    import __graft_entry__ as ge
    ge.build()
    return True


@pytest.fixture(scope="session")
def ref(built):
    """The unmodified reference where oracle/_ref/ is built, else the oracle port checked against the reference's digests."""
    lib = reference.load()
    lib.set_verbose(0)
    return lib


@pytest.fixture(scope="session")
def prod(built):
    from miniasm_b200 import capi
    lib = capi.load_product(strict=False)
    lib.set_verbose(0)
    return lib


@pytest.fixture(scope="session")
def paf_dir(tmp_path_factory):
    return str(tmp_path_factory.mktemp("paf"))
