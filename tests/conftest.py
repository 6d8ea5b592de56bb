import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import oracle_lib  # noqa: E402


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session", autouse=True)
def _build_oracles():
    # building the checkers is not using them; the reference build only happens where /root/reference is mounted
    oracle_lib.build_oracles()


@pytest.fixture(scope="session")
def port():
    return oracle_lib.Oracle("port")


@pytest.fixture(scope="session")
def ref():
    try:
        return oracle_lib.Oracle("ref")
    except FileNotFoundError:
        pytest.skip("oracle/_ref not built (no /root/reference on this box and no prebuilt library)")


PINNING = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pinning.npz")


@pytest.fixture(scope="session")
def _pinning_store():
    """The recorded oracle outputs of tests/golden/pinning.npz; while tests/golden/make_golden.py pinning runs the tests
    (SLB_RECORD_PINNING = the file to write), an empty store that is written out at the end of the session."""
    out = os.environ.get("SLB_RECORD_PINNING")
    if not out:
        yield dict(np.load(PINNING))
        return
    store = {}
    yield store
    np.savez_compressed(out, **store)


@pytest.fixture
def ref_or_recorded(request, _pinning_store):
    """The reference build when it exists; otherwise the outputs recorded for this test's own inputs (oracle_lib.Recorded)."""
    try:
        live = oracle_lib.Oracle("ref")
    except FileNotFoundError:
        live = None
    if os.environ.get("SLB_RECORD_PINNING"):
        live = live or oracle_lib.Oracle("port")
        _pinning_store["source"] = np.array(live.kind)
        return oracle_lib.Recorded(_pinning_store, request.node.name, live=live)
    return live or oracle_lib.Recorded(_pinning_store, request.node.name)


@pytest.fixture(scope="session")
def best_oracle():
    """The strongest checker present: the reference build when it exists, else the port."""
    try:
        return oracle_lib.Oracle("ref")
    except FileNotFoundError:
        return oracle_lib.Oracle("port")


@pytest.fixture
def rng():
    return np.random.Generator(np.random.PCG64(0x5E1E217E))
