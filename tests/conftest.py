import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu)")


@pytest.fixture(scope="session")
def port():
    """plain-C restatement oracle (always buildable)"""
    from oracle import oracle as O
    if not O.available("port"):
        assert O.build("port"), "could not build oracle/libfm_oracle.so"
    return O.Oracle("port")


@pytest.fixture
def ref(request):
    """the reference's own headers compiled unmodified (oracle/_ref) where that build exists; elsewhere a replay of the
    plain-C restatement's recorded answers to the same calls (tests/pinning_snapshot.py), not the reference"""
    from oracle import oracle as O
    from tests import pinning_snapshot
    if pinning_snapshot.RECORD_FROM is not None:
        yield pinning_snapshot.Recorder(pinning_snapshot.RECORD_FROM, request.node.nodeid, pinning_snapshot.RECORDED)
    elif O.available("ref"):
        yield O.Oracle("ref")
    else:
        replay = pinning_snapshot.Replay(request.node.nodeid)
        yield replay
        replay.finish()


@pytest.fixture(scope="session")
def gpu_ctx():
    """engine context on cuda:0 -- fails loudly if the CUDA extension is missing"""
    from fmwr_b200 import _lib
    return _lib.Context(0)
