"""Records tests/golden/pinning_port_snapshot.json.gz: the plain-C restatement's (oracle/fm_oracle.c) answers to every
call tests/test_oracle_pinning.py makes of the `ref` fixture, replayed there where the reference build (oracle/_ref) is
absent (tests/pinning_snapshot.py).

    python tests/golden/record_pinning_snapshot.py

The snapshot is of the restatement, not of the reference: the reference's sources are not part of the repository.
Record it again only after a deliberate change of the restatement, and only once that change has been checked against
the reference (tests/test_golden.py everywhere; tests/test_oracle_pinning.py live wherever oracle/_ref can be built)."""
import os
import shutil
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402
from tests import pinning_snapshot  # noqa: E402


def private_port(tmp):
    """the restatement on its own copy of the library: the tests drive `port` next to it, and the random streams are
    process-wide state of a loaded library"""
    copy = os.path.join(tmp, os.path.basename(O.lib_path("port")))
    shutil.copy(O.lib_path("port"), copy)
    lib_path = O.lib_path
    O.lib_path = lambda k: copy
    try:
        return O.Oracle("port")
    finally:
        O.lib_path = lib_path


def main():
    if not O.available("port"):
        assert O.build("port"), "cannot build oracle/libfm_oracle.so (oracle/Makefile)"
    import pytest
    with tempfile.TemporaryDirectory() as tmp:
        pinning_snapshot.RECORD_FROM = private_port(tmp)
        rc = pytest.main(["-q", "-p", "no:cacheprovider", os.path.join(ROOT, "tests", "test_oracle_pinning.py")])
        assert rc == 0, "the pinning tests must pass while recording"
        pinning_snapshot.save(pinning_snapshot.RECORDED)
    print("wrote", pinning_snapshot.PATH, os.path.getsize(pinning_snapshot.PATH), "bytes,", len(pinning_snapshot.RECORDED), "tests")


if __name__ == "__main__":
    main()
