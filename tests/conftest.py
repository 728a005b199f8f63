import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def oracle():
    from oracle.pyoracle import Oracle, build
    build(ref=True)  # liboracle.so always; oracle/_ref only when /root/reference is present
    return Oracle()


@pytest.fixture(scope="session")
def ref():
    """The compiled reference where oracle/_ref was built; elsewhere its stored results (tests/refgolden.py)."""
    from oracle.pyoracle import Ref
    import refgolden
    if not Ref.available():
        yield refgolden.Replay.load()
        return
    path = os.environ.get("CBS_REF_GOLDEN_RECORD")
    if not path:
        yield Ref()
        return
    rec = refgolden.Recorder(Ref(), path)
    yield rec
    rec.save()


@pytest.fixture(scope="session")
def ctx():
    import genomic_b200
    c = genomic_b200.Context(0)  # raises if the CUDA library or the device is missing: no fallback
    yield c
    c.close()
