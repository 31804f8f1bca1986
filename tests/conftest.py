import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
for p in (str(ROOT), str(ROOT / "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on a B200)")


@pytest.fixture(scope="session")
def oracle():
    from vp8fix import Oracle, build_oracle
    build_oracle()
    return Oracle()


@pytest.fixture(scope="session")
def reference():
    """The original decoder's library (oracle/_ref, built by oracle/Makefile from the original's sources), or None where it
    is not built: then the tests compare with its digests in tests/golden/ref_checks.json (ref_digests)."""
    from vp8fix import Reference
    return Reference() if Reference.available() else None


@pytest.fixture(scope="session")
def ref_digests():
    import json
    from vp8fix import GOLDEN
    return json.loads((GOLDEN / "ref_checks.json").read_text())


@pytest.fixture(scope="session")
def lib():
    """libvp8gpu.so, built in-tree if stale. Loading it needs no GPU."""
    import importlib
    build = importlib.import_module("webp_decoder_b200.build")
    build.build_library()
    import webp_decoder_b200 as W
    W.load_library()
    return W


@pytest.fixture(scope="session")
def golden():
    import json
    from vp8fix import GOLDEN
    return json.loads((GOLDEN / "digests.json").read_text())


@pytest.fixture(scope="session")
def parsed_golden(lib, golden):
    """All golden .webp inputs parsed by the product's host front end: name -> (kf, frame, keepalive)."""
    from vp8fix import GOLDEN
    from webp_decoder_b200 import parse as P
    names = sorted(golden)
    pf = P.parse_batch([(GOLDEN / "webp" / n).read_bytes() for n in names])
    return {n: (pf.kfs[i], pf.frames[i], pf) for i, n in enumerate(names)}


@pytest.fixture(scope="session")
def gpu_ctx(lib):
    ctx = lib.Context(0)
    yield ctx
    ctx.close()
