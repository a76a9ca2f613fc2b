import os
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
# the host-buffer pipeline sizes its chunks by the postings a batch references (engine.cu: chunk_postings); the test indexes are tiny, so
# without this every batch would take the single-call form and the chunked path would go untested
os.environ.setdefault("TRN_CHUNK_POSTINGS", "1")
os.environ.setdefault("TRN_CHUNK_RULE", "postings")  # (and keep it from being resized by the previous batch's tiny result)
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")


@pytest.fixture(scope="session", autouse=True)
def _native_built():
    # build (or reuse) the in-tree native library; no CPU fallback exists
    from trinity_b200.build import build_native
    build_native()
    yield


@pytest.fixture(scope="session")
def ref():
    """The reference's outputs: its own code (oracle/_ref/libtrinity_ref.so) while recording, tests/golden/reference_calls.json.gz
    otherwise (refharness.py).  TEST-ONLY."""
    from refharness import load_golden_ref
    return load_golden_ref()


@pytest.fixture(scope="session")
def real_ref():
    """The reference's own code, for tests that run it rather than compare with its outputs; build() makes oracle/_ref only where the
    reference sources are readable, elsewhere these tests skip."""
    from refharness import load_ref, reference_built
    if not reference_built():
        pytest.skip("oracle/_ref (the reference's own code) is not built here")
    return load_ref()
