import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
# the reference's test voice (27 MB, too large to store) where build() staged it; its config and sentences are stored
REAL_VOICE = os.path.join(ROOT, "oracle", "_ref", "voice", "test_voice.onnx")
REAL_VOICE_CONFIG = os.path.join(GOLDEN, "reference", "test_voice.onnx.json")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


def real_voice_path():
    return REAL_VOICE if os.path.exists(REAL_VOICE) else None


def real_fixture_lines():
    import json
    return [json.loads(l) for l in open(os.path.join(GOLDEN, "reference", "test_en-us.jsonl"))]


@pytest.fixture(scope="session")
def lib_built():
    """Build the C-ABI library once per session (nvcc cross-compiles without a GPU)."""
    from piper_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.load()
