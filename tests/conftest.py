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
def port_lib():
    from oracle import okv
    okv.build(ref=False)
    return okv.load_port()


@pytest.fixture(scope="session", autouse=True)
def _built_library():
    """librsp_b200.so is built in-tree (nvcc, sm_100a); rebuild only when sources are newer.  No GPU needed."""
    from rocksplicator_b200 import build
    build.build()


# tests/emul (CPU emulation of the CUDA slice the engine uses — test infrastructure, see tests/emul/include/
# cuda_runtime.h): tests/test_emul_cpu.py re-runs the GPU parity tests in a SUBPROCESS with this variable set, so the
# ctypes binding in that process binds the emulated library instead of librsp_b200.so.  Never set on a GPU box.
if os.environ.get("RSP_TEST_EMUL_LIB"):
    from rocksplicator_b200 import engine as _engine
    _engine.SO_PATH = os.environ["RSP_TEST_EMUL_LIB"]
    if os.environ.get("RSP_TEST_EMUL_ARENA"):  # tiny arena slabs: every device allocation becomes its own malloc (ASan)
        _orig_init = _engine.Engine.__init__

        def _init(self, device=0, max_shards=0, arena_bytes=0, l0_compaction_trigger=0):
            _orig_init(self, device, max_shards, arena_bytes or int(os.environ["RSP_TEST_EMUL_ARENA"]), l0_compaction_trigger)
        _engine.Engine.__init__ = _init
