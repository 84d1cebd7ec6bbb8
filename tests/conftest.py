import os
import shutil
import sys
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def built():
    """Build the CUDA library and the oracle once per session (nvcc cross-compiles without a GPU)."""
    import __graft_entry__ as g

    g.build()
    return True


@pytest.fixture(scope="session")
def oracle(built):
    from oracle import oracle as O

    O.lib()
    return O


@pytest.fixture()
def engine(built):
    import fma_b200

    eng = fma_b200.Engine(0)
    yield eng
    eng.close()


@pytest.fixture()
def sock_dir():
    """A directory for unix sockets.  An AF_UNIX path holds at most 107 bytes, which a socket under tmp_path exceeds when the
    temporary directory has a long name, so the sockets go to a short directory under /tmp."""
    d = tempfile.mkdtemp(prefix="fma-", dir="/tmp")
    yield d
    shutil.rmtree(d, ignore_errors=True)
