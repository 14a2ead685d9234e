import shutil
import sys
import tempfile
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def ctx():
    """One amplisolve_b200 context on cuda:0.  GPU tests fail (not skip) without the native library."""
    from amplisolve_b200 import Context
    c = Context(0)
    yield c
    c.close()


@pytest.fixture
def socket_path():
    """A path for the resident service's UNIX socket.  sun_path holds at most 107 bytes, which a pytest tmp_path under a deep
    TMPDIR or checkout exceeds, so the socket lives in a fresh directory of its own under /tmp."""
    d = tempfile.mkdtemp(prefix="as_sock_", dir="/tmp")
    try:
        yield str(Path(d) / "as.sock")
    finally:
        shutil.rmtree(d, ignore_errors=True)
