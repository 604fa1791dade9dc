import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "timeout: per-test limit (pytest-timeout)")


@pytest.fixture(scope="session")
def oracles():
    """Build the CPU checkers (restatement always; the compiled reference where /root/reference is)."""
    from oracle import bindings
    bindings.build()
    return bindings


@pytest.fixture()
def sock_dir():
    """A fresh directory for Unix domain sockets, removed afterwards.  A socket's path must fit sun_path
    (108 bytes), which a path under pytest's tmp_path does not when TMPDIR is deep, so it lives under /tmp."""
    import pathlib
    import shutil
    import tempfile
    d = tempfile.mkdtemp(prefix="oim-", dir="/tmp")
    yield pathlib.Path(d)
    shutil.rmtree(d, ignore_errors=True)


@pytest.fixture(scope="session")
def gpu():
    """liboimgpu.so initialised on cuda:0.  Fails loudly when the extension is missing."""
    import torch
    assert torch.cuda.is_available(), "gpu-marked test without a CUDA device"
    from oim_b200 import build, lib
    build.build()
    torch.cuda.init()
    torch.zeros(1, device="cuda:0")
    lib.init([0])
    yield lib
    lib.fini()
