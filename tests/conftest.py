import os
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
for _p in (str(ROOT), str(ROOT / "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)
os.environ.setdefault("PYTHONDONTWRITEBYTECODE", "1")

# The golden network tensors were recorded from PyTorch's float32 CPU convolutions (oneDNN) with 8 threads on an
# AVX-512 host, and the oracle tests reproduce them bit for bit or to 2e-5.  oneDNN's blocking, and with it the
# float32 summation order, changes with the thread count (below 8) and with the instruction set it dispatches to,
# so both are fixed here, before the first convolution: 8 threads on any host, AVX-512 kernels at most.
os.environ.setdefault("ONEDNN_MAX_CPU_ISA", "AVX512_CORE")
import torch  # noqa: E402

torch.set_num_threads(8)

GOLDEN = ROOT / "tests" / "golden"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def golden():
    import numpy as np

    def load(name):
        return np.load(GOLDEN / name, allow_pickle=False)
    return load


@pytest.fixture(scope="session")
def lib():
    """The C-ABI library, built in-tree if needed (nvcc cross-compiles without a GPU)."""
    from yolo_nano_b200 import build, _lib
    build.build()
    return _lib.load()
