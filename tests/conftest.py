import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")


@pytest.fixture(scope="session")
def _recorded_files():
    """tests/golden/recorded_<module>.npz, loaded on first use; with INERF_RECORD_GOLDEN=DIR, filled by the tests and written
    to DIR at the end of the session."""
    import numpy as np
    out_dir = os.environ.get("INERF_RECORD_GOLDEN")
    files = {}
    yield files, out_dir
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        for module, store in files.items():
            np.savez_compressed(os.path.join(out_dir, f"recorded_{module}.npz"), **store)


@pytest.fixture
def recorded(request, _recorded_files):
    """helpers.Recorded for the calling test: the reference outputs it compares with."""
    import numpy as np
    from helpers import GOLDEN, Recorded
    files, out_dir = _recorded_files
    module = request.node.module.__name__.rsplit(".", 1)[-1]
    if module not in files:
        path = os.path.join(GOLDEN, f"recorded_{module}.npz")
        files[module] = {} if out_dir else dict(np.load(path))
    return Recorded(files[module], request.node.name, bool(out_dir))


@pytest.fixture(scope="session")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")
