import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    # the C-ABI library is a build artefact (git-ignored); compile it once if this checkout does not have it yet
    from opticalflowdiffusion_b200 import build as fd_build
    if not os.path.exists(fd_build.LIB):
        fd_build.build()


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:  # pragma: no cover
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


GOLDEN_THREADS = 8       # intra-op threads the goldens were computed with (oracle/make_goldens.py)


@pytest.fixture
def golden_threads():
    """Run the test on GOLDEN_THREADS CPU threads.  The CPU convolutions split their sums by thread count, and the oracle
    tests' fp32 tolerances against the reference's goldens are set at the last bits of that summation order."""
    import torch
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.fixture(scope="session")
def golden():
    import numpy as np

    def load(name):
        return np.load(os.path.join(GOLDEN, name + ".npz"))
    return load
