import os
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if os.path.dirname(os.path.abspath(__file__)) not in sys.path:
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

GOLDEN = os.path.join(REPO, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(autouse=True)
def _deterministic_library_knobs():
    """Every test starts from the same library state: cuDNN heuristics (no per-box autotune),
    deterministic algorithms, fp32 (no TF32) convolutions and matmuls.  A test that checks the
    benchmarked configuration (TF32 convs, cuDNN autotune) switches them on itself; whatever a
    test (or `Learner.__init__`, which honours cfg.CUDNN_BENCHMARK) changed is undone here."""
    import torch
    saved = (torch.backends.cudnn.benchmark, torch.backends.cudnn.deterministic,
             torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.benchmark = False
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    (torch.backends.cudnn.benchmark, torch.backends.cudnn.deterministic,
     torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32) = saved


@pytest.fixture(scope="session")
def golden():
    def load(name):
        return np.load(os.path.join(GOLDEN, name + ".npz"))
    return load
