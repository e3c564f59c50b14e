import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu under gpurun)")


@pytest.fixture(scope="session")
def golden():
    import numpy as np
    import torch

    def load(name):
        path = os.path.join(ROOT, "tests", "golden", name + ".npz")
        with np.load(path) as z:
            return {k: torch.from_numpy(z[k]) for k in z.files}
    return load


@pytest.fixture
def golden_threads():
    """CPU results are bit-exact only at the torch thread count the golden vectors were
    generated with (oracle/make_golden.py), whatever the machine's core count."""
    import torch
    from oracle.make_golden import GOLDEN_THREADS
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.fixture(autouse=True)
def _inference_mode_for_gpu_tests(request):
    """The engine is forward-only and refuses to run with grad enabled on parameters that
    require grad (it would silently return detached tensors); the reference's eval loop runs
    under torch.no_grad() (eval.py:213) and so do the GPU tests."""
    if request.node.get_closest_marker("gpu") is None:
        yield
        return
    import torch
    with torch.no_grad():
        yield
