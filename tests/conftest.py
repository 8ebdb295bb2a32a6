import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu on the GPU box")


@pytest.fixture(autouse=True)
def _seed_everything(request):
    """Every test starts from the same random state: model initialisation (torch's orthogonal init) must not vary from run to run.  The DQN
    family's double-Q argmax is discontinuous -- a GPU / oracle difference of 1e-7 in two nearly tied online Q-values selects a different target
    action and moves the gradient by ~1/filled-steps -- so an unseeded initialisation made ~8 % of the random cases fail at random
    (tools/grad_stress.py).  Tests that compare against the oracle additionally check the oracle's argmax margin (oracle.learner_ref.double_q_margin)."""
    import random

    import numpy as np

    random.seed(12345); np.random.seed(12345)
    threads = None
    try:
        import torch

        torch.manual_seed(12345)
        threads = torch.get_num_threads()
    except ImportError:
        pass
    yield
    # run.main pins torch to one thread like the reference (run.py:29).  The CPU oracle's float32 reductions (bias gradients: sums over ~13k rows)
    # are sequential in that mode and carry ~1e-5 of rounding error of their own, which made an oracle comparison that ran AFTER a driver test fail
    # at 1.5e-5 while passing (7e-7) on its own: the thread count is process state and must not leak between tests.
    if threads is not None:
        import torch

        if torch.get_num_threads() != threads:
            torch.set_num_threads(threads)
