import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: needs the original multiagent-rl-rm sources (RLRM_REFERENCE_ROOT)")


def golden_names():
    """Training-trace fixtures (eval_*.npz: tests/test_eval.py, mdp_*.npz: tests/test_mdp.py)."""
    return sorted(f[:-4] for f in os.listdir(GOLDEN_DIR) if f.endswith(".npz") and not f.startswith(("eval_", "mdp_")))


def load_golden(name):
    import json

    import numpy as np

    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    meta = json.loads(str(z["meta"]))
    return meta, {k: z[k] for k in z.files if k != "meta"}


@pytest.fixture(scope="session")
def cuda_device():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")
