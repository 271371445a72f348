import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden_block_cases():
    import torch
    d = os.path.join(ROOT, "tests", "golden", "block_cases")      # one file per case, keyed by its name
    return {f[:-len(".pt")]: torch.load(os.path.join(d, f), map_location="cpu", weights_only=False)
            for f in sorted(os.listdir(d)) if f.endswith(".pt")}


@pytest.fixture(scope="session")
def golden_gnn_case():
    import torch
    return torch.load(os.path.join(ROOT, "tests", "golden", "gnn_shipped_weights.pt"), map_location="cpu",
                      weights_only=False)
