import os
import sys
import warnings

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
warnings.filterwarnings("ignore")

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden():
    import torch

    import seeded_inputs

    cache = {}

    def load(name):
        if name not in cache:
            data = torch.load(os.path.join(GOLDEN, name + ".pt"), map_location="cpu", weights_only=False)
            cache[name] = seeded_inputs.restore(name, data)
        return cache[name]

    return load
