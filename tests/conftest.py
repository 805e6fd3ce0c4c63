import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _has_cuda() -> bool:
    try:
        import torch

        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    has = None
    for item in items:
        if "gpu" in item.keywords:
            if has is None:
                has = _has_cuda()
            if not has:
                item.add_marker(pytest.mark.skip(reason="no CUDA device"))


@pytest.fixture(scope="session")
def gold_dir():
    return GOLD


def load_golden_json(name):
    with open(os.path.join(GOLD, name)) as fh:
        return json.load(fh)


def load_golden_counts(name):
    return np.load(os.path.join(GOLD, f"{name}.npz"))["counts"]


@pytest.fixture(scope="session")
def host_libs():
    """Build the host and oracle libraries once per session (gcc only, no GPU needed)."""
    from trueconsense_b200 import build
    from oracle import pileup

    build.build_host()
    pileup.build()
    return True
