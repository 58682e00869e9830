import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: needs the read-only reference tree at /root/reference")


def pytest_collection_modifyitems(config, items):
    import torch
    have_gpu = torch.cuda.is_available()
    for item in items:
        if "gpu" in item.keywords and not have_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device in this container"))


GOLDEN = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="session")
def golden_tiny():
    from oracle.make_golden import load_nvae_tiny
    return load_nvae_tiny(os.path.join(GOLDEN, "nvae_tiny.pt"))


@pytest.fixture(scope="session")
def golden_c32():
    import torch
    return torch.load(os.path.join(GOLDEN, "nvae_c32_vgg11.pt"), weights_only=True)
