import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    import torch
    has_gpu = torch.cuda.is_available()
    skip_gpu = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(skip_gpu)


@pytest.fixture(scope="session")
def layout():
    from mapperatorinator_b200 import TokenLayout
    return TokenLayout.from_json(os.path.join(GOLDEN, "tokenizer_v29.json"))
