import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

os.environ.setdefault("RELORA_B200_NO_WANDB", "1")
os.environ.setdefault("WANDB_MODE", "disabled")
os.environ.setdefault("TOKENIZERS_PARALLELISM", "false")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")
    config.addinivalue_line("markers", "multigpu: needs >= 2 CUDA devices")
    config.addinivalue_line("markers", "slow: long-running")


def pytest_collection_modifyitems(config, items):
    try:
        import torch

        have_cuda = torch.cuda.is_available()
        n_gpu = torch.cuda.device_count() if have_cuda else 0
    except Exception:
        have_cuda, n_gpu = False, 0
    skip_gpu = pytest.mark.skip(reason="no CUDA device")
    skip_multi = pytest.mark.skip(reason="needs >= 2 CUDA devices")
    for item in items:
        if "gpu" in item.keywords and not have_cuda:
            item.add_marker(skip_gpu)
        if "multigpu" in item.keywords and n_gpu < 2:
            item.add_marker(skip_multi)
