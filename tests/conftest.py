import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `pytest -m gpu`)")
    config.addinivalue_line("markers", "multigpu: needs >= 2 CUDA devices")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        n = torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        n = 0
    skip_gpu = pytest.mark.skip(reason="no CUDA device")
    skip_multi = pytest.mark.skip(reason="needs >= 2 CUDA devices")
    for item in items:
        if "gpu" in item.keywords and n == 0:
            item.add_marker(skip_gpu)
        if "multigpu" in item.keywords and n < 2:
            item.add_marker(skip_multi)


def _drop_process_group():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        dist.destroy_process_group()


@pytest.fixture(autouse=True)
def _cpu_unless_marked_gpu(request, monkeypatch):
    """Tests not marked `gpu` check the CPU / gloo paths.  The trainer, main.py and the launcher take CUDA whenever it is
    available, so on a machine with a GPU these tests see none (the ranks they start set CUDA_VISIBLE_DEVICES="" themselves:
    setting it here would leave torch's device count cached at 0 for the `gpu` tests).  The launcher also reuses an initialised
    default process group, so these tests start and end without one: a `gpu` test's NCCL group is no group for CPU tensors,
    and theirs is none for CUDA tensors."""
    if "gpu" in request.keywords:
        yield
        return
    import torch
    _drop_process_group()
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    yield
    _drop_process_group()


@pytest.fixture
def workdir(tmp_path, monkeypatch):
    """Run inside a scratch cwd: the trainer writes tensorboard/, checkpoints/, results.csv there."""
    monkeypatch.chdir(tmp_path)
    return tmp_path
