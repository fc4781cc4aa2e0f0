import os
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ.setdefault("MASTER_ADDR", "127.0.0.1")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: test needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "dist: spawns multiple processes (gloo on CPU, NCCL on GPU)")


@pytest.fixture(autouse=True)
def _cpu_tier_sees_no_gpu(request, monkeypatch):
    """A test without the `gpu` marker belongs to the CPU tier (gloo, models and data on the CPU) and runs the same on a
    GPU machine: the processes it starts get CUDA_VISIBLE_DEVICES="", and in this process the CUDA probe and the
    accelerator answer "cpu".  The real probe runs first, so this process keeps its GPUs for the `gpu` tests."""
    import torch

    if request.node.get_closest_marker("gpu") is not None or not torch.cuda.is_available():
        return
    from colossalai_b200 import accelerator

    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    monkeypatch.setattr(accelerator, "_ACCELERATOR", accelerator.CpuAccelerator())


@pytest.fixture(autouse=True)
def _clear_cuda_cache():
    yield
    try:
        import torch

        if torch.cuda.is_available():
            torch.cuda.empty_cache()
    except Exception:
        pass
