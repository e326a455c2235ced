import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line(
        "markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)"
    )
    config.addinivalue_line(
        "markers", "multigpu: needs >= 2 GPUs; skipped otherwise"
    )


def pytest_collection_modifyitems(config, items):
    have_gpu = None
    for item in items:
        if "gpu" in item.keywords:
            if have_gpu is None:
                have_gpu = _gpu_ready()
            if have_gpu is not True:
                item.add_marker(pytest.mark.skip(reason=have_gpu))


def _gpu_ready():
    """True, or the reason the ``gpu`` tests cannot run here: a plain ``pytest`` on a machine
    without CUDA skips them instead of failing 200+ times.  With a GPU present they always
    run -- a missing ``libctgb200.so`` must fail loudly there, never skip."""
    try:
        import torch

        if not torch.cuda.is_available():
            return "no CUDA device"
    except Exception as exc:  # pragma: no cover
        return f"torch unavailable: {exc}"
    return True
