import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        have_gpu = torch.cuda.is_available()
    except Exception:
        have_gpu = False
    for item in items:
        if "gpu" in item.keywords and not have_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))


@pytest.fixture(scope="session")
def golden():
    """The reference's recorded outputs (tests/golden/make_golden.py): spectrograms and metadata, and the waveforms."""
    out = {}
    for name in ("reference_golden.npz", "reference_golden_waves.npz"):
        with np.load(os.path.join(ROOT, "tests", "golden", name)) as z:
            out.update({k: z[k] for k in z.files})
    return out
