import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: needs the unmodified upstream model.py / util.py (SAT_REFERENCE_DIR or oracle/_ref/)")


def pytest_collection_modifyitems(config, items):
    import torch
    from oracle import ref_harness
    has_gpu = torch.cuda.is_available()
    has_ref = ref_harness.available()
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))
        if "reference" in item.keywords and not has_ref:
            item.add_marker(pytest.mark.skip(reason="the unmodified upstream reference is not present"))


def golden_arrays(name):
    """Arrays of the golden case `name`: tests/golden/<name>.npz plus any tests/golden/<name>.<part>.npz (a case too large for
    one file of at most 1 MB is split by array name)."""
    import glob
    import numpy as np
    z = {}
    for path in [os.path.join(GOLDEN, name + ".npz")] + sorted(glob.glob(os.path.join(GOLDEN, glob.escape(name) + ".*.npz"))):
        with np.load(path) as f:
            z.update({k: f[k] for k in f.files})
    return z


def load_golden(name):
    import torch
    z = golden_arrays(name)
    W = {k[2:]: torch.from_numpy(z[k]) for k in z if k.startswith("W/")}
    G = {k[2:]: torch.from_numpy(z[k]) for k in z if k.startswith("G/")}
    return z, W, G


@pytest.fixture(scope="session")
def golden_loader():
    return load_golden
