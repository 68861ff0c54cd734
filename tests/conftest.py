import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
GOLDEN_CASES = ["tiny", "small_diag", "k10d128"]


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session", params=GOLDEN_CASES)
def golden(request):
    """A golden case: the reference's outputs, and the seeded feature maps `it<i>_x_add` it ran on.  The feature
    gradients `it<i>_grad_x` and normalised features `it0_push_feat` are stored at the patches `sample` selects."""
    import numpy as np
    import headline_case as HC
    z = np.load(os.path.join(GOLDEN_DIR, request.param + ".npz"))
    d = {k: z[k] for k in z.files}
    d["name"] = request.param
    B, D, H, W, seed, s = (int(d[k]) for k in "B D H W seed hw_stride".split())
    for it in range(int(d["iters"])):
        d["it%d_x_add" % it] = HC.fixture_features(B, D, H, W, seed, it)
    d["sample"] = np.s_[:, :, ::s, ::s]
    return d
