import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu under gpurun)")


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


def load_golden(name):
    import numpy as np
    import torch
    from oracle import gen_golden
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    out = gen_golden.seeded_inputs(name) if name in gen_golden.OUTPUTS_ONLY else {}
    for k in z.files:
        a = z[k]
        out[k] = torch.from_numpy(a) if a.dtype.kind in "fi" and a.ndim > 0 else a
    return out
