import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box: pytest -m gpu)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden_dir():
    return os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="session")
def moe_small(golden_dir):
    """The reference's MOE::forward fixture (tests/golden/make_golden.py), stored in parts of under 1 MB each."""
    import numpy as np
    out = {}
    for part in ("gate", "up", "down", "io"):
        with np.load(os.path.join(golden_dir, f"moe_small_{part}.npz")) as g:
            out.update({k: g[k] for k in g.files})
    return out


@pytest.fixture(scope="session")
def oracle():
    from oracle.bindings import Oracle
    return Oracle()


@pytest.fixture(scope="session")
def ref():
    from oracle.bindings import Ref
    if not Ref.available():
        pytest.skip("oracle/_ref not built (needs /root/reference)")
    return Ref.get(min(os.cpu_count() or 1, 16))
