import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_addoption(parser):
    parser.addoption("--trrt-so", default=None, help="run against another build of libthetarrt.so (e.g. the checked build, "
                                                    "profiles/tools/checked_build.sh)")


def pytest_configure(config):
    so = config.getoption("--trrt-so")
    if so:
        from theta_rrt_b200 import _lib
        _lib.SO_PATH = os.path.abspath(so)
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "reference: needs the unmodified eshira/theta-rrt sources (directory in THETA_RRT_REFERENCE)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    from oracle import live_reference
    have_ref = live_reference.available()
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))
        if "reference" in item.keywords and not have_ref:
            item.add_marker(pytest.mark.skip(reason="eshira/theta-rrt sources not found (set THETA_RRT_REFERENCE)"))


@pytest.fixture(scope="session")
def maps():
    """map1 / map2 / blank as bool arrays, from the committed fixture (tests/golden/maps.npz)."""
    import numpy as np
    z = np.load(os.path.join(GOLDEN, "maps.npz"))
    return {k: z[k].astype(bool) for k in z.files}
