import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "3d-gaussian-splatting_b200")
ORACLE = os.path.join(ROOT, "oracle")
for p in (PKG, ORACLE, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")


@pytest.fixture(scope="session")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


def _ensure_built():
    """The in-tree .so files normally travel with the snapshot; on a bare checkout build them
    (nvcc, ~2 min).  A failing build is an error, never a skip or a fallback."""
    import glob
    if glob.glob(os.path.join(PKG, "gaussian*.so")) and os.path.exists(os.path.join(PKG, "libgs_b200.so")):
        return
    import importlib.util
    spec = importlib.util.spec_from_file_location("gs_b200_build", os.path.join(PKG, "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.build_all()


@pytest.fixture(scope="session")
def gs(cuda):
    """Our extension + autograd boundary.  Fails (does not skip) when it cannot be built / loaded."""
    _ensure_built()
    import gaussian   # noqa: F401  built in-tree by 3d-gaussian-splatting_b200/build.py
    import renderer
    return gaussian, renderer
