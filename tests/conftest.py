import os
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _have_gpu() -> bool:
    if os.environ.get("ACB_FORCE_NO_GPU"):
        return False
    try:
        import ctypes
        cudart = None
        for name in ("libcudart.so", "libcudart.so.12", "/usr/local/cuda/lib64/libcudart.so"):
            try:
                cudart = ctypes.CDLL(name)
                break
            except OSError:
                continue
        if cudart is None:
            import torch
            return torch.cuda.is_available()
        n = ctypes.c_int(0)
        return cudart.cudaGetDeviceCount(ctypes.byref(n)) == 0 and n.value > 0
    except Exception:
        return False


HAVE_GPU = _have_gpu()


def pytest_collection_modifyitems(config, items):
    if HAVE_GPU:
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container (GPU tests run under gpurun)")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def oracle():
    import refs
    refs.ensure_built()
    return refs.OracleLib()


@pytest.fixture()
def reflib(request):
    """The unmodified reference compiled in place, as recorded for this test (refs.Recorded; process-global state
    when live: one user at a time)."""
    import refs
    with refs.recorded(request, lambda: refs.RefLib("O2")) as r:
        yield r


@pytest.fixture(scope="session")
def native():
    """libacars_b200.so, built in-tree; the tests fail (not skip) when it cannot be built/loaded."""
    from acarsdec_b200 import build, api
    build.build()
    return api.load()
