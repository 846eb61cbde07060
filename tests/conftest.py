import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def fx():
    from is3d_b200 import tables
    return tables.load_fixture()


NEEDS_PRODUCT_LIB = ("test_abi", "test_class_api", "test_host_layer", "test_yield", "test_gpu_", "test_decays")
_LIB_PROBLEM = None


@pytest.fixture(scope="session", autouse=True)
def _built():
    """Build the checkers (C oracle; the reference binaries, where IS3D_REFERENCE names an iS3D checkout, are built by __graft_entry__.build) and,
    when nvcc is available, the product library.  Without a CUDA toolkit the oracle / sharding tests still run; the tests that load
    libis3d_b200.so are skipped with a message instead of failing (ADVICE r1)."""
    global _LIB_PROBLEM
    import shutil
    import subprocess
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "oracle"])
    from is3d_b200 import api, build
    if not os.path.exists(api.LIB_PATH):
        if shutil.which("nvcc") or os.path.exists("/usr/local/cuda/bin/nvcc"):
            build.build()
        else:
            _LIB_PROBLEM = "libis3d_b200.so is not built and nvcc is not available: run `python -m is3d_b200.build` on a machine with the CUDA toolkit"


def pytest_runtest_setup(item):
    if _LIB_PROBLEM and any(item.fspath.basename.startswith(p) for p in NEEDS_PRODUCT_LIB):
        pytest.skip(_LIB_PROBLEM)
