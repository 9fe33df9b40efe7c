import ctypes
import os
import sys
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("BARK_B200_QUIET", "1")

import __graft_entry__ as graft  # noqa: E402

# generated weight files, cached between sessions; per user, since another user's directory of the same name is not writable
FIXTURE_DIR = os.environ.get("BARK_B200_FIXTURES") or os.path.join(tempfile.gettempdir(), f"bark_b200_fixtures_{os.getuid()}")
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200")


def cuda_device_count() -> int:
    try:
        rt = ctypes.CDLL("libcudart.so.12")
    except OSError:
        try:
            rt = ctypes.CDLL("/usr/local/cuda/lib64/libcudart.so")
        except OSError:
            return 0
    n = ctypes.c_int(0)
    return n.value if rt.cudaGetDeviceCount(ctypes.byref(n)) == 0 else 0


def pytest_collection_modifyitems(config, items):
    if cuda_device_count() > 0:
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def pkg():
    if not os.path.exists(os.path.join(ROOT, "bark.cpp_b200", "libbark_b200.so")):
        graft.build()
    return graft.load_package()


@pytest.fixture(scope="session")
def weights_mod(pkg):
    import importlib
    return importlib.import_module("bark_cpp_b200.weights")


@pytest.fixture(scope="session")
def orc():
    m = graft.load_oracle_bindings()
    m.build_oracle()
    return m


@pytest.fixture(scope="session")
def weights_file(weights_mod):
    os.makedirs(FIXTURE_DIR, exist_ok=True)

    def get(config: str, ftype: str = "f16", seed: int = 1234) -> str:
        path = os.path.join(FIXTURE_DIR, f"{config}_{ftype}_{seed}.bin")
        if not os.path.exists(path):
            cfg = weights_mod.CONFIGS[config](weights_mod.F16 if ftype == "f16" else weights_mod.F32)
            weights_mod.write_weights(path + ".tmp", cfg, seed)
            os.replace(path + ".tmp", path)
        return path
    return get


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)
