import importlib.util
import os
import sys

import pytest

# Unless a test selects a backend itself (the tensor-core tests do), the suite runs the exact-fp32 CUDA-core convolutions:
# they are the device-side reference the 2e-5 op / module tolerances are written for.  The library default is "tc".
os.environ.setdefault("DVMVS_CONV_BACKEND", "fp32")

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG_DIR = os.path.join(REPO, "deep-video-mvs_b200")
for p in (REPO, PKG_DIR):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture(scope="session")
def synth():
    import synth_data
    return synth_data


@pytest.fixture(scope="session")
def cases():
    return _load("golden_cases", os.path.join(REPO, "tests", "golden", "cases.py"))


@pytest.fixture(scope="session")
def golden_ops():
    from oracle import npz_parts
    return npz_parts.load(os.path.join(REPO, "tests", "golden", "ops.npz"))


@pytest.fixture(scope="session")
def golden_modules():
    import numpy as np
    return np.load(os.path.join(REPO, "tests", "golden", "modules.npz"))


@pytest.fixture(scope="session")
def oracle():
    from oracle import dvmvs_oracle
    return dvmvs_oracle
