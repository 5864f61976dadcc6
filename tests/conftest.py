import ctypes
import os
import subprocess
import sys
import warnings

import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)
GOLDEN = os.path.join(REPO, "tests", "golden")

warnings.filterwarnings("ignore", message="torch.meshgrid")
warnings.filterwarnings("ignore", message=".*torch.jit.*is deprecated.*")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden_weights():
    return torch.load(os.path.join(GOLDEN, "weights_000007.pt"), map_location="cpu")


@pytest.fixture(scope="session")
def golden_stage_cases():
    return torch.load(os.path.join(GOLDEN, "stage_cases.pt"), map_location="cpu")


@pytest.fixture(scope="session")
def golden_net_case():
    return torch.load(os.path.join(GOLDEN, "net_case.pt"), map_location="cpu")


@pytest.fixture(scope="session")
def golden_config1():
    return torch.load(os.path.join(GOLDEN, "config1_case.pt"), map_location="cpu")


@pytest.fixture(scope="session")
def reference_net_calls():
    """How the unmodified reference network (models/net.py) constructs and calls its three PatchMatch modules on
    pm_cases.NET_CASE, every call's inputs and outputs, and its PatchMatch.forward schema (tests/golden/make_reference_golden.py)."""
    return torch.load(os.path.join(GOLDEN, "net_calls.pt"), map_location="cpu")


@pytest.fixture(scope="session")
def hostmath():
    """pm_math.cuh compiled for the host (test infrastructure, see tests/hostmath.cpp)."""
    src = os.path.join(REPO, "tests", "hostmath.cpp")
    hdrs = [os.path.join(REPO, "patchmatchnet_b200", "csrc", h) for h in ("pm_math.cuh", "pm_geo_math.cuh")]
    out = os.path.join(REPO, "tests", "_hostmath.so")
    if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(f) for f in [src] + hdrs):
        subprocess.run(
            ["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-o", out, "-x", "c++", src],
            check=True,
        )
    lib = ctypes.CDLL(out)
    for fn in ("hm_random_hypothesis", "hm_perturbed_hypothesis", "hm_depth_similarity", "hm_normalised_inverse_depth"):
        getattr(lib, fn).restype = ctypes.c_float
    lib.hm_random_hypothesis.argtypes = [ctypes.c_float, ctypes.c_int, ctypes.c_float, ctypes.c_float]
    lib.hm_perturbed_hypothesis.argtypes = [ctypes.c_float, ctypes.c_int, ctypes.c_int] + [ctypes.c_float] * 3
    lib.hm_depth_similarity.argtypes = [ctypes.c_float] * 3
    lib.hm_normalised_inverse_depth.argtypes = [ctypes.c_float] * 3
    return lib
