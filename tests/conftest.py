import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
# a checkout of the original attack-vc project (with the VSMask models/ and utils/), for test_oracle_vs_reference.py
# and tests/tools/make_golden.py; it is not part of this repository
REFERENCE = os.environ.get("ATTACK_VC_REFERENCE", "")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on a B200 via gpurun)")


def has_gpu() -> bool:
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if has_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def oracle():
    from oracle import adainvc_oracle
    return adainvc_oracle


@pytest.fixture(scope="session")
def golden():
    import numpy as np

    def load(name):
        return dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    return load


@pytest.fixture(scope="session")
def cpu_model(oracle):
    return oracle.OracleAdaInVC(oracle.SYNTH_CONFIG, seed=0)


@pytest.fixture(scope="session")
def gpu_model(oracle):
    import torch
    return oracle.OracleAdaInVC(oracle.SYNTH_CONFIG, seed=0).to("cuda")


@pytest.fixture(scope="session")
def engine(gpu_model):
    from attack_vc_b200 import Engine
    return Engine(gpu_model)
