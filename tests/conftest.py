import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from tests.golden import store  # noqa: E402

GOLDEN_CASES = ["glow_d43", "glow_d6_additive_relu", "realnvp_d6_bn", "realnvp_d5_mixed", "glow_d43_h256", "realnvp_d6_h128_bn",
                "toy_d2", "glow_d43_h512", "glow_d43_h128_depth2"]
# ResidualNet s / t networks: served by the exact fp32 kernel only (the f16 tensor-core modes reject them)
FP32_ONLY_CASES = ["realnvp_d6_residual", "realnvp_d5_residual2_bn", "glow_d6_invconv", "glow_d43_invconv_plain"]
ALL_CASES = GOLDEN_CASES + FP32_ONLY_CASES


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if not has_gpu:
        skip = pytest.mark.skip(reason="no CUDA device")
        for it in items:
            if "gpu" in it.keywords:
                it.add_marker(skip)


@pytest.fixture(scope="session")
def golden():
    cache = {}

    def load(name):
        if name not in cache:
            cache[name] = store.load(name)
        return cache[name]
    return load
