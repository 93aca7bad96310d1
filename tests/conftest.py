import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "reference: needs the original Fair-MARL project (FAIRMARL_REFERENCE_ROOT)")


def pytest_generate_tests(metafunc):
    """Every GPU test runs under both kernel mappings: 'auto' (agent-warp where compiled, i.e. the
    product default) and 'group' (group-per-env kernels forced)."""
    if metafunc.module.__name__.endswith(("test_gpu_formation", "test_gpu_policy")):
        return                                  # kernels with a single mapping
    if metafunc.definition.get_closest_marker("gpu") and "kernel_mapping" in metafunc.fixturenames:
        metafunc.parametrize("kernel_mapping", ["auto", "group"], indirect=True)


@pytest.fixture(autouse=True)
def kernel_mapping(request):
    import parity_util
    parity_util.MAPPING = getattr(request, "param", "auto")
    yield parity_util.MAPPING
    parity_util.MAPPING = "auto"


def _gpu_ready() -> bool:
    try:
        import torch
        from fair_marl_b200.build import library_path
        return torch.cuda.is_available() and os.path.isfile(library_path())
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    from oracle.reference_shim import SKIP_REASON, reference_available
    have_ref, have_gpu = reference_available(), _gpu_ready()
    skip_ref = pytest.mark.skip(reason=SKIP_REASON)
    skip_gpu = pytest.mark.skip(reason="no CUDA device (or libfairmarl.so not built): GPU parity tests run on the B200 box")
    for item in items:
        if not have_ref and "reference" in item.keywords:
            item.add_marker(skip_ref)
        if not have_gpu and "gpu" in item.keywords:
            item.add_marker(skip_gpu)
