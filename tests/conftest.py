import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")
    config.addinivalue_line("markers", "needs_reference: needs the reference checkout (COOPSEARCH_REFERENCE, else BASELINE.json reference_path)")


def pytest_collection_modifyitems(config, items):
    from oracle import refharness
    have_ref = refharness.reference_available()
    try:
        import torch
        have_gpu = torch.cuda.is_available()
    except Exception:  # pragma: no cover
        have_gpu = False
    for item in items:
        if "needs_reference" in item.keywords and not have_ref:
            item.add_marker(pytest.mark.skip(reason="no reference checkout (COOPSEARCH_REFERENCE, BASELINE.json reference_path) and no staged oracle/_ref"))
        if "gpu" in item.keywords and not have_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))


@pytest.fixture
def oracle_squares_by_multiplication():
    """The C oracle squares coordinate differences with libm pow(v, 2.0) like the reference's Python `**`; the CUDA kernels
    multiply.  pow(v, 2.0) != v * v in the last bit for ~0.08 % of arguments, which only shows in the repulsion force of
    agents closer than force_dist.  Tests that demand bit-identical float64 positions from the GPU over long runs switch
    the oracle to multiplication; everything else runs against the reference's own arithmetic."""
    from oracle import c_oracle
    c_oracle.set_square("mul")
    yield
    c_oracle.set_square("pow")
