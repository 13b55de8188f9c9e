import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with `pytest -m gpu` on the GPU box)")


@pytest.fixture(scope="session")
def coracle():
    from oracle.oracle import COracle, build
    build(ref=False)
    return COracle()


@pytest.fixture
def refkernels(request):
    """The original SIMD kernel, one per instruction-set build ({isa: RefKernel}), replayed from tests/golden (reference_calls.py)."""
    from reference_calls import reference
    return reference(request, "kernels")


@pytest.fixture
def refhmm(request):
    """The original hmm::evaluate / hmm::align / PairHMMWrapper / HaplotypeLikelihoodArray (RefHMM), replayed from tests/golden."""
    from reference_calls import reference
    return reference(request, "hmm")


@pytest.fixture(scope="session")
def kats():
    import json
    with open(os.path.join(ROOT, "tests", "golden", "pair_hmm_kats.json")) as f:
        return json.load(f)["cases"]


@pytest.fixture(scope="session")
def engine():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    from octopus_b200 import PairHMMEngine
    return PairHMMEngine(0)
