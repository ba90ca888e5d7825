import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_addoption(parser):
    parser.addoption("--record-reference", action="store_true",
                     help="compute the reference answers under tests/golden/ with the reference's own code (oracle/_ref) and rewrite them")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def oracle():
    from oracle.pyoracle import Oracle
    return Oracle()


@pytest.fixture(scope="session")
def reflib():
    from oracle.pyoracle import RefLib
    if not RefLib.available():
        pytest.skip("oracle/_ref/libmash_ref.so not built (reference sources absent)")
    return RefLib()


@pytest.fixture(scope="module")
def ref(request):
    """The reference's answers for this module's inputs (fixtures.ReferenceAnswers), recorded under tests/golden/ with
    --record-reference."""
    import fixtures
    name = request.module.REFERENCE_ANSWERS
    reference = request.module.reference() if request.config.getoption("--record-reference") else None
    answers = fixtures.ReferenceAnswers(name, reference)
    yield answers
    answers.save()


@pytest.fixture(scope="session")
def golden():
    import fixtures
    return fixtures.Golden()


@pytest.fixture(scope="session")
def gpu():
    """The product: the C-ABI library through its ctypes host mirror. Fails loudly without CUDA."""
    import mash_b200
    return mash_b200.Engine(device=0)
