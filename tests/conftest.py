import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def sq():
    import sqeazy_b200

    if not os.path.exists(sqeazy_b200.LIB_PATH):
        import __graft_entry__

        __graft_entry__.build()
    sqeazy_b200.lib()
    return sqeazy_b200


@pytest.fixture(scope="session")
def port():
    from oracle import oracle

    return oracle.port()


@pytest.fixture(scope="session")
def ref():
    """the reference's own stage code, oracle/_ref: built only from the reference's sources, which are not part of this
    repository; the tests that pin the oracle port itself need it and skip without it"""
    from oracle import oracle

    r = oracle.ref()
    if not r.available:
        pytest.skip("oracle/_ref (the reference's compiled stage code, built from sources outside this repository) not built")
    return r


@pytest.fixture(scope="session")
def ref_or_standin():
    """oracle/_ref where it is built, else oracle.Standin (liblz4 for LZ4, the golden-pinned C port for the filters);
    which of the two a run used is printed in the report header"""
    from oracle import oracle

    r = oracle.ref()
    if r.available:
        return r
    s = oracle.standin()
    if not s.available:
        pytest.skip("neither oracle/_ref nor liblz4 for oracle.Standin")
    return s


def pytest_report_header(config):
    from oracle import oracle

    if os.path.exists(oracle._REF_SO):
        return "reference comparisons: oracle/_ref (the reference's own code)"
    return "reference comparisons: oracle.Standin (oracle/_ref not built; tests that need the reference itself skip)"


@pytest.fixture(scope="session")
def golden():
    path = os.path.join(ROOT, "tests", "golden", "golden_v1.npz")
    return np.load(path)


@pytest.fixture(scope="session")
def cuda(sq):
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    sq.set_device(0)
    return torch
