import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `pytest -m gpu`)")


def norm_model(M):
    """Scale/sign normalisation used for every model comparison (F and H are defined up to scale, LAPACK/Jacobi
    eigenvector signs are arbitrary): unit Frobenius norm, largest-magnitude entry positive."""
    import numpy as np
    M = np.asarray(M, dtype=np.float64)
    n = np.linalg.norm(M)
    if n == 0:
        return M
    M = M / n
    return M * np.sign(M.flat[np.argmax(np.abs(M))])


@pytest.fixture(scope="session")
def ref_oracle():
    """The original project's answers (tests/reference_calls.py): replayed from golden data, or answered by the compiled
    reference and recorded to the file DGB200_RECORD_REFERENCE names."""
    from tests.reference_calls import ReferenceCalls
    record_to = os.environ.get("DGB200_RECORD_REFERENCE")
    oracle = ReferenceCalls(record_to)
    yield oracle
    if record_to:
        oracle.save()
