import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


def _ref_available():
    return os.path.isdir(os.path.join(REF_DIR, "cvxopt")) and any(
        f.startswith("base.") for f in os.listdir(os.path.join(REF_DIR, "cvxopt")))


@pytest.fixture(scope="session")
def ref():
    """The unmodified reference (cvxopt) built into oracle/_ref by oracle/build_ref.sh."""
    if not _ref_available():
        pytest.skip("oracle/_ref not built (oracle/build_ref.sh builds it from the reference's sources)")
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    import cvxopt
    from cvxopt import solvers
    solvers.options["show_progress"] = False
    return cvxopt


@pytest.fixture
def ref_golden(request):
    """ref_golden(label, compute) -> the reference's stored result (tests/reference_results.py)"""
    import reference_results

    def get(label, compute):
        return reference_results.result(request.node, label, compute)
    return get
