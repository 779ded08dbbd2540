"""Stored results of the reference (cvxopt built into oracle/_ref by oracle/build_ref.sh).

The tests that compare with the reference read what it computed from tests/golden/reference/<test module>.npz, so
they run where the reference is not built.  The inputs are regenerated from their seeds by each test; only the
reference's outputs are stored, keyed by test (with its parameters) and a label.

To regenerate, build the reference and run the tests with CVXB_RECORD_REFERENCE=<directory>: every reference
result is then recomputed and written to <directory>/<test module>.npz (merged with what is already there), to be
copied into tests/golden/reference/."""
import atexit
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden", "reference")
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
RECORD_DIR = os.environ.get("CVXB_RECORD_REFERENCE") or None

_loaded = {}
_recorded = {}


def _load(module):
    if module not in _loaded:
        path = os.path.join(GOLDEN_DIR, module + ".npz")
        _loaded[module] = dict(np.load(path, allow_pickle=False)) if os.path.exists(path) else {}
    return _loaded[module]


def _import_reference():
    if not os.path.isdir(os.path.join(REF_DIR, "cvxopt")):
        pytest.fail("CVXB_RECORD_REFERENCE is set but oracle/_ref is not built (oracle/build_ref.sh)")
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    from cvxopt import solvers
    solvers.options["show_progress"] = False


def _to_array(v):
    if isinstance(v, str):
        return np.array(v)
    a = np.array(v, copy=True)
    if a.dtype.kind in "iub":
        return a.astype(np.int64)
    return a.astype(np.float64)


def _from_array(a):
    return a.item() if a.ndim == 0 else a.copy()       # the tests update some of these in place


def _write():
    os.makedirs(RECORD_DIR, exist_ok=True)
    for module, values in _recorded.items():
        path = os.path.join(RECORD_DIR, module + ".npz")
        merged = dict(np.load(path, allow_pickle=False)) if os.path.exists(path) else {}
        merged.update(values)
        np.savez(path, **merged)


def result(node, label, compute):
    """The reference's result named `label` in test `node`: a dict of arrays, numbers and strings.

    `compute()` runs the reference and returns that dict (cvxopt matrices are converted to numpy); it is called only
    when recording."""
    module = node.module.__name__.rsplit(".", 1)[-1]
    prefix = "%s|%s|" % (node.name, label)
    if RECORD_DIR:
        _import_reference()
        values = {k: _to_array(v) for k, v in compute().items()}
        if not _recorded:
            atexit.register(_write)
        _recorded.setdefault(module, {}).update({prefix + k: v for k, v in values.items()})
        return {k: _from_array(v) for k, v in values.items()}
    stored = _load(module)
    values = {k[len(prefix):]: _from_array(v) for k, v in stored.items() if k.startswith(prefix)}
    if not values:
        pytest.fail("no stored reference result %r for %s in tests/golden/reference/%s.npz (see "
                    "tests/reference_results.py to regenerate)" % (label, node.name, module))
    return values


def W_arrays(W, prefix="W."):
    """a scaling dictionary (cvxopt matrices or numpy) as flat named arrays (copies)"""
    def vec(a):
        return np.array(a, dtype=np.float64).reshape(-1)
    out = {prefix + "d": vec(W["d"]), prefix + "di": vec(W["di"]), prefix + "beta": vec([float(b) for b in W["beta"]])}
    for k, a in enumerate(W["v"]):
        out["%sv%d" % (prefix, k)] = vec(a)
    for key in ("r", "rti"):
        for k, a in enumerate(W[key]):
            out["%s%s%d" % (prefix, key, k)] = np.array(a, dtype=np.float64)
    if "dnl" in W:
        out[prefix + "dnl"], out[prefix + "dnli"] = vec(W["dnl"]), vec(W["dnli"])
    return out


def W_from_arrays(values, dims, prefix="W."):
    """inverse of W_arrays: numpy arrays, 'r' / 'rti' blocks in column-major storage"""
    W = {"d": np.asarray(values[prefix + "d"], dtype=np.float64).reshape(-1),
         "di": np.asarray(values[prefix + "di"], dtype=np.float64).reshape(-1),
         "beta": [float(b) for b in np.asarray(values[prefix + "beta"]).reshape(-1)],
         "v": [np.asarray(values["%sv%d" % (prefix, k)]).reshape(-1) for k in range(len(dims["q"]))],
         "r": [np.asfortranarray(values["%sr%d" % (prefix, k)]) for k in range(len(dims["s"]))],
         "rti": [np.asfortranarray(values["%srti%d" % (prefix, k)]) for k in range(len(dims["s"]))]}
    if prefix + "dnl" in values:
        W["dnl"] = np.asarray(values[prefix + "dnl"]).reshape(-1)
        W["dnli"] = np.asarray(values[prefix + "dnli"]).reshape(-1)
    return W
