"""Nesterov-Todd scaling (SURVEY.md §8 rows a1, a2, f2): misc.compute_scaling / misc.update_scaling.

CPU part: the oracle's restatements against the reference itself (its stored results, tests/reference_results.py) —
'l', 'q' and 's' cones, mnl > 0.
GPU part: cvxopt_b200.scaling (device kernels: elementwise 'l', one CTA per 'q' cone, Cholesky + one-sided Jacobi
SVD for 's') against the reference: d, di, v, beta, lambda elementwise; for 's' blocks the quantities that do not
depend on the sign/order conventions of the SVD (r r', rti rti', rti' r = I, r' z r = diag(lambda)); and whole
solver runs with both functions swapped into cvxopt.misc."""
import numpy as np
import pytest

import kkt_oracle as ko
from problems import cone_dim, cone_lp, cone_point
from reference_results import W_arrays, W_from_arrays

CASES = [
    ({"l": 7, "q": [], "s": []}, 0),
    ({"l": 3, "q": [5, 2, 9], "s": []}, 0),
    ({"l": 0, "q": [], "s": [4, 1, 9]}, 0),
    ({"l": 6, "q": [4, 7], "s": [5, 3]}, 3),
    ({"l": 2, "q": [3], "s": [70]}, 0),             # 's' block above the in-CTA SVD size
]


def _points(dims, mnl, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    s = np.concatenate([rng.uniform(0.5, 2.0, mnl), cone_point(dims, rng)])
    z = np.concatenate([rng.uniform(0.5, 2.0, mnl), cone_point(dims, rng)])
    return s, z, rng


def _scaled_iterates(dims, mnl, rng):
    """new iterates in the current scaling: interior points for the mnl/'l'/'q' rows, Cholesky factors (zero
    above the diagonal) in the 's' blocks — what coneprog hands to update_scaling (coneprog.py:1366-1395)"""
    def one():
        x = np.concatenate([rng.uniform(0.5, 2.0, mnl), cone_point(dims, rng)])
        off = mnl + dims["l"] + sum(dims["q"])
        for k in dims["s"]:
            X = x[off:off + k * k].reshape(k, k, order="F")
            x[off:off + k * k] = np.linalg.cholesky(X).reshape(-1, order="F")
            off += k * k
        return x
    return one(), one()


def _nlam(dims, mnl):
    return mnl + dims["l"] + sum(dims["q"]) + sum(dims["s"])


def _ref_W_to_np(W):
    out = {"d": np.array(W["d"]).ravel(), "di": np.array(W["di"]).ravel(), "v": [np.array(v).ravel() for v in W["v"]],
           "beta": [float(b) for b in W["beta"]], "r": [np.array(r) for r in W["r"]],
           "rti": [np.array(r) for r in W["rti"]]}
    if "dnl" in W:
        out["dnl"], out["dnli"] = np.array(W["dnl"]).ravel(), np.array(W["dnli"]).ravel()
    return out


def _compare_W(got, want, lam_got, lam_want, dims, mnl, tol=1e-11):
    """everything that is unique; 's' blocks through sign/order-free products"""
    for key in ("d", "di") + (("dnl", "dnli") if mnl else ()):
        np.testing.assert_allclose(np.asarray(got[key]).ravel(), np.asarray(want[key]).ravel(), rtol=tol)
    for k in range(len(dims["q"])):
        np.testing.assert_allclose(np.asarray(got["v"][k]).ravel(), np.asarray(want["v"][k]).ravel(), rtol=tol,
                                   atol=tol)
        np.testing.assert_allclose(float(got["beta"][k]), float(want["beta"][k]), rtol=tol)
    np.testing.assert_allclose(lam_got, lam_want, rtol=tol, atol=tol)
    for k in range(len(dims["s"])):
        rg, rw = np.asarray(got["r"][k]), np.asarray(want["r"][k])
        tg, tw = np.asarray(got["rti"][k]), np.asarray(want["rti"][k])
        scale = np.abs(rw @ rw.T).max()
        np.testing.assert_allclose(rg @ rg.T, rw @ rw.T, rtol=0, atol=1e-10 * scale)
        scale = np.abs(tw @ tw.T).max()
        np.testing.assert_allclose(tg @ tg.T, tw @ tw.T, rtol=0, atol=1e-10 * scale)
        np.testing.assert_allclose(tg.T @ rg, np.eye(rg.shape[0]), rtol=0, atol=1e-10)


@pytest.mark.parametrize("dims,mnl", CASES)
def test_oracle_scaling_matches_reference(ref_golden, dims, mnl):
    s, z, rng = _points(dims, mnl, seed=3)
    sn, zn = _scaled_iterates(dims, mnl, rng)

    def reference():
        from cvxopt import matrix, misc
        lam_r = matrix(0.0, (_nlam(dims, mnl), 1))
        Wr = misc.compute_scaling(matrix(s), matrix(z), lam_r, dims, mnl if mnl else None)
        out = dict(W_arrays(Wr, "W."), lam=+lam_r)
        sr, zr = matrix(sn), matrix(zn)
        misc.update_scaling(Wr, lam_r, sr, zr)
        out.update(W_arrays(Wr, "Wu."), lamu=lam_r, s=sr, z=zr)
        return out
    want = ref_golden("scaling", reference)
    lam_o = np.zeros(_nlam(dims, mnl))
    Wo = ko.compute_scaling(s.copy(), z.copy(), lam_o, dims, mnl if mnl else None)
    _compare_W(Wo, W_from_arrays(want, dims, "W."), lam_o, want["lam"].ravel(), dims, mnl)
    # update: both start from the SAME W (the scaled iterates are coordinates with respect to W, and the SVD's
    # sign conventions make W itself non-unique for 's' blocks)
    so, zo = sn.copy(), zn.copy()
    Wo = W_from_arrays(want, dims, "W.")
    lam_o = want["lam"].ravel().copy()
    ko.update_scaling(Wo, lam_o, so, zo)
    _compare_W(Wo, W_from_arrays(want, dims, "Wu."), lam_o, want["lamu"].ravel(), dims, mnl)
    nlq = mnl + dims["l"] + sum(dims["q"])
    np.testing.assert_allclose(so[:nlq], want["s"].ravel()[:nlq], rtol=1e-12)
    np.testing.assert_allclose(zo[:nlq], want["z"].ravel()[:nlq], rtol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("dims,mnl", CASES + [({"l": 0, "q": [64] * 64, "s": []}, 0), ({"l": 0, "q": [], "s": [200]}, 0)])
def test_device_scaling_matches_reference(ref, dims, mnl):
    import cvxopt_b200
    from cvxopt import matrix, misc
    s, z, rng = _points(dims, mnl, seed=5)
    n = _nlam(dims, mnl)
    lam_r = matrix(0.0, (n, 1))
    Wr = misc.compute_scaling(matrix(s), matrix(z), lam_r, dims, mnl if mnl else None)
    lam_g = matrix(0.0, (n, 1))
    before = cvxopt_b200.launch_count()
    Wg = cvxopt_b200.scaling.compute_scaling(matrix(s), matrix(z), lam_g, dims, mnl if mnl else None,
                                             new_matrix=lambda r, c: matrix(0.0, (r, c)))
    assert cvxopt_b200.launch_count() > before
    assert ("dnl" in Wg) == ("dnl" in Wr)
    _compare_W(_ref_W_to_np(Wg), _ref_W_to_np(Wr), np.array(lam_g).ravel(), np.array(lam_r).ravel(), dims, mnl)
    # defining property of the 's' scaling: r' z r = diag(lambda)
    off, lo = mnl + dims["l"] + sum(dims["q"]), mnl + dims["l"] + sum(dims["q"])
    for k, m in enumerate(dims["s"]):
        Z = z[off:off + m * m].reshape(m, m, order="F")
        Z = np.tril(Z) + np.tril(Z, -1).T
        r = np.array(Wg["r"][k])
        lam = np.array(lam_g).ravel()[lo:lo + m]
        np.testing.assert_allclose(r.T @ Z @ r, np.diag(lam), rtol=0, atol=1e-10 * lam.max())
        off += m * m
        lo += m
    # update: both start from the SAME W (the reference's): the scaled iterates are coordinates with respect to W
    sn, zn = _scaled_iterates(dims, mnl, rng)
    sr, zr, sg, zg = matrix(sn), matrix(zn), matrix(sn), matrix(zn)
    Wg = {"d": +Wr["d"], "di": +Wr["di"], "v": [+v for v in Wr["v"]], "beta": list(Wr["beta"]),
          "r": [+r for r in Wr["r"]], "rti": [+r for r in Wr["rti"]]}
    if "dnl" in Wr:
        Wg["dnl"], Wg["dnli"] = +Wr["dnl"], +Wr["dnli"]
    lam_g = +lam_r
    misc.update_scaling(Wr, lam_r, sr, zr)
    cvxopt_b200.scaling.update_scaling(Wg, lam_g, sg, zg)
    _compare_W(_ref_W_to_np(Wg), _ref_W_to_np(Wr), np.array(lam_g).ravel(), np.array(lam_r).ravel(), dims, mnl,
               tol=1e-10)
    nlq = mnl + dims["l"] + sum(dims["q"])
    np.testing.assert_allclose(np.array(sg).ravel()[:nlq], np.array(sr).ravel()[:nlq], rtol=1e-12)
    np.testing.assert_allclose(np.array(zg).ravel()[:nlq], np.array(zr).ravel()[:nlq], rtol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("dims,n,seed", [
    ({"l": 0, "q": [16] * 6, "s": []}, 40, 11),
    ({"l": 10, "q": [7, 3], "s": [6, 9]}, 25, 12),
    ({"l": 0, "q": [], "s": [24]}, 30, 13),
])
def test_solvers_with_device_scaling_swapped_in(ref, dims, n, seed):
    """unmodified solvers.conelp with misc.compute_scaling / misc.update_scaling replaced by the device versions
    (and the device kktsolver): same iteration count and objectives as the all-reference run"""
    import cvxopt_b200
    from cvxopt import matrix, misc, solvers
    c, G, h = cone_lp(n, dims, seed)
    cm, Gm, hm = matrix(c), matrix(G), matrix(h)
    want = solvers.conelp(cm, Gm, hm, dims, kktsolver="chol")
    saved = misc.compute_scaling, misc.update_scaling
    misc.compute_scaling = lambda s, z, lmbda, dims, mnl=None: cvxopt_b200.scaling.compute_scaling(
        s, z, lmbda, dims, mnl, new_matrix=lambda r, c: matrix(0.0, (r, c)))
    misc.update_scaling = cvxopt_b200.scaling.update_scaling
    f = cvxopt_b200.kkt_chol(Gm, dims)
    try:
        got = solvers.conelp(cm, Gm, hm, dims, kktsolver=lambda W: f(W))
    finally:
        misc.compute_scaling, misc.update_scaling = saved
        f.close()
    assert want["status"] == got["status"] == "optimal" and want["iterations"] == got["iterations"]
    np.testing.assert_allclose(got["primal objective"], want["primal objective"], rtol=1e-8)
    np.testing.assert_allclose(got["dual objective"], want["dual objective"], rtol=1e-8)
    np.testing.assert_allclose(np.array(got["x"]), np.array(want["x"]), rtol=1e-6, atol=1e-8)
