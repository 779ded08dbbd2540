"""Pins the numpy restatement (oracle/kkt_oracle.py) against the reference itself — CPU only.  The reference's
results are stored under tests/golden/reference (tests/reference_results.py)."""
import numpy as np
import pytest

import kkt_oracle as ko
from problems import cone_dim, cone_point, dense_qp, random_scaling
from reference_results import W_arrays, W_from_arrays

DIMS = [
    {"l": 7, "q": [], "s": []},
    {"l": 0, "q": [4, 9, 1], "s": []},
    {"l": 3, "q": [5], "s": [3, 1, 6]},
    {"l": 0, "q": [], "s": [8]},
]


def to_ref_W(W):
    from cvxopt import matrix as m
    out = {"d": m(W["d"]), "di": m(W["di"]), "v": [m(v) for v in W["v"]],
           "beta": list(W["beta"]), "r": [m(r) for r in W["r"]], "rti": [m(r) for r in W["rti"]]}
    return out


@pytest.mark.parametrize("dims", DIMS)
def test_compute_scaling_matches_reference(ref_golden, dims):
    rng = np.random.Generator(np.random.PCG64(3))
    s, z = cone_point(dims, rng), cone_point(dims, rng)
    nl = dims["l"] + sum(dims["q"]) + sum(dims["s"])
    lm = np.zeros(nl)
    W = ko.compute_scaling(s.copy(), z.copy(), lm, dims)

    def reference():
        from cvxopt import matrix, misc
        lmr = matrix(0.0, (nl, 1))
        Wr = misc.compute_scaling(matrix(s), matrix(z), lmr, dims)
        return dict(W_arrays(Wr), lmbda=lmr)
    want = ref_golden("compute_scaling", reference)
    Wr = W_from_arrays(want, dims)
    np.testing.assert_allclose(lm, want["lmbda"].ravel(), rtol=1e-12, atol=1e-13)
    np.testing.assert_allclose(W["d"], Wr["d"], rtol=1e-14)
    for a, b in zip(W["v"], Wr["v"]):
        np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(W["beta"], Wr["beta"], rtol=1e-13)
    # r is unique only up to the sign of the singular vectors: compare r r' and rti rti'
    for a, b in zip(W["r"], Wr["r"]):
        np.testing.assert_allclose(a @ a.T, b @ b.T, rtol=1e-9, atol=1e-11)


@pytest.mark.parametrize("dims", DIMS)
@pytest.mark.parametrize("trans", ["N", "T"])
@pytest.mark.parametrize("inverse", ["N", "I"])
def test_scale_matches_reference(ref_golden, dims, trans, inverse):
    W, _ = random_scaling(dims, seed=5)
    rng = np.random.Generator(np.random.PCG64(8))
    x = np.asfortranarray(rng.standard_normal((cone_dim(dims), 3)))

    def reference():
        from cvxopt import matrix, misc
        xr = matrix(x)
        misc.scale(xr, to_ref_W(W), trans=trans, inverse=inverse)
        return {"x": xr}
    want = ref_golden("scale", reference)
    ko.scale(x, W, trans, inverse)
    np.testing.assert_allclose(x, want["x"], rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("dims", DIMS)
def test_pack_unpack_match_reference(ref_golden, dims):
    rng = np.random.Generator(np.random.PCG64(9))
    K = cone_dim(dims)
    _, _, _, cdim, cp = ko.cone_sizes(dims)
    x = rng.standard_normal(K)
    z = rng.standard_normal(K)
    X = np.asfortranarray(rng.standard_normal((K, 4)))

    def reference():
        from cvxopt import matrix, misc
        yr = matrix(0.0, (cp, 1))
        misc.pack(matrix(x), yr, dims)
        zr = matrix(z)
        misc.unpack(yr, zr, dims)
        Xr = matrix(X)
        misc.pack2(Xr, dims)
        return {"y": yr, "z": zr, "X": Xr}
    want = ref_golden("pack_unpack", reference)
    y = np.zeros(cp)
    ko.pack(x, y, dims)
    assert np.array_equal(y, want["y"].ravel())
    ko.unpack(y, z, dims)
    assert np.array_equal(z, want["z"].ravel())
    ko.pack2(X, dims)
    assert np.array_equal(X[:cp], want["X"][:cp])


def _solve_reference(factory, W, H, x, y, z):
    """x, y, z after the reference's solve f(x, y, z) with f = factory(W[, H]) (inputs are copied)"""
    from cvxopt import matrix
    f = factory(to_ref_W(W), matrix(H)) if H is not None else factory(to_ref_W(W))
    xr, yr, zr = matrix(x), matrix(y, (len(y), 1)), matrix(z)
    f(xr, yr, zr)
    return {"x": xr, "y": yr, "z": zr}


def _compare_solution(dims, x, y, z, want, tol, atol):
    np.testing.assert_allclose(x, want["x"].ravel(), rtol=tol, atol=atol)
    if y is not None and len(y):
        np.testing.assert_allclose(y, want["y"].ravel(), rtol=tol, atol=atol)
    # strict upper triangles of 's' blocks are not significant; compare packed
    _, _, _, _, cp = ko.cone_sizes(dims)
    a, b = np.zeros(cp), np.zeros(cp)
    ko.pack(z, a, dims)
    ko.pack(want["z"].ravel(), b, dims)
    np.testing.assert_allclose(a, b, rtol=tol, atol=atol)


@pytest.mark.parametrize("dims", DIMS)
def test_kkt_chol_matches_reference(ref_golden, dims):
    n = 6
    rng = np.random.Generator(np.random.PCG64(21))
    K = cone_dim(dims)
    G = np.asfortranarray(rng.standard_normal((K, n)))
    B = rng.standard_normal((n, n))
    H = np.asfortranarray(B @ B.T + np.eye(n))
    W, _ = random_scaling(dims, seed=2)
    f_or = ko.KktChol(G, dims).factor(W, H)
    x, z = rng.standard_normal(n), rng.standard_normal(K)

    def reference():
        from cvxopt import matrix, misc
        return _solve_reference(misc.kkt_chol(matrix(G), dims, matrix(0.0, (0, n))), W, H, x, np.zeros(0), z)
    want = ref_golden("solve", reference)
    f_or(x, None, z)
    _compare_solution(dims, x, None, z, want, 1e-10, 1e-12)


@pytest.mark.parametrize("dims", DIMS)
@pytest.mark.parametrize("with_H", [True, False])
def test_kkt_chol_with_equalities_matches_reference(ref_golden, dims, with_H):
    """p > 0: the oracle's Schur-complement elimination vs the reference's QR-based kkt_chol."""
    n, p = 7, 3
    rng = np.random.Generator(np.random.PCG64(31))
    K = cone_dim(dims)
    G = np.asfortranarray(rng.standard_normal((K, n)))
    A = np.asfortranarray(rng.standard_normal((p, n)))
    B = rng.standard_normal((n, n))
    H = np.asfortranarray(B @ B.T + np.eye(n)) if with_H else None
    W, _ = random_scaling(dims, seed=3)
    if K < n and H is None:
        pytest.skip("singular even with A'A")
    f_or = ko.KktChol(G, dims, A).factor(W, H)
    x, y, z = rng.standard_normal(n), rng.standard_normal(p), rng.standard_normal(K)

    def reference():
        from cvxopt import matrix, misc
        return _solve_reference(misc.kkt_chol(matrix(G), dims, matrix(A)), W, H, x, y, z)
    want = ref_golden("solve", reference)
    f_or(x, y, z)
    _compare_solution(dims, x, y, z, want, 1e-9, 1e-11)


@pytest.mark.parametrize("solver", ["kkt_ldl2", "kkt_chol2"])
@pytest.mark.parametrize("p", [0, 3])
@pytest.mark.parametrize("dims", DIMS)
def test_same_system_as_reference_ldl2_and_chol2(ref_golden, dims, p, solver):
    """kkt_ldl2 (misc.py:1128) and kkt_chol2 (misc.py:1352) solve the system kkt_chol solves: the oracle's
    elimination agrees with both, which is what lets cvxopt_b200.kkt_ldl2 / kkt_chol2 share the device path."""
    if solver == "kkt_chol2" and (dims["q"] or dims["s"]):
        def reference():
            from cvxopt import matrix, misc
            try:
                misc.kkt_chol2(matrix(0.0, (cone_dim(dims), 4)), dims, matrix(0.0, (0, 4)))
            except ValueError:
                return {"raised": "ValueError"}
            return {"raised": ""}
        assert ref_golden("raises", reference)["raised"] == "ValueError"
        return
    n = 8
    rng = np.random.Generator(np.random.PCG64(41))
    K = cone_dim(dims)
    G = np.asfortranarray(rng.standard_normal((K, n)))
    A = np.asfortranarray(rng.standard_normal((p, n)))
    B = rng.standard_normal((n, n))
    H = np.asfortranarray(B @ B.T + np.eye(n))
    W, _ = random_scaling(dims, seed=5)
    f_or = ko.KktChol(G, dims, A if p else None).factor(W, H)
    x, y, z = rng.standard_normal(n), rng.standard_normal(p), rng.standard_normal(K)

    def reference():
        from cvxopt import matrix, misc
        factory = getattr(misc, solver)(matrix(G), dims, matrix(A) if p else matrix(0.0, (0, n)))
        return _solve_reference(factory, W, H, x, y, z)
    want = ref_golden("solve", reference)
    f_or(x, y if p else None, z)
    _compare_solution(dims, x, y if p else None, z, want, 1e-9, 1e-11)


@pytest.mark.parametrize("dims", DIMS)
def test_ipm_side_cone_algebra_matches_reference(ref_golden, dims):
    """scale2 / sprod / sinv / sdot / max_step / trisc / triusc restatements vs misc_solvers."""
    rng = np.random.Generator(np.random.PCG64(41))
    K = cone_dim(dims)
    W, lm = random_scaling(dims, seed=6)
    # every input first, in the order the random stream produces them
    x_scale2 = {inv: cone_point(dims, rng) for inv in "NI"}
    x_sprod, y_sprod = cone_point(dims, rng), cone_point(dims, rng)
    x_diag, x_sinv = cone_point(dims, rng), cone_point(dims, rng)
    x_dot, y_dot = cone_point(dims, rng), cone_point(dims, rng)
    x_step = rng.standard_normal(K)
    for k_off, k in zip(np.cumsum([dims["l"] + sum(dims["q"])] + [s * s for s in dims["s"]])[:-1], dims["s"]):
        X = x_step[k_off:k_off + k * k].reshape(k, k, order="F"); X[:] = (X + X.T) / 2
        x_step[k_off:k_off + k * k] = X.reshape(-1, order="F")
    x_tri = {"trisc": rng.standard_normal(K), "triusc": rng.standard_normal(K)}
    ns = sum(dims["s"])

    def reference():
        from cvxopt import matrix as m, misc
        out = {}
        for inv in "NI":
            xr = m(x_scale2[inv])
            misc.scale2(m(lm), xr, dims, inverse=inv)
            out["scale2_" + inv] = xr
        xr = m(x_sprod)
        misc.sprod(xr, m(y_sprod), dims)
        out["sprod"] = xr
        xr = m(x_diag)
        misc.sprod(xr, m(lm), dims, diag="D")
        out["sprod_D"] = xr
        xr = m(x_sinv)
        misc.sinv(xr, m(lm), dims)
        out["sinv"] = xr
        out["sdot"] = misc.sdot(m(x_dot), m(y_dot), dims)
        out["max_step"] = misc.max_step(m(x_step), dims)
        if ns:
            xr, sigr = m(x_step), m(0.0, (ns, 1))
            out["max_step_sigma"] = misc.max_step(xr, dims, 0, sigr)
            out["sigma"], out["max_step_x"] = sigr, xr
        for name in ("trisc", "triusc"):
            xr = m(x_tri[name])
            getattr(misc, name)(xr, dims)
            out[name] = xr
        return out
    want = ref_golden("cone_algebra", reference)
    for inv in "NI":
        x = x_scale2[inv]
        ko.scale2(lm, x, dims, inverse=inv)
        np.testing.assert_allclose(x, want["scale2_" + inv].ravel(), rtol=1e-12, atol=1e-13)
    ko.sprod(x_sprod, y_sprod, dims)
    mask = np.ones(K, bool)
    off = dims["l"] + sum(dims["q"])
    for k in dims["s"]:
        M = np.ones((k, k), bool); M[np.triu_indices(k, 1)] = False
        mask[off:off + k * k] = M.reshape(-1, order="F"); off += k * k
    np.testing.assert_allclose(x_sprod[mask], want["sprod"].ravel()[mask], rtol=1e-12, atol=1e-12)
    ko.sprod(x_diag, lm, dims, diag="D")
    np.testing.assert_allclose(x_diag[mask], want["sprod_D"].ravel()[mask], rtol=1e-11, atol=1e-12)
    ko.sinv(x_sinv, lm, dims)
    np.testing.assert_allclose(x_sinv[mask], want["sinv"].ravel()[mask], rtol=1e-11, atol=1e-12)
    np.testing.assert_allclose(ko.sdot(x_dot, y_dot, dims), want["sdot"], rtol=1e-13)
    np.testing.assert_allclose(ko.max_step(x_step.copy(), dims), want["max_step"], rtol=1e-10, atol=1e-12)
    if ns:      # with sigma: eigenvalues in sigma, eigenvectors (up to sign) in the 's' blocks of x
        xo, sigo = x_step.copy(), np.zeros(ns)
        np.testing.assert_allclose(ko.max_step(xo, dims, sigma=sigo), want["max_step_sigma"], rtol=1e-10, atol=1e-12)
        np.testing.assert_allclose(sigo, want["sigma"].ravel(), rtol=1e-10, atol=1e-11)
        xr = want["max_step_x"].ravel()
        off = dims["l"] + sum(dims["q"])
        for k in dims["s"]:
            Qo = xo[off:off + k * k].reshape(k, k, order="F"); Qr = xr[off:off + k * k].reshape(k, k, order="F")
            np.testing.assert_allclose(np.abs(np.sum(Qo * Qr, axis=0)), np.ones(k), atol=1e-8)
            off += k * k
    for name in ("trisc", "triusc"):
        x = x_tri[name]
        getattr(ko, name)(x, dims)
        assert np.array_equal(x, want[name].ravel())


def test_reference_known_answer_coneqp(ref_golden):
    """reference tests/test_examples.py:27-29 (examples/doc/chap8/coneqp.py): the only
    reference test whose numbers flow through kkt_chol: the reference's own run gives the published answer."""
    def reference():
        from cvxopt import matrix, solvers
        A = matrix([[.3, -.4, -.2, -.4, 1.3], [.6, 1.2, -1.7, .3, -.3], [-.3, .0, .6, -1.2, -2.0]])
        b = matrix([1.5, .0, -1.2, -.7, .0])
        m, n = A.size
        I = matrix(0.0, (n, n))
        I[::n + 1] = 1.0
        G = matrix([-I, matrix(0.0, (1, n)), I])
        h = matrix(n * [0.0] + [1.0] + n * [0.0])
        dims = {"l": n, "q": [n + 1], "s": []}
        return {"x": solvers.coneqp(A.T * A, -A.T * b, G, h, dims, kktsolver="chol")["x"]}
    x = ref_golden("coneqp", reference)["x"]
    np.testing.assert_allclose(np.array(x).ravel(), [0.72558319, 0.61806264, 0.30253528], atol=1e-5)
