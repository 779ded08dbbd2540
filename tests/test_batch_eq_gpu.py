"""Batch QP solver with equality constraints A x = b vs the reference: a Python loop over
solvers.qp(P, q, G, h, A, b, kktsolver='chol2') on the same problems (its stored results, tests/reference_results.py).
Same status and iteration count per problem, objectives to rtol 1e-8, x and y to 1e-6, s and z to 1e-5."""
import numpy as np
import pytest

from problems import dense_qp

pytestmark = pytest.mark.gpu


def eq_qp(n, m, p, seed):
    """dense_qp(n, m, seed) with p equality rows A x = b through its strictly feasible point x0"""
    P, q, G, h = dense_qp(n, m, seed)
    rng = np.random.Generator(np.random.PCG64(seed))       # replay dense_qp's draws up to x0
    rng.standard_normal((n, n)); rng.standard_normal(n); rng.standard_normal((m, n))
    x0 = rng.standard_normal(n)
    rng.uniform(0.1, 1.1, m)
    A = rng.standard_normal((p, n))
    return P, q, G, h, A, A @ x0, x0


def singular_S_qp(n, m, k, seed):
    """P zero on the last k coordinates, G with zero columns there, p = k rows of A that are generic on them:
    P + G'G is singular, [P; A; G] has rank n"""
    P, q, G, h, A, b, x0 = eq_qp(n, m, k, seed)
    P[-k:, :] = 0.0
    P[:, -k:] = 0.0
    G[:, -k:] = 0.0
    h = G @ x0 + np.random.Generator(np.random.PCG64(seed + 1000)).uniform(0.1, 1.1, m)
    return P, q, G, h, A, A @ x0


def make_batch(B, n, m, p, seed0=0, singular=()):
    probs = [singular_S_qp(n, m, p, seed0 + k) if k in singular else eq_qp(n, m, p, seed0 + k)[:6] for k in range(B)]
    return tuple(np.stack([pr[i] for pr in probs]) for i in range(6))


def ref_loop(P, q, G, h, A, b):
    from cvxopt import lapack, matrix, solvers
    out = {}
    for k in range(P.shape[0]):
        sol = solvers.qp(matrix(P[k]), matrix(q[k]), matrix(G[k]), matrix(h[k]), matrix(A[k]), matrix(b[k]),
                         kktsolver="chol2")
        out.update({"%d.%s" % (k, key): sol[key] for key in ("status", "iterations", "primal objective",
                                                               "dual objective", "x", "y", "s", "z")})
        # kkt_chol2's first factorisation (W = I): S = G'G + P; the 'singular' branch is taken where it fails
        S = matrix(G[k].T @ G[k] + P[k])
        try:
            lapack.potrf(S)
            out["%d.singular" % k] = 0
        except ArithmeticError:
            out["%d.singular" % k] = 1
    return out


def per_problem(ref, B):
    return [{key.split(".", 1)[1]: v for key, v in ref.items() if key.split(".", 1)[0] == str(k)} for k in range(B)]


def assert_matches(got, want, B):
    for k in range(B):
        assert got["status"][k] == want[k]["status"] == "optimal", k
        assert got["iterations"][k] == want[k]["iterations"], (k, got["iterations"], want[k]["iterations"])
        np.testing.assert_allclose(got["primal objective"][k], want[k]["primal objective"], rtol=1e-8)
        np.testing.assert_allclose(got["dual objective"][k], want[k]["dual objective"], rtol=1e-8)
        np.testing.assert_allclose(got["x"][k], np.array(want[k]["x"]).ravel(), rtol=1e-6, atol=1e-8)
        np.testing.assert_allclose(got["y"][k], np.array(want[k]["y"]).ravel(), rtol=1e-6, atol=1e-8)
        np.testing.assert_allclose(got["s"][k], np.array(want[k]["s"]).ravel(), rtol=1e-5, atol=1e-7)
        np.testing.assert_allclose(got["z"][k], np.array(want[k]["z"]).ravel(), rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("B,n,m,p", [(5, 30, 70, 1), (3, 150, 321, 12), (2, 257, 300, 40), (1, 300, 640, 64)])
def test_batch_eq_matches_reference_loop(ref_golden, B, n, m, p):
    import cvxopt_b200
    P, q, G, h, A, b = make_batch(B, n, m, p, seed0=10 * B + p)
    want = per_problem(ref_golden("qp_loop", lambda: ref_loop(P, q, G, h, A, b)), B)
    got = cvxopt_b200.qp_batch(P, q, G, h, A, b)
    assert got["y"].shape == (B, p)
    assert_matches(got, want, B)


def test_singular_S_matches_reference(ref_golden):
    """problems whose P + G'G is singular factor S + A'A (kkt_chol2's 'singular' branch), the others do not"""
    from cvxopt_b200.batch import QPBatch
    B, n, m, k = 6, 40, 90, 3
    sing = (1, 2, 4)
    P, q, G, h, A, b = make_batch(B, n, m, k, seed0=700, singular=sing)
    want = per_problem(ref_golden("qp_loop", lambda: ref_loop(P, q, G, h, A, b)), B)
    assert [w["singular"] for w in want] == [int(i in sing) for i in range(B)]
    bt = QPBatch(B, n, m, 0, p=k)
    try:
        bt.load(P, q, G, h, A, b)
        bt.solve()
        got = bt.results()
        flags = bt.singular()
    finally:
        bt.close()
    assert list(flags) == [i in sing for i in range(B)]
    assert_matches(got, want, B)


def test_int8_syrk_path_with_equality_constraints(ref_golden, monkeypatch):
    """B = 1 with the int8-slice SYRK forced: the equality elimination runs after the single-problem Cholesky"""
    from cvxopt_b200.batch import QPBatch
    n, m, p = 300, 640, 24
    P, q, G, h, A, b = make_batch(1, n, m, p, seed0=900)
    want = per_problem(ref_golden("qp_loop", lambda: ref_loop(P, q, G, h, A, b)), 1)
    monkeypatch.setenv("CVXB_OZAKI", "2")
    bt = QPBatch(1, n, m, 0, p=p)
    try:
        bt.load(P, q, G, h, A, b)
        bt.solve()
        got = bt.results()
        assert bt.stats()["syrk_path"] == "int8"
    finally:
        bt.close()
    assert_matches(got, want, 1)


def test_compaction_with_equality_constraints(monkeypatch):
    """finished problems swapped out of the active prefix carry A, b and their p-vectors along: results are those
    of the uncompacted loop, in the caller's order, and a second solve repeats them"""
    import cvxopt_b200
    from cvxopt_b200.batch import QPBatch
    B, n, m, p = 24, 40, 90, 5
    P, q, G, h, A, b = make_batch(B, n, m, p, seed0=500, singular=(4, 13))
    for k in range(0, B, 3):
        q[k] *= 1e3
        h[k] *= 1e-2
        b[k] *= 1e-2
    monkeypatch.setenv("CVXB_BATCH_COMPACT", "0")
    plain = cvxopt_b200.qp_batch(P, q, G, h, A, b, nsub=1)
    monkeypatch.setenv("CVXB_BATCH_COMPACT", "1")
    bt = QPBatch(B, n, m, 0, p=p)
    try:
        bt.load(P, q, G, h, A, b)
        bt.solve()
        r1 = bt.results()
        f1 = bt.singular()
        bt.solve()
        r2 = bt.results()
        f2 = bt.singular()
    finally:
        bt.close()
    assert len(set(plain["iterations"])) > 1
    assert all(s == "optimal" for s in plain["status"])
    for r, f in ((r1, f1), (r2, f2)):
        assert list(f) == [k in (4, 13) for k in range(B)]
        assert list(r["iterations"]) == list(plain["iterations"])
        assert list(r["status_code"]) == list(plain["status_code"])
        for key in ("x", "y", "s", "z", "primal objective", "dual objective"):
            np.testing.assert_array_equal(r[key], plain[key])


def test_subbatches_and_distributed_entry_with_equality_constraints():
    import cvxopt_b200
    B, n, m, p = 7, 60, 130, 4
    P, q, G, h, A, b = make_batch(B, n, m, p, seed0=40, singular=(3,))
    one = cvxopt_b200.qp_batch(P, q, G, h, A, b, nsub=1)
    three = cvxopt_b200.qp_batch(P, q, G, h, A, b, nsub=3)
    assert three["nsub"] == 3
    assert all(s == "optimal" for s in one["status"])
    assert list(one["iterations"]) == list(three["iterations"])
    for key in ("x", "y", "primal objective"):
        np.testing.assert_allclose(three[key], one[key], rtol=1e-12, atol=1e-12)
    dist = cvxopt_b200.qp_batch_distributed(P, q, G, h, A=A, b=b, nsub=1)["all"]
    assert list(dist["iterations"]) == list(one["iterations"])
    for key in ("x", "y", "s", "z", "primal objective", "dual objective"):
        np.testing.assert_allclose(dist[key], one[key], rtol=1e-12, atol=1e-12)


def test_p0_unchanged():
    """A with no rows is the problem without A, bit for bit"""
    import cvxopt_b200
    B, n, m = 4, 50, 110
    P, q, G, h, _, _ = make_batch(B, n, m, 0, seed0=60)
    old = cvxopt_b200.qp_batch(P, q, G, h)
    new = cvxopt_b200.qp_batch(P, q, G, h, np.zeros((B, 0, n)), np.zeros((B, 0)))
    assert new["y"].shape == (B, 0)
    assert list(new["iterations"]) == list(old["iterations"])
    for key in ("x", "s", "z", "primal objective", "dual objective"):
        np.testing.assert_array_equal(new[key], old[key])


def test_rank_deficient_A_raises():
    """Rank(A) < p.  A zero row leaves an exactly zero pivot in the Cholesky factor of A S^-1 A'.  (A repeated row
    would not be a sure case: its pivot is the rounding residue of x - (x / sqrt(x))^2, of either sign, in the
    reference's LAPACK as much as here.)"""
    import cvxopt_b200
    P, q, G, h, A, b = make_batch(2, 30, 70, 3, seed0=80)
    A[1, 2] = 0.0
    b[1, 2] = 0.0
    with pytest.raises(ValueError, match="Rank"):
        cvxopt_b200.qp_batch(P, q, G, h, A, b)


def test_rank_deficient_PAG_raises():
    import cvxopt_b200
    P, q, G, h, A, b = make_batch(2, 30, 70, 3, seed0=90, singular=(0,))
    A[0, :, -1] = 0.0                      # the last coordinate is in no row of [P; A; G]
    with pytest.raises(ValueError, match="Rank"):
        cvxopt_b200.qp_batch(P, q, G, h, A, b)
